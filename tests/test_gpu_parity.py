"""GPU tier (-m gpu): parity of the CUDA path, called through the C ABI, against the compiled reference
(oracle/_ref where it was built, and what it returned as recorded in tests/golden/reference/), the C restatement and the
committed digests.  Bit-exact."""
import ctypes as C
import hashlib
import json
import zlib

import numpy as np
import pytest

import jpegdec_b200 as J
from tests import common as T
from tests import synth

pytestmark = pytest.mark.gpu
MODES = [("sse", 0), ("scalar", 1)]


def _ref(mode):
    from oracle import refdrv
    return refdrv.Ref(mode) if refdrv.available(mode) else None


@pytest.fixture(scope="module")
def ctxs():
    c = {0: J.Context(0, 0), 1: J.Context(0, 1)}
    yield c
    for x in c.values():
        x.close()


def test_native_library_is_the_one_running(ctxs):
    assert J.lib().JPEGB200_deviceCount() >= 1
    outs, st, tim, cnt = J.decode_batch_to_host(ctxs[0], [T.image("tulips")], 0, 0)
    assert st == [0] and cnt["launches"] >= 5 and cnt["events"] >= 7


@pytest.mark.parametrize("mode,arith", MODES)
def test_fixture_batch_all_pixel_types_and_scales(ctxs, mode, arith):
    """One mixed batch (different sizes, subsamplings, Huffman table sets, DRI / no DRI) per pixel type x scale."""
    d = T.digests()
    blobs = [T.image(n) for n in T.VALID]
    ref = _ref(mode)
    for pt, ptn in T.PTS:
        for opt, sn in T.SCALES:
            outs, st, tim, cnt = J.decode_batch_to_host(ctxs[arith], blobs, pt, opt)
            assert st == [0] * len(blobs)
            for n, o, data in zip(T.VALID, outs, blobs):
                want = d[n]["%s/%s/%s" % (mode, ptn, sn)]
                assert list(o.shape) == want["shape"]
                assert T.sha(o) == want["sha"], (n, mode, ptn, sn)
                if ref is not None and n in ("tulips", "zebra"):
                    rc, err, img, _ = ref.decode_cb(data, pt, opt, want_log=False)
                    assert np.array_equal(o, img)


@pytest.mark.parametrize("mode,arith", MODES)
def test_synthetic_formats(ctxs, mode, arith):
    """grayscale, 4:4:4, 4:2:2, 4:4:0, odd sizes, no restart markers, high quality -- vs the C restatement
    (itself pinned to the reference on the same cases in the CPU tier) and the live reference when present."""
    import cv2
    cases = {"gray": synth.synth_jpeg(640, 360, 1, 75, gray=True),
             "s444": synth.synth_jpeg(333, 251, 2, 80, subsampling="4:4:4"),
             "s422": synth.synth_jpeg(333, 251, 3, 80, subsampling="4:2:2"),
             "odd420": synth.synth_jpeg(301, 203, 4, 90, restart_rows=0),
             "q98": synth.synth_jpeg(256, 256, 5, 98),
             "hd": synth.synth_jpeg(1920, 1080, 6, 75)}
    ok, enc = cv2.imencode(".jpg", synth.synth_pixels(200, 150, 7),
                           [cv2.IMWRITE_JPEG_QUALITY, 85, cv2.IMWRITE_JPEG_SAMPLING_FACTOR, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_440])
    cases["s440"] = enc.tobytes()
    from tests.test_oracle import _odd_restart_cases
    odd = _odd_restart_cases()                     # DRI = 1 / 7 MCUs / 2 rows, q100, q5 (all 333x251)
    cases.update(odd)
    ref = _ref(mode)
    for pt, ptn in T.PTS:
        for opt, sn in T.SCALES:
            names = [n for n in cases if not (n == "gray" and pt == 2)]
            outs, st, tim, cnt = J.decode_batch_to_host(ctxs[arith], [cases[n] for n in names], pt, opt)
            assert st == [0] * len(names)
            for n, o in zip(names, outs):
                if n == "s440" and pt == 2 and opt == 4:
                    continue  # reference bug: JPEGPutMCU12 1/4 RGB8888 writes through &pOutput (jpeg.inl:4629)
                info = J.Batch  # noqa
                w = {"gray": 640, "s444": 333, "s422": 333, "odd420": 301, "q98": 256, "hd": 1920, "s440": 200}.get(n, 333)
                h = {"gray": 360, "s444": 251, "s422": 251, "odd420": 203, "q98": 256, "hd": 1080, "s440": 150}.get(n, 251)
                rc, want = T.oracle_decode(cases[n], pt, opt, arith, w, h)
                assert rc == 1 and np.array_equal(o, want), (n, mode, ptn, sn)
                if ref is not None and n in ("hd", "s422"):
                    rc, err, img, _ = ref.decode_cb(cases[n], pt, opt, want_log=False)
                    assert np.array_equal(o, img), (n, mode, ptn, sn)


@pytest.mark.parametrize("mode,arith", MODES)
def test_dither_batch(ctxs, mode, arith):
    d = T.digests()
    names = ["tulips", "zebra", "ncc1701", "sciopero"]
    for pt, ptn in T.DITHERS:
        outs, st, tim, cnt = J.decode_batch_to_host(ctxs[arith], [T.image(n) for n in names], pt, 0)
        assert st == [0] * len(names)
        for n, o in zip(names, outs):
            want = d[n]["%s/%s/full" % (mode, ptn)]
            inf = d[n]["info"]
            rc, w2 = T.oracle_decode(T.image(n), pt, 0, arith, inf["width"], inf["height"])
            wb = (inf["width"] * T.bpp_of(pt) + 7) // 8
            assert np.array_equal(o[:, :wb], w2[:o.shape[0], :wb]), (n, mode, ptn)


def _collect(j, pt, options, x=0, y=0):
    """decode through the draw callback; returns (rc, log, tight image assembled like oracle/ref_shim.c does)."""
    log, blocks = [], []

    def draw(d):
        nbytes = ((d.iWidth * d.iBpp + 7) // 8) * d.iHeight
        buf = C.string_at(d.pPixels, nbytes)
        log.append((d.x, d.y, d.iWidth, d.iHeight, d.iWidthUsed, d.iBpp))
        blocks.append(buf)
        return 1
    return draw, log, blocks


CALLBACK_CASES = [("sciopero", 0, 0, 10, 20, 0), ("sciopero", 2, 0, 0, 0, 0), ("sciopero", 3, 0, 0, 0, 0),
                  ("sciopero", 0, 2, 0, 0, 0), ("sciopero", 0, 4, 3, 5, 0), ("sciopero", 0, 8, 0, 0, 0),
                  ("tulips", 0, 0, 0, 0, 0), ("tulips", 0, J.JPEG_USES_DMA, 0, 0, 0), ("tulips", 0, 0, 0, 0, 3),
                  ("ncc1701", 2, 0, 0, 0, 0), ("zebra", 1, 0, 0, 0, 0), ("zebra", 0, 2, 0, 0, 0), ("lange", 3, 4, 0, 0, 0),
                  ("tulips", 0, J.JPEG_LUMA_ONLY, 0, 0, 0)]


def _callback_key(mode, case):
    return "%s/%s/%d/%d/%d/%d/%d" % ((mode,) + case)


def record_callbacks(refs):
    out = {}
    for mode, arith in MODES:
        for case in CALLBACK_CASES:
            name, pt, opt, xo, yo, maxm = case
            rc_r, err_r, img_r, log_r = refs[mode].decode_cb(T.image(name), pt, opt, xoff=xo, yoff=yo, max_mcus=maxm)
            out[_callback_key(mode, case)] = {"rc": rc_r, "log": T.log_sha([r[:6] for r in log_r]), "shape": list(img_r.shape),
                                              "sha": T.sha(img_r)}
    return out


@pytest.mark.parametrize("mode,arith", MODES)
def test_single_image_api_callbacks_match_reference(mode, arith):
    """JPEG_openRAM -> setPixelType -> decode: same callback sequence (x, y, iWidth, iHeight, iWidthUsed, iBpp)
    and same delivered pixels as the reference, incl. decode offset, JPEG_USES_DMA and setMaxOutputSize."""
    want = T.reference_calls("gpu_callbacks")
    for case in CALLBACK_CASES:
        name, pt, opt, xo, yo, maxm = case
        g = want[_callback_key(mode, case)]
        data = T.image(name)
        j = J.JPEGDEC()
        draw, log, blocks = _collect(j, pt, opt)
        assert j.openRAM(data, draw) == 1
        j.setArithMode(arith)
        j.setPixelType(pt)
        if maxm:
            j.setMaxOutputSize(maxm)
        rc = j.decode(xo, yo, opt)
        assert rc == g["rc"] == 1, (name, pt, opt, j.getLastError())
        assert T.log_sha(log) == g["log"], (name, pt, opt)
        # assemble the tight image from the delivered blocks
        out = np.zeros(g["shape"], np.uint8)
        for (x, y, w, h, wu, bpp), buf in zip(log, blocks):
            pitch = (w * bpp + 7) // 8
            a = np.frombuffer(buf, dtype=np.uint8).reshape(h, pitch)
            bw = wu * bpp // 8
            x0 = (x - xo) * bpp // 8
            out[y - yo:y - yo + h, x0:x0 + bw] = a[:, :bw]
        assert T.sha(out) == g["sha"], (name, pt, opt)
        j.close()


# framebuffer mode: tulips has a multiple-of-16 width (reference pitch = image width, identical bytes); the others have a
# width / height that is not a multiple of the MCU: the reference's SSE2 build stores whole MCUs (the right edge runs on into
# the next line), its scalar build clips -- the visible w x h region must match either way
FRAMEBUFFER_CASES = [("tulips", 640, 480, pt) for pt in (0, 2, 3)] + \
    [(name, w, h, pt) for name, w, h in (("sciopero", 300, 300), ("ncc1701", 240, 77), ("zebra", 320, 240)) for pt in (0, 2)]


def record_framebuffer_crop_thumb_dither(refs):
    out = {}
    for mode, arith in MODES:
        ref = refs[mode]
        for name, w, h, pt in FRAMEBUFFER_CASES:
            rc_r, err_r, fb_r = ref.decode_fb(T.image(name), pt, 0)
            n = w * h * T.bpp_of(pt) // 8
            out["%s/fb/%s/%d" % (mode, name, pt)] = {"rc": rc_r, "bytes": int(fb_r.size), "sha": T.sha(fb_r[:n])}
        rc_r, err_r, img_r, log_r = ref.decode_cb(T.image("tulips"), 0, 0, crop=(50, 50, 125, 170))
        out[mode + "/crop"] = {"rc": rc_r, "log": T.log_sha([r[:6] for r in log_r]), "sha": T.sha(img_r[:176, :256])}
        rc_r, err_r, img_r, log_r = ref.decode_cb(T.image("thumb_test"), 0, J.JPEG_EXIF_THUMBNAIL)
        out[mode + "/thumb"] = {"rc": rc_r, "log": T.log_sha([r[:6] for r in log_r]), "shape": list(img_r.shape), "sha": T.sha(img_r)}
        rc_r, err_r, img_r, log_r = ref.decode_dither(T.image("zebra"), J.ONE_BIT_DITHERED, 0)
        out[mode + "/dither"] = {"rc": rc_r, "log": T.log_sha([r[:6] for r in log_r]), "shape": list(img_r.shape),
                                 "sha": T.sha(img_r[:, :40])}
    return out


@pytest.mark.parametrize("mode,arith", MODES)
def test_single_image_api_framebuffer_crop_thumb_dither(mode, arith):
    want = T.reference_calls("gpu_framebuffer_crop_thumb_dither")
    for name, w, h, pt in FRAMEBUFFER_CASES:
        g = want["%s/fb/%s/%d" % (mode, name, pt)]
        d2 = T.image(name)
        j = J.JPEGDEC(); assert j.openRAM(d2); j.setArithMode(arith); j.setPixelType(pt)
        fb = np.zeros(g["bytes"], np.uint8); j.setFramebuffer(fb)
        assert j.decode(0, 0, 0) == g["rc"] == 1
        n = w * h * T.bpp_of(pt) // 8
        assert T.sha(fb[:n]) == g["sha"], (name, pt, mode)
    # crop through callbacks (reference test 2): exactly the snapped rectangle, same pixels
    data = T.image("tulips")
    g = want[mode + "/crop"]
    j = J.JPEGDEC(); draw, log, blocks = _collect(j, 0, 0)
    assert j.openRAM(data, draw); j.setArithMode(arith); j.setCropArea(50, 50, 125, 170)
    assert j.decode(0, 0, 0) == 1
    assert T.log_sha(log) == g["log"]
    out = np.zeros((176, 256), np.uint8)
    for (x, y, w, h, wu, bpp), buf in zip(log, blocks):
        a = np.frombuffer(buf, dtype=np.uint8).reshape(h, w * 2)
        out[y:y + h, x * 2:(x + wu) * 2] = a[:, :wu * 2]
    assert T.sha(out) == g["sha"]
    # EXIF thumbnail (reference test 10): 320x240
    tdata = T.image("thumb_test")
    g = want[mode + "/thumb"]
    j = J.JPEGDEC(); draw, log, blocks = _collect(j, 0, 0)
    assert j.openRAM(tdata, draw) and j.hasThumb() and (j.getThumbWidth(), j.getThumbHeight()) == (320, 240)
    j.setArithMode(arith)
    assert j.decode(0, 0, J.JPEG_EXIF_THUMBNAIL) == g["rc"] == 1
    assert (j.getWidth(), j.getHeight()) == (320, 240)
    assert T.log_sha(log) == g["log"]
    out = np.zeros(g["shape"], np.uint8)
    for (x, y, w, h, wu, bpp), buf in zip(log, blocks):
        a = np.frombuffer(buf, dtype=np.uint8).reshape(h, w * 2)
        out[y:y + h, x * 2:(x + wu) * 2] = a[:, :wu * 2]
    assert T.sha(out) == g["sha"]
    # decodeDither through the callback
    zdata = T.image("zebra")
    g = want[mode + "/dither"]
    j = J.JPEGDEC(); draw, log, blocks = _collect(j, 6, 0)
    assert j.openRAM(zdata, draw); j.setArithMode(arith); j.setPixelType(J.ONE_BIT_DITHERED)
    dbuf = np.zeros((320 + 32) * 16, np.uint8)
    assert j.decodeDither(dbuf, 0) == g["rc"] == 1
    assert T.log_sha(log) == g["log"]
    out = np.zeros(g["shape"], np.uint8)
    for (x, y, w, h, wu, bpp), buf in zip(log, blocks):
        a = np.frombuffer(buf, dtype=np.uint8).reshape(h, (w + 7) // 8)
        out[y:y + h, :(wu + 7) // 8] = a[:, :(wu + 7) // 8]
    assert T.sha(out[:, :40]) == g["sha"]


def test_corrupt_inputs_do_not_poison_the_batch(ctxs):
    """reference tests 4-8 + 11 (MacOS/JPEGDEC_Test/JPEGDEC_Test/main.cpp:164-216, :262-300): corrupt files
    return 0/1 without crashing; a bad image must not disturb its neighbours in the same batch."""
    good = T.image("tulips")
    want = J.decode_batch_to_host(ctxs[0], [good], 0, 0)[0][0]
    blobs = [good] + [T.image("corrupt%d" % i) for i in range(1, 6)] + [good]
    rng = np.random.default_rng(3)
    for k in range(12):  # entropy-segment corruption
        b = bytearray(good)
        for _ in range(4):
            b[int(rng.integers(700, len(b) - 2))] = int(rng.integers(0, 256))
        blobs.append(bytes(b))
    base2 = T.image("sciopero")                 # no restart markers: chunk-parallel path
    for k in range(8):
        b = bytearray(base2)
        for _ in range(3):
            b[int(rng.integers(700, len(b) - 2))] = int(rng.integers(0, 256))
        blobs.append(bytes(b))
    blobs.append(bytes(base2[:len(base2) // 2]) + b"\x00" * 64)   # truncated scan
    blobs.append(good)
    outs, st, tim, cnt = J.decode_batch_to_host(ctxs[0], blobs, 0, 0)
    assert all(s in range(6) for s in st)
    d = T.digests()
    for i in range(1, 6):
        if not d["corrupt%d" % i]["open"]:
            assert st[i] == d["corrupt%d" % i]["info"]["error"]
    for i in (0, 6, len(blobs) - 1):
        assert st[i] == 0 and np.array_equal(outs[i], want)


def test_batch_properties_at_baseline_size(ctxs):
    """BASELINE.json configs[1] shape: 1024 x 1920x1080 -> RGB8888.  Size-independent properties: every copy of a
    unique image in the batch yields the same CRC as that image decoded alone; the checksum of checksums is
    identical across two runs; a sample is bit-exact vs the C restatement."""
    uniq = synth.synth_set(8, 1920, 1080, quality=75)
    n = 1024
    bufs = [np.frombuffer(uniq[i % 8], dtype=np.uint8) for i in range(n)]
    L = J.lib()

    def run():
        b = J.Batch(ctxs[0], [x.ctypes.data for x in bufs], [len(x) for x in bufs], J.RGB8888, 0)
        b.alloc_device_output(); b.upload(); b.decode(J.JPEGB200_OUT_DEVICE); b.download()
        st = b.wait()
        crcs = []
        for i in range(n):
            crcs.append(zlib.crc32(b.read_output(i).tobytes()) if i < 16 or i % 97 == 0 else None)
        cnt = b.counters()
        b.close()
        return st, crcs, cnt
    st, crcs, cnt = run()
    assert st == [0] * n
    alone, st1, _, _ = J.decode_batch_to_host(ctxs[0], uniq, J.RGB8888, 0)
    base = [zlib.crc32(a.tobytes()) for a in alone]
    for i, c in enumerate(crcs):
        if c is not None:
            assert c == base[i % 8], i
    st2, crcs2, _ = run()
    assert crcs2 == crcs
    rc, want = T.oracle_decode(uniq[3], J.RGB8888, 0, 0, 1920, 1080)
    assert rc == 1 and np.array_equal(alone[3], want)
    assert cnt["segments"] == n * 68 and cnt["blocks"] == n * 8160 * 6


def test_restart_free_scans_chunk_parallel(ctxs):
    """SURVEY.md 8(f)2: files without restart markers (one long dependent bit stream) are decoded chunk-parallel."""
    cases = {"hd": (synth.synth_jpeg(1920, 1080, 9, 75, restart_rows=0), 1920, 1080),
             "uhd": (synth.synth_jpeg(3840, 2160, 3, 85, restart_rows=0), 3840, 2160),
             "gray": (synth.synth_jpeg(2048, 1536, 1, 75, gray=True, restart_rows=0), 2048, 1536),
             "s444": (synth.synth_jpeg(1024, 768, 2, 96, subsampling="4:4:4", restart_rows=0), 1024, 768),
             "q98": (synth.synth_jpeg(512, 512, 5, 98, restart_rows=0), 512, 512),
             # 4 blocks per MCU: chunks whose first block is not the first block of an MCU
             "s422": (synth.synth_jpeg(1000, 700, 4, 85, subsampling="4:2:2", restart_rows=0), 1000, 700)}
    import cv2
    ok, enc = cv2.imencode(".jpg", synth.synth_pixels(999, 701, 6),
                           [cv2.IMWRITE_JPEG_QUALITY, 70, cv2.IMWRITE_JPEG_SAMPLING_FACTOR, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_440])
    cases["s440"] = (enc.tobytes(), 999, 701)
    names = list(cases)
    for arith in (0, 1):
        for pt in (0, 3):
            outs, st, tim, cnt = J.decode_batch_to_host(ctxs[arith], [cases[n][0] for n in names], pt, 0)
            assert st == [0] * len(names)
            for n, o in zip(names, outs):
                data, w, h = cases[n]
                rc, want = T.oracle_decode(data, pt, 0, arith, w, h)
                assert rc == 1 and np.array_equal(o, want), (n, arith, pt)


def test_one_call_decode_batch_pipelines_jobs_and_matches_the_single_job_path(ctxs):
    """JPEGB200_decodeBatch with host outputs cuts the batch into jobs on separate streams (more than 64 images, and
    small images so that a job is grown to hold enough pixels); every image must equal the one-job result, a corrupt
    file must get its own status at its own index, and the summed counters must cover every image."""
    ref = _ref("sse")
    base = [synth.synth_jpeg(160 + 16 * (s % 5), 96 + 8 * (s % 3), s, 70 + s % 20) for s in range(12)]
    big = [synth.synth_jpeg(1920, 1080, 100 + s, 75) for s in range(3)]
    jp = [base[i % 12] for i in range(200)] + [big[i % 3] for i in range(70)]
    bad = 137
    jp[bad] = jp[bad][:200]
    want, st_want, _, _ = J.decode_batch_to_host(ctxs[0], jp, J.RGB8888, 0)
    bufs = [np.frombuffer(j, dtype=np.uint8) for j in jp]
    outs = [np.zeros_like(w) if w is not None else np.zeros(16, dtype=np.uint8) for w in want]
    pitches = [int(o.shape[1]) if o.ndim == 2 else 0 for o in outs]
    rc, st, cnt = J.decode_batch(ctxs[0], [b.ctypes.data for b in bufs], [len(b) for b in bufs], J.RGB8888, 0,
                                 [o.ctypes.data for o in outs], pitches)
    assert rc == 2 and st == st_want and st[bad] != 0 and sum(1 for x in st if x) == 1
    for i, (o, w) in enumerate(zip(outs, want)):
        if w is not None and st[i] == 0:
            assert np.array_equal(o, w), i
    assert cnt["output_bytes"] == sum(int(w.size) for w in want if w is not None)
    assert cnt["launches"] >= 10           # several jobs ran
    if ref is not None:
        for i in (0, 7, 199, 200, 269):
            rc1, err, img, _ = ref.decode_cb(jp[i], J.RGB8888, 0, want_log=False)
            assert rc1 == 1 and np.array_equal(img, outs[i][:, :img.shape[1]]), i


def test_progressive_files_give_the_dc_thumbnail(ctxs):
    """SURVEY.md 8(f)4.  Batch API: progressive files decode at JPEG_SCALE_EIGHTH (DC of the first scan), next to baseline
    files in the same batch; without the 1/8 option a progressive file gets JPEG_UNSUPPORTED_FEATURE at its own index.
    Single-image API: JPEG_decode forces 1/8 like the reference (src/jpeg.inl:4964-4966)."""
    g = json.load(open(T.GOLD + "/progressive.json"))
    names = ["prog_420", "prog_420_dri", "prog_444", "prog_422", "prog_gray"]
    base = T.image("tulips")
    for mode, arith in MODES:
        for pt, ptn in ((0, "565le"), (1, "565be"), (2, "8888")):
            use = [n for n in names if "%s/%s/opt8" % (mode, ptn) in g[n]]
            blobs = [base] + [T.image(n) for n in use] + [base]
            outs, st, tim, cnt = J.decode_batch_to_host(ctxs[arith], blobs, pt, J.JPEG_SCALE_EIGHTH)
            assert st == [0] * len(blobs)
            assert np.array_equal(outs[0], outs[-1])
            for n, o in zip(use, outs[1:-1]):
                want = g[n]["%s/%s/opt8" % (mode, ptn)]
                assert list(o.shape) == want["shape"] and T.sha(o) == want["sha"], (n, mode, ptn)
            ref = _ref(mode)
            if ref is not None:
                rc, err, img, _ = ref.decode_cb(base, pt, J.JPEG_SCALE_EIGHTH, want_log=False)
                assert np.array_equal(outs[0], img)
    outs, st, tim, cnt = J.decode_batch_to_host(ctxs[0], [base, T.image("prog_420"), base], 0, 0)
    assert st[0] == 0 and st[2] == 0 and st[1] == 3 and np.array_equal(outs[0], outs[2])     # JPEG_UNSUPPORTED_FEATURE
    # single-image API, options = 0, through the callback
    for name in ("prog_420", "prog_gray"):
        data = T.image(name)
        j = J.JPEGDEC(); draw, log, blocks = _collect(j, 0, 0)
        assert j.openRAM(data, draw) and j.getJPEGType() == 1
        assert j.decode(0, 0, 0) == 1
        oh, ow2 = g[name]["sse/565le/opt0"]["shape"]
        out = np.zeros((oh, ow2), np.uint8)
        for (x, y, w, h, wu, bpp), buf in zip(log, blocks):
            a = np.frombuffer(buf, dtype=np.uint8).reshape(h, w * 2)
            out[y:y + h, x * 2:(x + wu) * 2] = a[:, :wu * 2]
        assert T.sha(out) == g[name]["sse/565le/opt0"]["sha"], name


def _gpu_sweep_files():
    rng = np.random.default_rng(77)
    files = []
    for case in range(48):
        w, h = int(rng.integers(16, 420)), int(rng.integers(16, 300))
        q = int(rng.integers(15, 101))
        gray = bool(rng.integers(0, 6) == 0)
        sub = ["4:2:0", "4:2:0", "4:2:2", "4:4:4"][int(rng.integers(0, 4))]
        files.append((synth.synth_jpeg(w, h, 5000 + case, q, subsampling=sub, gray=gray, restart_rows=int(rng.integers(0, 3))), gray))
    return files


def record_gpu_sweep(refs):
    files = _gpu_sweep_files()
    out = {"input/%d" % i: {"input": T.sha(np.frombuffer(d, dtype=np.uint8))} for i, (d, g) in enumerate(files)}
    for mode, arith in MODES:
        for pt in (0, 2, 3):
            for opt in (0, 2):
                for i, (d, gray) in enumerate(files):
                    if not (gray and pt == 2):
                        rc, err, img, _ = refs[mode].decode_cb(d, pt, opt, want_log=False)
                        out["%s/%d/%d/%d" % (mode, pt, opt, i)] = {"rc": rc, "shape": list(img.shape), "sha": T.sha(img)}
    return out


def test_seeded_random_sweep_on_the_gpu(ctxs):
    """Seeded random 4:2:0 / 4:4:4 / 4:2:2 / gray files of random size and quality (15..100: every mix of the IDCT kernel's
    block classes), random restart interval, decoded in mixed batches per pixel type at full size and 1/2, both arithmetic
    modes, against what the compiled reference returned for them."""
    files = _gpu_sweep_files()
    want = T.reference_calls("gpu_sweep")
    for i, (d, gray) in enumerate(files):
        T.check_input(want["input/%d" % i], d, i)
    for mode, arith in MODES:
        for pt in (0, 2, 3):
            for opt in (0, 2):
                use = [i for i, (d, g) in enumerate(files) if not (g and pt == 2)]
                outs, st, tim, cnt = J.decode_batch_to_host(ctxs[arith], [files[i][0] for i in use], pt, opt)
                assert st == [0] * len(use)
                for k, (i, o) in enumerate(zip(use, outs)):
                    g = want["%s/%d/%d/%d" % (mode, pt, opt, i)]
                    assert g["rc"] == 1 and list(o.shape) == g["shape"] and T.sha(o) == g["sha"], (k, mode, pt, opt)


def test_pipeline_switches_give_the_default_result():
    """JPEGDEC_B200_ENTROPY=raw (the entropy kernel un-stuffs inside its bit reader) against the default pipeline (jdk_unstuff_segs
    first, plain word reader), in a subprocess because the switch is read once: same status, same pixels, same event counts."""
    import os
    import subprocess
    import sys
    code = r'''
import sys, zlib, numpy as np
sys.path.insert(0, %r)
import jpegdec_b200 as J
from tests import common as T, synth
blobs = [T.image(n) for n in ("tulips", "sciopero", "st_peters", "zebra", "croptest", "lange", "ncc1701", "corrupt2", "prog_420")]
blobs += [synth.synth_jpeg(1920, 1080, s, 75) for s in range(4)] + [synth.synth_jpeg(333, 251, 9, 97, subsampling="4:4:4", restart_rows=0)]
blobs += [synth.synth_jpeg(257, 129, 10, 100, restart_rows=1), synth.synth_jpeg(64, 48, 11, 30, restart_rows=1)]
b = bytearray(blobs[0]); b[3000] = 0xFF; b[3001] = 0x37; blobs.append(bytes(b))      # stray marker inside a segment
ctx = J.Context(0, 0)
for pt in (0, 2, 3):
    for opt in (0, 2, 4, 8):
        outs, st, tim, cnt = J.decode_batch_to_host(ctx, blobs, pt, opt)
        print(pt, opt, st, [zlib.crc32(o.tobytes()) if o is not None else None for o in outs], cnt["events"], cnt["event_candidates"])
''' % T.ROOT
    res = []
    # third run: restart-free scans with a single entry-state pass, which forces batchWait's iterate-to-the-fix-point fallback
    for extra in ({}, {"JPEGDEC_B200_ENTROPY": "raw"}, {"JPEGDEC_B200_CHUNK_PASSES": "1"}):
        env = dict(os.environ)
        env.pop("JPEGDEC_B200_ENTROPY", None)
        env.pop("JPEGDEC_B200_CHUNK_PASSES", None)
        env.update(extra)
        r = subprocess.run([sys.executable, "-c", code], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, env=env, timeout=900)
        assert r.returncode == 0, r.stdout[-2000:]
        res.append(r.stdout)
    assert res[0] == res[1] == res[2] and len(res[0].splitlines()) == 12


# ---------------------------------------------------------------------------------------------------------------------
# BASELINE.json shapes (configs[2]..[4]) against the compiled reference, bit for bit
# ---------------------------------------------------------------------------------------------------------------------
def _ref_or_restatement(mode, arith, data, pt, opt, w, h):
    """expected tight image: the compiled reference when it travelled with the snapshot, else the C restatement"""
    ref = _ref(mode)
    if ref is not None:
        rc, err, img, _ = ref.decode_cb(data, pt, opt, want_log=False)
        assert rc == 1
        return img
    rc, img = T.oracle_decode(data, pt, opt, arith, w, h)
    assert rc == 1
    return img


@pytest.mark.parametrize("mode,arith", MODES)
def test_uhd_q85_dri_to_rgb565_at_full_quarter_eighth(ctxs, mode, arith):
    """BASELINE.json configs[2] and [3]: 3840x2160 4:2:0 q85, DRI = one MCU row -> RGB565 at full size (JPEGPutMCU22 RGB565
    branch, jpeg.inl:4149-4306), 1/2, 1/4 (:2305-2326, :3627-3748) and 1/8 (DC only, :5146-5154); 8 seeds, one batch per scale."""
    jp = synth.synth_set(8, 3840, 2160, quality=85, seed0=4200)
    for opt in (0, 2, 4, 8):
        for pt in ((J.RGB565_LITTLE_ENDIAN, J.RGB565_BIG_ENDIAN) if opt in (0, 4) else (J.RGB565_LITTLE_ENDIAN,)):
            outs, st, tim, cnt = J.decode_batch_to_host(ctxs[arith], jp, pt, opt)
            assert st == [0] * len(jp)
            assert cnt["segments"] == 135 * len(jp) and cnt["blocks"] == 194400 * len(jp)
            for k, (d, o) in enumerate(zip(jp, outs)):
                want = _ref_or_restatement(mode, arith, d, pt, opt, 3840, 2160)
                assert o.shape == want.shape and np.array_equal(o, want), (k, mode, pt, opt)


@pytest.mark.parametrize("mode,arith", MODES)
def test_g2k_gray_and_444_to_dithered_and_gray(ctxs, mode, arith):
    """BASELINE.json configs[4]: 2048x1536 1-component and 4:4:4 colour q75 -> 1/2/4-bpp Floyd-Steinberg (JPEGDither,
    jpeg.inl:4871-4940, driven per MCU row :5309-5311) and the un-dithered 8-bit variant, against the compiled reference."""
    ref = _ref(mode)
    files = [synth.synth_jpeg(2048, 1536, 7300 + s, 75, gray=True) for s in range(2)]
    files += [synth.synth_jpeg(2048, 1536, 7400 + s, 75, subsampling="4:4:4") for s in range(2)]
    for pt in (J.ONE_BIT_DITHERED, J.TWO_BIT_DITHERED, J.FOUR_BIT_DITHERED, J.EIGHT_BIT_GRAYSCALE):
        outs, st, tim, cnt = J.decode_batch_to_host(ctxs[arith], files, pt, 0)
        assert st == [0] * len(files)
        wb = 2048 * T.bpp_of(pt) // 8
        for k, (d, o) in enumerate(zip(files, outs)):
            if ref is not None:
                if pt == J.EIGHT_BIT_GRAYSCALE:
                    rc, err, img, _ = ref.decode_cb(d, pt, 0, want_log=False)
                else:
                    rc, err, img, _ = ref.decode_dither(d, pt, 0)
                assert rc == 1
            else:
                rc, img = T.oracle_decode(d, pt, 0, arith, 2048, 1536)
                assert rc == 1
            assert o.shape[0] == 1536 and np.array_equal(o[:, :wb], img[:1536, :wb]), (k, mode, pt)


def test_device_output_batch_larger_than_one_job(ctxs):
    """JPEGB200_decodeBatch with JPEGB200_OUT_DEVICE and more compressed bytes than one job takes (192 MiB): the call cuts the
    batch into jobs that write straight into the caller's device memory.  Every image is verified on the device: its digest
    (JPEGB200_digestDevice) must equal the digest of the reference's pixels for that seed."""
    ctx = ctxs[0]
    uniq = synth.synth_set(8, 1920, 1080, quality=75, seed0=900)
    n = 800                                                      # ~230 MB compressed -> two jobs
    bufs = [np.frombuffer(uniq[i % 8], dtype=np.uint8) for i in range(n)]
    assert sum(len(b) for b in bufs) > (192 << 20)
    per = 1920 * 1080 * 4
    stride = (per + 255) & ~255
    dev = ctx.device_alloc(stride * n)
    try:
        outs = [dev + i * stride for i in range(n)]
        rc, st, cnt = J.decode_batch(ctx, [b.ctypes.data for b in bufs], [len(b) for b in bufs], J.RGB8888, 0, outs, None, J.JPEGB200_OUT_DEVICE)
        assert rc == 1 and st == [0] * n
        tms, jobs = ctx.last_call_timings()
        assert jobs >= 2 and cnt["blocks"] == n * 8160 * 6 and cnt["d2h_bytes"] < (1 << 20)
        dig = ctx.digest_device(outs, [per] * n)
        want = [J.digest_host(_ref_or_restatement("sse", 0, uniq[k], J.RGB8888, 0, 1920, 1080)) for k in range(8)]
        assert [dig[i] for i in range(n)] == [want[i % 8] for i in range(n)]
        # the digest sees single-pixel differences: flip one byte of image 5 on the host copy
        img5 = ctx.device_read(outs[5], per)
        assert J.digest_host(img5) == want[5]
        img5[1234567] ^= 1
        assert J.digest_host(img5) != want[5]
    finally:
        ctx.device_free(dev)


def test_rejected_last_file_with_arena_layout_outputs(ctxs):
    """A job whose LAST file has a corrupt header, decoded into host buffers laid out like the device arena (tight images,
    256-byte aligned, back to back): the single-copy download must still deliver every good image."""
    good = [synth.synth_jpeg(320, 240, 60 + s, 80) for s in range(3)]
    blobs = good + [b"\xff\xd8\xff\xe0 not a jpeg at all" + bytes(300)]
    per = 320 * 240 * 2
    stride = (per + 255) & ~255
    arena = np.zeros(stride * 4, dtype=np.uint8)
    bufs = [np.frombuffer(x, dtype=np.uint8) for x in blobs]
    rc, st, cnt = J.decode_batch(ctxs[0], [b.ctypes.data for b in bufs], [len(b) for b in bufs], 0, 0,
                                 [arena.ctypes.data + i * stride for i in range(4)], None, 0)
    assert rc == 2 and st[:3] == [0, 0, 0] and st[3] != 0
    for i in range(3):
        want = _ref_or_restatement("sse", 0, good[i], 0, 0, 320, 240)
        assert np.array_equal(arena[i * stride:i * stride + per].reshape(240, 640), want), i


def test_two_threads_two_contexts(ctxs):
    """Two host threads, each with its own context, decoding different batches at the same time (ctypes releases the GIL
    inside the calls): results equal the single-threaded ones, error text and pools are per context / per thread."""
    import threading
    sets = [[synth.synth_jpeg(640 + 16 * t, 360, 300 + 10 * t + s, 70 + 5 * t) for s in range(6)] for t in range(2)]
    want = [J.decode_batch_to_host(ctxs[0], sets[t], J.RGB8888, 0)[0] for t in range(2)]
    errs = []

    def work(t):
        try:
            c = J.Context(0, 0)
            for it in range(6):
                outs, st, tim, cnt = J.decode_batch_to_host(c, sets[t], J.RGB8888, 0)
                assert st == [0] * 6
                for a, b in zip(outs, want[t]):
                    assert np.array_equal(a, b)
                j = J.JPEGDEC()                          # and the single-image API from this thread
                fb = np.zeros(want[t][0].size + 64 * 1024 * 4, np.uint8)
                assert j.openRAM(sets[t][it % 6]); j.setPixelType(J.RGB8888); j.setFramebuffer(fb)
                assert j.decode(0, 0, 0) == 1
                j.close()
            c.close()
        except Exception as e:  # noqa
            errs.append((t, repr(e)))
    th = [threading.Thread(target=work, args=(t,)) for t in range(2)]
    [x.start() for x in th]
    [x.join() for x in th]
    assert not errs, errs


CROP_SCALE_CASES = [(name, crop, pt, opt)
                    for name, crops in (("tulips", [(96, 64, 256, 192), (50, 50, 125, 170), (0, 0, 64, 64)]), ("zebra", [(32, 16, 128, 96)]))
                    for crop in crops for pt in (0, 2, 3) for opt in (0, 2, 4, 8)]


def _crop_scale_key(mode, name, crop, pt, opt):
    return "%s/%s/%s/%d/%d" % (mode, name, ",".join(map(str, crop)), pt, opt)


def _crop_geometry(j, opt):
    """(snapped crop x, scaled width of the MCU-aligned image)"""
    cx, cy, cw, ch = j.getCropArea()
    sh = {0: 0, 2: 1, 4: 2, 8: 3}[opt]
    mcu_w = (16 if j.getSubSample() in (0x21, 0x22) else 8) >> sh
    return cx, -(-j.getWidth() // (mcu_w << sh)) * mcu_w


def _crop_groups(log, cx, aligned_w, shape):
    """per callback: (rows of the image it covers, byte offset, bytes it wrote, bytes it spans); None when it places nothing.
    A group that reaches the image's right edge before it is full carries stale bytes in the reference (never written) beyond
    the last MCU it placed: only the written part is compared."""
    for (x, y, w, h, wu, bpp) in log:
        written = min(wu, aligned_w - (cx + x))
        bw, x0 = written * bpp // 8, x * bpp // 8
        ys = slice(max(y, 0), min(y + h, shape[0]))
        if x0 < 0 or ys.start >= ys.stop or bw <= 0:
            yield None
        else:
            yield ys, x0, bw, wu * bpp // 8


def record_crop_scale(refs):
    out = {}
    for mode, arith in MODES:
        for name, crop, pt, opt in CROP_SCALE_CASES:
            data = T.image(name)
            rc_r, err_r, img_r, log_r = refs[mode].decode_cb(data, pt, opt, crop=crop)
            log = [tuple(r[:6]) for r in log_r]
            j = J.JPEGDEC(); assert j.openRAM(data); j.setPixelType(pt); j.setCropArea(*crop)
            cx, aligned_w = _crop_geometry(j, opt)
            cx, cy, cw, ch = j.getCropArea()
            j.close()
            want = img_r.copy()
            for grp in _crop_groups(log, cx, aligned_w, img_r.shape):
                if grp is not None:
                    ys, x0, bw, span = grp
                    want[ys, x0 + bw:x0 + span] = 0
            rec = {"rc": rc_r, "log": T.log_sha(log), "shape": list(img_r.shape), "sha": T.sha(want)}
            if opt == 0:
                rec["framebuffer"] = T.sha(img_r[:ch, :cw * T.bpp_of(pt) // 8])
            out[_crop_scale_key(mode, name, crop, pt, opt)] = rec
    return out


@pytest.mark.parametrize("mode,arith", MODES)
def test_crop_times_scale_callbacks_and_framebuffer(mode, arith):
    """setCropArea combined with 1/2, 1/4, 1/8 (SURVEY.md A.5: the reference compares scaled MCU positions with the unscaled
    crop rectangle) through the callback and into a framebuffer: same callback sequence, same pixels as the reference
    (src/jpeg.inl:5111-5137, :5114-5124); the geometry alone is pinned on the CPU in tests/test_host.py."""
    want = T.reference_calls("gpu_crop_scale")
    for name, crop, pt, opt in CROP_SCALE_CASES:
        data = T.image(name)
        g = want[_crop_scale_key(mode, name, crop, pt, opt)]
        j = J.JPEGDEC(); draw, log, blocks = _collect(j, pt, opt)
        assert j.openRAM(data, draw); j.setArithMode(arith); j.setPixelType(pt); j.setCropArea(*crop)
        assert j.decode(0, 0, opt) == g["rc"] == 1
        assert T.log_sha(log) == g["log"], (name, crop, pt, opt)
        out = np.zeros(g["shape"], np.uint8)
        cx, aligned_w = _crop_geometry(j, opt)
        for grp, (x, y, w, h, wu, bpp), buf in zip(_crop_groups(log, cx, aligned_w, out.shape), log, blocks):
            if grp is None:
                continue
            ys, x0, bw, span = grp
            a = np.frombuffer(buf, dtype=np.uint8).reshape(h, w * bpp // 8)
            out[ys, x0:x0 + bw] = a[ys.start - y:ys.stop - y, :bw][:, :out.shape[1] - x0]
        assert T.sha(out) == g["sha"], (name, crop, pt, opt)
        j.close()
        if opt == 0:
            # framebuffer + crop (pitch = crop width, :5116): the cropped image the callbacks deliver.  (The reference
            # itself clobbers the first pixels of most lines here: the one MCU its inclusive crop test lets through
            # past the right edge is stored beyond the pitch -- documented deviation, DESIGN.md.)
            j = J.JPEGDEC(); assert j.openRAM(data); j.setArithMode(arith); j.setPixelType(pt); j.setCropArea(*crop)
            cx, cy, cw, ch = j.getCropArea()
            bypp = T.bpp_of(pt) // 8
            fb = np.zeros((ch + 32) * cw * bypp, np.uint8); j.setFramebuffer(fb)
            assert j.decode(0, 0, opt) == 1
            got = fb[:ch * cw * bypp].reshape(ch, cw * bypp)
            assert T.sha(got) == g["framebuffer"], (name, crop, pt, opt, "framebuffer")
            j.close()
