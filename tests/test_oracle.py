"""CPU tier: the checkers themselves.  (1) the C restatement (oracle/jpegdec_oracle.c) and the sequential
stepper of the kernels' per-thread code (tests/hostsim) reproduce the digests the *compiled reference*
produced for every bundled image x pixel type x scale x arithmetic build (tests/golden/digests.json, written
by tests/golden/make_golden.py); (2) they reproduce what the compiled reference returned for dithered, synthetic and
seeded random files (tests/golden/reference/, written by tests/golden/make_reference_golden.py)."""
import numpy as np
import pytest

from tests import common as T

MODES = [("sse", 0), ("scalar", 1)]


@pytest.mark.parametrize("name", T.VALID)
def test_restatement_matches_reference_digests(name):
    d = T.digests()[name]
    data = T.image(name)
    w, h = d["info"]["width"], d["info"]["height"]
    for mode, arith in MODES:
        for pt, ptn in T.PTS:
            for opt, sn in T.SCALES:
                want = d["%s/%s/%s" % (mode, ptn, sn)]
                rc, out = T.oracle_decode(data, pt, opt, arith, w, h)
                assert rc == want["rc"]
                assert list(out.shape) == want["shape"]
                assert T.sha(out) == want["sha"], (name, mode, ptn, sn)


@pytest.mark.parametrize("name", T.VALID)
def test_kernel_stepper_matches_reference_digests(name):
    d = T.digests()[name]
    data = T.image(name)
    w, h = d["info"]["width"], d["info"]["height"]
    for mode, arith in MODES:
        for pt, ptn in T.PTS:
            for opt, sn in T.SCALES:
                want = d["%s/%s/%s" % (mode, ptn, sn)]
                rc, out, nev = T.hostsim_decode(data, pt, opt, arith, w, h)
                assert rc == want["rc"]
                assert T.sha(out) == want["sha"], (name, mode, ptn, sn)
                if pt == 0:      # the un-stuffed (CLEAN) reader of the same walk
                    rc, out, nev = T.hostsim_decode(data, pt, opt, arith, w, h, clean=True)
                    assert rc == want["rc"] and T.sha(out) == want["sha"], (name, mode, ptn, sn, "clean")


def test_window_quirk_events_are_needed():
    """SURVEY.md fact 4: tulips has 7 truncated coefficient reads; without emulating them the frame differs."""
    data = T.image("tulips")
    rc, out, nev = T.hostsim_decode(data, 0, 0, 0, 640, 480)
    assert nev == 7
    rc, out, nev = T.hostsim_decode(T.image("sciopero"), 0, 0, 0, 300, 300)
    assert nev == 9


def test_committed_golden_frame():
    want = np.fromfile(T.GOLD + "/frames/tulips_sse_rgb565le_full.bin", dtype=np.uint8).reshape(480, 1280)
    rc, out = T.oracle_decode(T.image("tulips"), 0, 0, 0, 640, 480)
    assert rc == 1 and np.array_equal(out, want)


DITHER_NAMES = ["tulips", "zebra", "ncc1701", "lange"]


def _dither_cases(name):
    """(key, mode, arith, pt, opt, width, height, bytes of a row that hold image pixels)"""
    inf = T.digests()[name]["info"]
    for mode, arith in MODES:
        for pt, ptn in T.DITHERS:
            for opt in (0, 2):
                s = 1 if opt else 0
                wb = ((((inf["width"] + (1 << s) - 1) >> s) * T.bpp_of(pt)) + 7) // 8
                yield "%s/%s/%s/%d" % (name, mode, ptn, opt), mode, arith, pt, opt, inf["width"], inf["height"], wb


def record_dither(refs):
    out = {}
    for name in DITHER_NAMES:
        for key, mode, arith, pt, opt, w, h, wb in _dither_cases(name):
            rc, err, img, log = refs[mode].decode_dither(T.image(name), pt, opt)
            out[key] = {"rc": rc, "rows": img.shape[0], "sha": T.sha(img[:, :wb])}
    return out


@pytest.mark.parametrize("name", DITHER_NAMES)
def test_dither_restatement_vs_live_reference(name):
    want = T.reference_calls("oracle_dither")
    data = T.image(name)
    for key, mode, arith, pt, opt, w, h, wb in _dither_cases(name):
        g = want[key]
        rc2, out = T.oracle_decode(data, pt, opt, arith, w, h)
        assert g["rc"] == rc2 == 1
        assert T.sha(out[:g["rows"], :wb]) == g["sha"], key


def _synthetic_format_cases():
    """4:2:2, 4:4:4, grayscale, no-restart odd-sized 4:2:0: bundled images do not cover them."""
    from tests import synth
    return {"gray": (synth.synth_jpeg(320, 200, 1, 75, gray=True), 320, 200),
            "s444": (synth.synth_jpeg(173, 131, 2, 80, subsampling="4:4:4"), 173, 131),
            "s422": (synth.synth_jpeg(173, 131, 3, 80, subsampling="4:2:2"), 173, 131),
            "odd420": (synth.synth_jpeg(301, 203, 4, 90, restart_rows=0), 301, 203)}


def _synthetic_format_keys(cases):
    for mode, arith in MODES:
        for n in cases:
            for pt, ptn in T.PTS:
                if n == "gray" and pt == 2:
                    continue  # reference writes 16-bit pixels into a 32-bit buffer here (JPEGPutMCUGray): undefined
                for opt, sn in T.SCALES:
                    yield "%s/%s/%s/%s" % (mode, n, ptn, sn), mode, arith, n, pt, opt


def record_synthetic_formats(refs):
    cases = _synthetic_format_cases()
    out = {"input/" + n: {"input": T.sha(np.frombuffer(d, dtype=np.uint8))} for n, (d, w, h) in cases.items()}
    for key, mode, arith, n, pt, opt in _synthetic_format_keys(cases):
        data, w, h = cases[n]
        rc0, inf = refs[mode].info(data)
        assert (inf.width, inf.height) == (w, h)
        rc, err, img, _ = refs[mode].decode_cb(data, pt, opt, want_log=False)
        out[key] = {"rc": rc, "shape": list(img.shape), "sha": T.sha(img)}
    return out


def test_synthetic_formats_vs_live_reference():
    """4:2:2, 4:4:4, grayscale, no-restart odd-sized 4:2:0: the C restatement and the kernel stepper against what the
    compiled reference returned for the same files."""
    want = T.reference_calls("oracle_synthetic")
    cases = _synthetic_format_cases()
    for n, (data, w, h) in cases.items():
        T.check_input(want["input/" + n], data, n)
    for key, mode, arith, n, pt, opt in _synthetic_format_keys(cases):
        data, w, h = cases[n]
        g = want[key]
        rc1, o1 = T.oracle_decode(data, pt, opt, arith, w, h)
        rc2, o2, _ = T.hostsim_decode(data, pt, opt, arith, w, h)
        assert g["rc"] == rc1 == rc2 == 1
        assert list(o1.shape) == g["shape"] and T.sha(o1) == g["sha"], key
        assert list(o2.shape) == g["shape"] and T.sha(o2) == g["sha"], key


@pytest.mark.parametrize("name", ["sciopero", "st_peters", "zebra", "octocat_small", "batman", "ncc1701", "lange"])
def test_chunk_parallel_decode_of_restart_free_scans(name):
    """SURVEY.md 8(f)2: scans without restart markers go through jd_chunk.h (speculative chunk parse to a fix point,
    prefix sums, emit, phase/DC stitch).  Same digests as the reference, and the entry states settle in a few passes."""
    d = T.digests()[name]
    data = T.image(name)
    w, h = d["info"]["width"], d["info"]["height"]
    assert d["info"]["res_interval"] == 0
    for mode, arith in MODES:
        for pt, ptn in T.PTS:
            for opt, sn in ((0, "full"), (4, "quarter")):
                want = d["%s/%s/%s" % (mode, ptn, sn)]
                rc, out, nev = T.hostsim_decode(data, pt, opt, arith, w, h, chunked=True)
                assert rc == want["rc"] and T.sha(out) == want["sha"], (name, mode, ptn, sn)
    assert 2 <= T.hostsim().hostsim_last_chunk_iters() <= 8


def test_chunk_parallel_decode_synthetic_vs_restatement():
    from tests import synth
    cases = {"hd": (synth.synth_jpeg(1920, 1080, 9, 75, restart_rows=0), 1920, 1080),
             "gray": (synth.synth_jpeg(640, 360, 1, 75, gray=True, restart_rows=0), 640, 360),
             "s444": (synth.synth_jpeg(333, 251, 2, 96, subsampling="4:4:4", restart_rows=0), 333, 251),
             "s422": (synth.synth_jpeg(333, 251, 3, 80, subsampling="4:2:2", restart_rows=0), 333, 251)}
    for n, (data, w, h) in cases.items():
        for arith in (0, 1):
            rc1, want = T.oracle_decode(data, 0, 0, arith, w, h)
            rc2, got, _ = T.hostsim_decode(data, 0, 0, arith, w, h, chunked=True)
            assert rc1 == rc2 == 1 and np.array_equal(got, want), n
            assert T.hostsim().hostsim_last_chunk_iters() <= 8


def test_chunk_parallel_random_sweep_vs_restatement():
    """Seeded random restart-free files (size, quality 15..100, sampling, gray): the chunk-parallel path -- speculative parse
    passes, then jd_decode_segment started in the middle of the stream at each chunk's first block, whatever its position in the
    MCU -- against the sequential C restatement, pixel for pixel."""
    from tests import synth
    rng = np.random.default_rng(1234)
    for case in range(28):
        w, h = int(rng.integers(16, 360)), int(rng.integers(16, 260))
        q = int(rng.integers(15, 101))
        gray = bool(rng.integers(0, 5) == 0)
        sub = ["4:2:0", "4:2:2", "4:4:4", "4:2:0"][int(rng.integers(0, 4))]
        data = synth.synth_jpeg(w, h, 7000 + case, q, subsampling=sub, gray=gray, restart_rows=0)
        pt = 3 if gray else int(rng.integers(0, 3)) * (1 if rng.integers(0, 2) else 0)   # GRAY8 for gray files, else RGB565 LE / BE / RGB8888
        arith = int(rng.integers(0, 2))
        rc1, want = T.oracle_decode(data, pt, 0, arith, w, h)
        rc2, got, _ = T.hostsim_decode(data, pt, 0, arith, w, h, chunked=True)
        assert rc1 == rc2 == 1 and np.array_equal(got, want), (case, w, h, q, sub, gray, pt, arith, len(data))


def _odd_restart_cases():
    import io
    from PIL import Image
    from tests import synth
    img = Image.fromarray(synth.synth_pixels(333, 251, 7))
    out = {}
    for name, kw in [("dri1", dict(restart_marker_blocks=1)), ("dri7", dict(restart_marker_blocks=7)),
                     ("rows2", dict(restart_marker_rows=2)), ("q100", dict(restart_marker_rows=1, quality=100)),
                     ("q5", dict(restart_marker_rows=1, quality=5))]:
        b = io.BytesIO()
        k = dict(quality=80, subsampling="4:2:0")
        k.update(kw)
        img.save(b, "JPEG", **k)
        out[name] = b.getvalue()
    return out


def test_unusual_restart_intervals_and_qualities():
    """DRI = 1 MCU (a marker after every MCU), 7 MCUs (not a divisor of the row), 2 rows; q100 (>= 10-bit magnitudes -> pair
    records) and q5 (almost all blocks DC-only): restatement and kernel stepper agree on every pixel."""
    for n, data in _odd_restart_cases().items():
        for arith in (0, 1):
            for pt in (0, 2):
                for opt in (0, 2, 8):
                    rc1, want = T.oracle_decode(data, pt, opt, arith, 333, 251)
                    rc2, got, _ = T.hostsim_decode(data, pt, opt, arith, 333, 251)
                    assert rc1 == rc2 == 1 and np.array_equal(got, want), (n, arith, pt, opt)


PROG = ["prog_420", "prog_420_dri", "prog_444", "prog_422", "prog_gray"]


@pytest.mark.parametrize("name", PROG)
def test_progressive_dc_thumbnail_restatement_and_kernel_stepper(name):
    """SURVEY.md 8(f)4: progressive files -> DC coefficients of the first scan -> 1/8 image (reference
    JPEGDecodeMCU_P src/jpeg.inl:1819-1884, forced JPEG_SCALE_EIGHTH :4964-4966).  The C restatement and the per-thread
    device code stepped on the CPU must both reproduce the digests recorded from the compiled reference."""
    import json
    import os
    g = json.load(open(os.path.join(T.GOLD, "progressive.json")))[name]
    data = T.image(name)
    for mode, arith in (("sse", 0), ("scalar", 1)):
        for pt, ptn in ((0, "565le"), (1, "565be"), (2, "8888")):
            key = "%s/%s/opt8" % (mode, ptn)
            if key not in g:
                continue
            assert g[key] == g["%s/%s/opt0" % (mode, ptn)]            # option 0 is forced to 1/8 by the reference
            rc, img = T.oracle_decode(data, pt, 8, arith, g["w"], g["h"])
            assert rc == 1 and list(img.shape) == g[key]["shape"] and T.sha(img) == g[key]["sha"], (name, key, "restatement")
            for opt in (0, 8):
                oh, pitch = T.tight_shape(g["w"], g["h"], pt, 8)
                rc, sim, nev = T.hostsim_decode(data, pt, opt | 8 if opt else 8, arith, g["w"], g["h"])
                assert rc == 1 and T.sha(sim) == g[key]["sha"], (name, key, "stepper")


def _seeded_sweep_cases():
    """120 seeded random files (size 8..260, quality 15..100, every sampling, gray, restart interval 0 / rows, baseline and
    progressive), each with a random arithmetic build, pixel type and scale."""
    from tests import synth
    rng = np.random.default_rng(20240923)
    for case in range(120):
        w, h = int(rng.integers(8, 261)), int(rng.integers(8, 261))
        q = int(rng.integers(15, 101))
        gray = bool(rng.integers(0, 5) == 0)
        sub = ["4:2:0", "4:2:2", "4:4:4"][int(rng.integers(0, 3))]
        rr = int(rng.integers(0, 3))
        prog = bool(rng.integers(0, 4) == 0)
        data = synth.synth_jpeg(w, h, 1000 + case, q, subsampling=sub, gray=gray, restart_rows=rr, progressive=prog)
        mode, arith = MODES[int(rng.integers(0, 2))]
        pts = [0, 1, 3] if gray else [0, 1, 2, 3]
        if prog:
            pts = [p for p in pts if p != 3]          # the reference crashes on progressive -> 8-bit gray
        pt = pts[int(rng.integers(0, len(pts)))]
        opt = 8 if prog else [0, 2, 4, 8][int(rng.integers(0, 4))]
        yield case, data, w, h, (q, sub, gray, rr, prog), mode, arith, pt, opt


def record_seeded_sweep(refs):
    out = {}
    for case, data, w, h, desc, mode, arith, pt, opt in _seeded_sweep_cases():
        rc, err, img, _ = refs[mode].decode_cb(data, pt, opt, want_log=False)
        assert rc == 1, (case, w, h, desc, err)
        out[str(case)] = {"input": T.sha(np.frombuffer(data, dtype=np.uint8)), "rc": rc, "shape": list(img.shape), "sha": T.sha(img)}
    return out


def test_seeded_random_sweep_vs_live_reference():
    """The seeded random files of _seeded_sweep_cases: the C restatement and the kernel stepper against what the compiled
    reference returned for them."""
    want = T.reference_calls("oracle_sweep")
    checked = 0
    for case, data, w, h, desc, mode, arith, pt, opt in _seeded_sweep_cases():
        g = want[str(case)]
        T.check_input(g, data, case)
        assert g["rc"] == 1
        rc1, o1 = T.oracle_decode(data, pt, opt, arith, w, h)
        rc2, o2, _ = T.hostsim_decode(data, pt, opt, arith, w, h)
        assert rc1 == 1 and rc2 == 1, (case, rc1, rc2)
        assert list(o1.shape) == g["shape"] and T.sha(o1) == g["sha"], ("restatement", case, w, h, desc, mode, pt, opt)
        assert list(o2.shape) == g["shape"] and T.sha(o2) == g["sha"], ("stepper", case, w, h, desc, mode, pt, opt)
        checked += 1
    assert checked == 120


def test_block_synchronous_walk_equals_the_flat_walk():
    """jd_decode_segment (jd_core.h: the block-synchronous entropy walk the kernels run, with the raw and with the un-stuffed
    CLEAN bit reader, fast 10-bit AC table, per-block capacity test) against jd_decode_segment_flat (one flat state machine per
    symbol): headers, records, window-phase maps, truncation events, status and failing MCU must be equal on every baseline
    fixture, on synthetic files of every sampling, and on corrupted scans."""
    import ctypes as C
    import glob
    import os
    from tests import synth
    L = T.hostsim()
    L.hostsim_walk_check.argtypes = [C.c_char_p, C.c_int] + [C.POINTER(C.c_int)] * 4
    files = {os.path.basename(f): open(f, "rb").read() for f in sorted(glob.glob(os.path.join(T.GOLD, "images", "*.jpg")))}
    files["hd"] = synth.synth_jpeg(1920, 1080, 3, 75)
    files["q98"] = synth.synth_jpeg(320, 240, 4, 98, restart_rows=0)
    files["q100"] = synth.synth_jpeg(160, 120, 8, 100)
    files["s422"] = synth.synth_jpeg(333, 251, 5, 85, subsampling="4:2:2", restart_rows=2)
    files["s444"] = synth.synth_jpeg(333, 251, 6, 60, subsampling="4:4:4")
    files["gray"] = synth.synth_jpeg(640, 360, 7, 75, gray=True)
    rng = np.random.default_rng(11)
    for k in range(40):                      # corrupted entropy data
        b = bytearray(files["tulips.jpg" if k % 2 else "sciopero.jpg"])
        for _ in range(3):
            b[int(rng.integers(700, len(b) - 2))] = int(rng.integers(0, 256))
        files["corrupt_scan_%d" % k] = bytes(b)
    checked = records = events = badsegs = 0
    for name, data in files.items():
        v = [C.c_int() for _ in range(4)]
        r = L.hostsim_walk_check(data, len(data), *[C.byref(x) for x in v])
        if r == -1:
            continue                          # header rejected / progressive: not this path
        assert r == 0, (name, r)
        checked += 1; records += v[1].value; events += v[2].value; badsegs += v[3].value
    assert checked >= 55 and records > 1000000 and events > 50 and badsegs > 0
