"""CPU tier: host logic of the product (no compute calls): C-ABI symbols, open() conformance against the
reference's recorded behaviour, crop snapping, table builders, loud failure without a GPU."""
import ctypes as C
import math
import os
import re

import numpy as np
import pytest

import jpegdec_b200 as J
from tests import common as T


def _declared_functions(header):
    txt = open(os.path.join(T.ROOT, "include", header)).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    txt = txt.split("#ifdef __cplusplus\n} /* extern")[0] if header == "JPEGDEC.h" else txt
    names = re.findall(r"^[A-Za-z_][A-Za-z0-9_ \*]*?\b((?:JPEG|JPEGB200)_[A-Za-z0-9_]+)\s*\(", txt, flags=re.M)
    return sorted(set(names))


@pytest.mark.parametrize("header", ["JPEGDEC.h", "jpegdec_b200.h"])
def test_every_declared_symbol_is_exported(header):
    L = C.CDLL(J.LIB_PATH)
    names = _declared_functions(header)
    assert len(names) >= 15
    for n in names:
        assert hasattr(L, n), "%s declared in include/%s but not exported" % (n, header)


def test_open_matches_reference_behaviour():
    d = T.digests()
    for name, rec in d.items():
        j = J.JPEGDEC()
        rc = j.openRAM(T.image(name))
        inf = rec["info"]
        assert rc == rec["open"], name
        if rc:
            assert (j.getWidth(), j.getHeight(), j.getSubSample(), j.getBpp()) == (
                inf["width"], inf["height"], inf["subsample"], inf["bpp"]), name
            assert j.getOrientation() == inf["orientation"]
            assert j.hasThumb() == inf["has_thumb"]
            assert (j.getThumbWidth(), j.getThumbHeight()) == (inf["thumb_w"], inf["thumb_h"])
            assert j.getLastError() == J.JPEG_SUCCESS
        else:
            assert j.getLastError() == inf["error"], name
        j.close()


def test_open_rejects_garbage():
    j = J.JPEGDEC()
    assert j.openRAM(b"\x00" * 100) == 0 and j.getLastError() == J.JPEG_INVALID_FILE      # < 256 bytes
    assert j.openRAM(b"\x12" * 1000) == 0 and j.getLastError() == J.JPEG_INVALID_FILE     # no SOI
    assert j.openRAM(b"\xff\xd8" + b"\xff\xc1" + b"\x00" * 600) == 0 and j.getLastError() == J.JPEG_UNSUPPORTED_FEATURE


def test_crop_snapping_known_answer():
    # reference test 2 (MacOS/JPEGDEC_Test/JPEGDEC_Test/main.cpp:106-137): (50,50,125,170) -> (48,48,128,176)
    j = J.JPEGDEC()
    assert j.openRAM(T.image("tulips"))
    j.setCropArea(50, 50, 125, 170)
    assert j.getCropArea() == (48, 48, 128, 176)
    j.setCropArea(-5, -5, 10000, 10000)
    x, y, w, h = j.getCropArea()
    assert (x, y) == (0, 0) and w == 640 - 16 and h == 480 - 16   # the reference's clamp (jpeg.inl:719-720)


def test_fuzzed_headers_never_crash():
    # reference tests 11-12 (main.cpp:262-300) at the open() level: byte inversions in the first 2000 bytes
    base = bytearray(T.image("tulips"))
    rng = np.random.default_rng(7)
    for i in list(range(0, 700)) + list(rng.integers(700, 2000, 300)):
        b = bytearray(base)
        b[i] ^= 0xFF
        j = J.JPEGDEC()
        rc = j.openRAM(bytes(b))
        assert rc in (0, 1)
        assert 0 <= j.getLastError() <= J.JPEG_ERROR_MEMORY


def test_aan_prescale_table_from_formula():
    L = C.CDLL(J.LIB_PATH)
    L.jd_aan_table.restype = C.POINTER(C.c_int)
    tab = [L.jd_aan_table()[i] for i in range(64)]
    s = [1.0] + [math.cos(k * math.pi / 16) * math.sqrt(2) for k in range(1, 8)]
    for r in range(8):
        for c in range(8):
            assert abs(tab[r * 8 + c] - 16384 * s[r] * s[c]) <= 1.0, (r, c)


def test_decode_without_gpu_fails_loudly():
    if J.lib().JPEGB200_deviceCount() > 0:
        pytest.skip("a GPU is present")
    j = J.JPEGDEC()
    assert j.openRAM(T.image("tulips"))
    fb = np.zeros((496, 1280), np.uint8)
    j.setFramebuffer(fb)
    assert j.decode(0, 0, 0) == 0
    assert j.getLastError() == J.JPEG_ERROR_MEMORY
    assert not fb.any()                      # nothing was computed on the CPU
    with pytest.raises(RuntimeError):
        J.Context()


def test_table_blob_roundtrip_host_side():
    blob = np.zeros(J.TABLE_BLOB_BYTES, np.uint8)
    assert J.lib().JPEGB200_exportTables(T.image("tulips"), len(T.image("tulips")), blob.ctypes.data) == 1
    blob2 = np.zeros(J.TABLE_BLOB_BYTES, np.uint8)
    J.lib().JPEGB200_exportTables(T.image("croptest"), len(T.image("croptest")), blob2.ctypes.data)
    assert blob[:8].tobytes() != b"\0" * 8
    # standard Huffman tables in both files -> same LUT hash, different quant
    assert (blob[:8] == blob2[:8]).all() == (blob[16:16 + 12800] == blob2[16:16 + 12800]).all()


class _Geom(C.Structure):
    _fields_ = [(n, C.c_int) for n in ("width", "height", "crop_x", "crop_y", "crop_w", "crop_h", "x_off", "y_off",
                                       "subsample", "pixel_type", "options", "max_mcus")]


class _Item(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("mcu_row", "mcu_col0", "n_mcus", "x", "y", "w", "h", "w_used", "buf")]


def _schedule(geom):
    L = J.lib()
    L.jd_delivery_schedule.argtypes = [C.POINTER(_Geom), C.POINTER(_Item), C.c_int]
    n = L.jd_delivery_schedule(C.byref(geom), None, 0)
    items = (_Item * max(n, 1))()
    assert L.jd_delivery_schedule(C.byref(geom), items, n) == n
    return [(it.x, it.y, it.w, it.h, it.w_used, it.buf) for it in items[:n]]


def test_delivery_schedule_equals_the_reference_callback_sequence():
    """The draw-callback geometry (jd_api.c jd_delivery_schedule: which MCUs go into which call, x / y / iWidth / iHeight /
    iWidthUsed, the JPEG_USES_DMA half) against the callback log of the compiled reference, WITHOUT a GPU: every fixture
    sampling x pixel type x scale x decode offset x setMaxOutputSize x crop -- including crop x scale, where the reference
    compares scaled MCU positions with the unscaled crop rectangle (SURVEY.md A.5: fewer rows at 1/2, no callbacks at 1/4
    and 1/8); reproduced literally (src/jpeg.inl:5062-5084, :5111, :5135, :5300-5336).  The reference's logs are recorded in
    tests/golden/reference/host_schedule.json: per fixture, one "rc err calls digest" entry per case, in case order."""
    want = T.reference_calls("host_schedule")
    checked = with_crop_scaled = 0
    for name, cases in _schedule_cases():
        assert len(cases) == len(want[name]), name
        for (data, w, h, sub, crop, pt, opt, xo, yo, maxm), rec in zip(cases, want[name]):
            rc, err, ncalls, digest = rec.split()
            rc, err, ncalls = int(rc), int(err), int(ncalls)
            assert rc in (0, 1)     # 0: the crop reaches below the image and the reference runs out of data
            j2 = J.JPEGDEC()
            assert j2.openRAM(data)
            if crop is not None:
                j2.setCropArea(*crop)
            cx, cy, cw, ch = j2.getCropArea()
            g = _Geom(w, h, cx, cy, cw, ch, xo, yo, sub, pt, opt, maxm if maxm else 1000)
            got = _schedule(g)
            if rc == 0:
                assert err == J.JPEG_DECODE_ERROR and cy + ch > h
                got = got[:ncalls]     # the calls made before the reference failed
            assert len(got) == ncalls and T.log_sha(got) == digest, (name, crop, pt, opt, xo, yo, maxm, got[:3])
            checked += 1
            with_crop_scaled += int(crop is not None and (opt & 14) != 0)
    assert checked > 1500 and with_crop_scaled > 300


def _schedule_cases():
    """[(fixture, [(data, w, h, subsampling, crop, pixel type, options, x offset, y offset, setMaxOutputSize)])]: every fixture
    sampling x pixel type x scale x decode offset x setMaxOutputSize x crop, with four seeded random crops per fixture"""
    rng = np.random.default_rng(5)
    out = []
    for name in ("tulips", "zebra", "ncc1701", "sciopero", "lange", "croptest", "octocat_small"):
        data = T.image(name)
        j = J.JPEGDEC()
        assert j.openRAM(data)
        w, h, sub = j.getWidth(), j.getHeight(), j.getSubSample()
        j.close()
        crops = [None, (50, 50, 125, 170), (96, 64, 256, 192), (0, 0, 64, 64), (16, 32, 100, 40)]
        crops += [(int(rng.integers(0, w)), int(rng.integers(0, h)), int(rng.integers(1, w)), int(rng.integers(1, h))) for _ in range(4)]
        cases = []
        for crop in crops:
            if crop is not None and (crop[0] + 16 >= w or crop[1] + 16 >= h):
                continue
            for pt in (0, 2, 3):
                for opt in (0, 2, 4, 8, J.JPEG_USES_DMA, 2 | J.JPEG_USES_DMA):
                    for (xo, yo, maxm) in ((0, 0, 0), (7, 3, 0), (0, 0, 3)):
                        if crop is not None and (xo or maxm) and opt:
                            continue
                        cases.append((data, w, h, sub, crop, pt, opt, xo, yo, maxm))
        out.append((name, cases))
    return out


def record_schedule(refs):
    out = {}
    for name, cases in _schedule_cases():
        out[name] = []
        for data, w, h, sub, crop, pt, opt, xo, yo, maxm in cases:
            rc, err, img, log = refs["sse"].decode_cb(data, pt, opt, xoff=xo, yoff=yo, crop=crop, max_mcus=maxm)
            calls = [(r[0], r[1], r[2], r[3], r[4], r[6]) for r in log]
            out[name].append("%d %d %d %s" % (rc, err, len(calls), T.log_sha(calls)))
    return out


def test_bench_reference_arm_line_has_the_contract_keys():
    """`bench.py --impl reference` (the reference's own CPU path on the host cores) needs no GPU: run one step here and check
    the JSON line it prints.  It times the reference itself, so it runs where build() could compile it into oracle/_ref."""
    import json, subprocess, sys
    from oracle import refdrv
    if not refdrv.available("sse"):
        pytest.skip("the reference build oracle/_ref/libjpegdec_ref_sse.so is not present")
    r = subprocess.run([sys.executable, os.path.join(T.ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-1500:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1                       # ONE JSON line
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["unit"] == "Mpixels/s" and d["higher_is_better"] is True and d["value"] > 0
    assert "workload" in d["config"] and d["steps"] == 1
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and cb["sample"] and abs(cb["value"] - d["value"]) < 1e-6 * d["value"] + 1e-9
    e = d["e2e"]
    assert e["h2d_bytes_per_step"] == 0 and e["d2h_bytes_per_step"] == 0 and e["unit"] == d["unit"] and abs(e["value"] - d["value"]) < 1e-6 * d["value"] + 1e-9
