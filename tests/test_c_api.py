"""The drop-in boundary from C and C++: programs written like the reference's own examples
(linux/examples/c_cmdline/main.c, linux/examples/jpeg_perf_test/main.cpp) compile against include/JPEGDEC.h and
link against libjpegdec_b200.so.  CPU tier: they build, open() works, decode fails loudly without a GPU.
GPU tier: their output is bit-exact with the compiled reference."""
import os
import subprocess

import numpy as np
import pytest

import jpegdec_b200 as J
from tests import common as T

HERE = os.path.join(T.ROOT, "tests", "c_api")
OUT = os.path.join(HERE, "_build")
LIBDIR = os.path.join(T.ROOT, "jpegdec_b200")


def _build():
    os.makedirs(OUT, exist_ok=True)
    common = ["-O2", "-Wall", "-I" + os.path.join(T.ROOT, "include")]
    link = ["-L" + LIBDIR, "-ljpegdec_b200", "-Wl,-rpath," + LIBDIR]
    subprocess.run(["gcc"] + common + [os.path.join(HERE, "accept.c"), "-o", os.path.join(OUT, "accept")] + link, check=True)
    subprocess.run(["g++"] + common + [os.path.join(HERE, "accept_cpp.cpp"), "-o", os.path.join(OUT, "accept_cpp")] + link, check=True)


def test_c_and_cpp_callers_build_and_fail_loudly_without_gpu():
    _build()
    img = os.path.join(T.GOLD, "images", "tulips.jpg")
    r = subprocess.run([os.path.join(OUT, "accept"), img, "0", "0"], stdout=subprocess.PIPE, text=True)
    assert "w=640 h=480 sub=0x22" in r.stdout
    if J.lib().JPEGB200_deviceCount() == 0:
        assert r.returncode == 3 and "err=5" in r.stdout          # JPEG_ERROR_MEMORY, nothing decoded on the CPU
    r = subprocess.run([os.path.join(OUT, "accept"), os.path.join(T.GOLD, "images", "corrupt1.jpg"), "0", "0"],
                       stdout=subprocess.PIPE, text=True)
    assert r.returncode == 2                                       # open fails like the reference (JPEG_DECODE_ERROR)


@pytest.mark.gpu
def test_c_and_cpp_callers_match_reference(tmp_path):
    from oracle import refdrv
    _build()
    ref = refdrv.Ref("sse") if refdrv.available("sse") else None
    img = os.path.join(T.GOLD, "images", "tulips.jpg")
    for pt, opt in ((0, 0), (2, 0), (3, 0)):
        out = str(tmp_path / ("o_%d_%d.raw" % (pt, opt)))
        r = subprocess.run([os.path.join(OUT, "accept"), img, str(pt), str(opt), out], stdout=subprocess.PIPE, text=True)
        assert r.returncode == 0, r.stdout
        got = np.fromfile(out, dtype=np.uint8)
        if ref is not None:
            rc, err, want, _ = ref.decode_cb(T.image("tulips"), pt, opt, want_log=False)
            assert np.array_equal(got, want.reshape(-1))
        else:
            assert T.sha(got.reshape(480, -1)) == T.digests()["tulips"]["sse/%s/full" % dict(T.PTS)[pt]]["sha"]
    r = subprocess.run([os.path.join(OUT, "accept"), img, "cb", "0"], stdout=subprocess.PIPE, text=True)
    assert r.returncode == 0 and "callbacks=150 pixels=307200" in r.stdout, r.stdout   # SURVEY.md appendix B
    r = subprocess.run([os.path.join(OUT, "accept_cpp"), img], stdout=subprocess.PIPE, text=True)
    assert r.returncode == 0 and r.stdout.count("rc=1") == 4, r.stdout


# ---- the reference's own programs, unmodified (SURVEY.md 8(f)3) ----
def _ref_examples():
    """Binaries built by oracle/ref_examples.py into oracle/_ref/examples.  Built here when the reference sources are present;
    elsewhere the ones build() made where they were present are used."""
    from oracle import ref_examples as B
    if B.available():
        B.build()
    names = ["ref_c_cmdline", "ref_perf_test", "ref_jpegdec_test"]
    paths = {n: os.path.join(B.OUT, n) for n in names}
    return paths if all(os.path.exists(p) for p in paths.values()) else None


def test_reference_programs_compile_unmodified_against_this_library():
    from oracle import ref_examples as B
    if not B.available():
        pytest.skip("reference sources not on this machine")
    ex = _ref_examples()
    assert ex is not None
    # the shadow tree holds links, not copies
    assert os.path.islink(os.path.join(B.SHADOW, "linux/examples/c_cmdline/main.c"))
    if J.lib().JPEGB200_deviceCount() == 0:
        r = subprocess.run([ex["ref_c_cmdline"], os.path.join(T.GOLD, "images", "tulips.jpg"), "/dev/null"],
                           stdout=subprocess.PIPE, text=True)
        assert r.returncode != 0 and "Decode failed" in r.stdout     # no CPU fallback behind the reference's API either


@pytest.mark.gpu
def test_reference_programs_run_on_the_gpu_and_match_the_reference_build(tmp_path):
    import hashlib
    import json
    ex = _ref_examples()
    if ex is None:
        pytest.skip("reference programs not built (build() makes them where the reference sources exist)")
    gold = json.load(open(os.path.join(T.GOLD, "ref_examples.json")))["fixtures"]
    for name, g in gold.items():
        bmp = str(tmp_path / (name + ".bmp"))
        r = subprocess.run([ex["ref_c_cmdline"], os.path.join(T.GOLD, "images", name + ".jpg"), bmp], stdout=subprocess.PIPE, text=True)
        assert r.returncode == 0, (name, r.stdout)
        data = open(bmp, "rb").read()
        assert len(data) == g["bmp_bytes"] and hashlib.sha256(data).hexdigest() == g["bmp_sha256"], name
    r = subprocess.run([ex["ref_c_cmdline"]], stdout=subprocess.PIPE, text=True)             # in-memory tulips, 4 scales
    assert r.returncode == 0 and all(s in r.stdout for s in ("full sized", "half sized", "quarter sized", "eighth sized")), r.stdout
    r = subprocess.run([ex["ref_perf_test"]], stdout=subprocess.PIPE, text=True)
    assert r.returncode == 0 and r.stdout.count("sized decode in") == 4, r.stdout
    r = subprocess.run([ex["ref_jpegdec_test"]], stdout=subprocess.PIPE, text=True, timeout=600)
    out = r.stdout
    assert r.returncode == 0 and "Total tests: 12" in out, out[-2000:]
    # every functional test of the reference's harness passes; its test 3 is a CPU timing heuristic (luma-only decode
    # must be >= 37.5 % faster than colour), which a launch-latency-bound single-image GPU decode does not satisfy
    for t in ("JPEG full image decode - PASSED", "JPEG DMA ping-pong buffer - PASSED", "JPEG EXIF Thumbnail - PASSED",
              "Single Byte Sequential Corruption Test - PASSED", "Multi-Byte Random Corruption Test - PASSED"):
        assert t in out, out[-3000:]
    assert out.count("JPEG full image decode - PASSED") == 2
    failed = int(out.split("passed,")[1].split("failed")[0])
    assert failed <= 1 and (failed == 0 or "JPEG color->gray image decode - FAILED" in out), out[-3000:]
