"""Shared helpers for the tests (test infrastructure)."""
import ctypes as C
import hashlib
import json
import os

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")
VALID = ["tulips", "st_peters", "sciopero", "zebra", "croptest", "octocat_small", "batman", "ncc1701", "lange"]
PTS = [(0, "rgb565le"), (1, "rgb565be"), (2, "rgb8888"), (3, "gray8")]
SCALES = [(0, "full"), (2, "half"), (4, "quarter"), (8, "eighth")]
DITHERS = [(6, "dither1"), (5, "dither2"), (4, "dither4")]


def image(name):
    return open(os.path.join(GOLD, "images", name + ".jpg"), "rb").read()


def digests():
    return json.load(open(os.path.join(GOLD, "digests.json")))


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()[:16]


def log_sha(log):
    """digest of a draw-callback log (a list of equal-length integer tuples)"""
    return sha(np.asarray(log, dtype=np.int64))


def reference_calls(name):
    """What the compiled reference returned for the calls one test compares with: {case key: record of digests}
    (tests/golden/reference/<name>.json, written by tests/golden/make_reference_golden.py)."""
    return json.load(open(os.path.join(GOLD, "reference", name + ".json")))


def check_input(rec, data, what):
    """synthetic inputs are re-encoded at test time: they must be the bytes the golden record was made from"""
    assert sha(np.frombuffer(data, dtype=np.uint8)) == rec["input"], \
        "%s: synthetic JPEG differs from the one the reference was run on (Pillow / OpenCV encoder changed?)" % (what,)


def bpp_of(pt):
    return {0: 16, 1: 16, 2: 32, 3: 8, 4: 4, 5: 2, 6: 1}[pt]


def tight_shape(w, h, pt, opt):
    s = 1 if opt & 2 else 2 if opt & 4 else 3 if opt & 8 else 0
    ow, oh = (w + (1 << s) - 1) >> s, (h + (1 << s) - 1) >> s
    return oh, (ow * bpp_of(pt) + 7) // 8


_oracle = None


def oracle():
    global _oracle
    if _oracle is None:
        L = C.CDLL(os.path.join(ROOT, "oracle", "liboracle.so"))
        L.oracle_decode.argtypes = [C.c_char_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int,
                                    C.POINTER(C.c_int), C.POINTER(C.c_int)]
        _oracle = L
    return _oracle


def oracle_decode(data, pt, opt, arith, w, h):
    """C restatement -> tight image [oh, pitch]."""
    oh, pitch = tight_shape(w, h, pt, opt)
    if pt >= 4:  # dithered rows are as wide as the MCU-aligned image in the reference's callback
        pitch = ((w + 31) * bpp_of(pt) + 7) // 8
    out = np.zeros((oh, pitch), dtype=np.uint8)
    ow, ohh = C.c_int(), C.c_int()
    rc = oracle().oracle_decode(data, len(data), pt, opt, arith, out.ctypes.data, pitch, C.byref(ow), C.byref(ohh))
    return rc, out


_sim = None


def hostsim():
    global _sim
    if _sim is None:
        L = C.CDLL(os.path.join(ROOT, "tests", "hostsim", "_build", "libhostsim.so"))
        L.hostsim_decode.argtypes = [C.c_char_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int] + [C.POINTER(C.c_int)] * 4
        L.hostsim_open.argtypes = [C.c_char_p, C.c_int] + [C.POINTER(C.c_int)] * 9
        L.hostsim_last_chunk_iters.restype = C.c_int
        L.hostsim_last_chunk_dc_mismatch.restype = C.c_int
        _sim = L
    return _sim


def hostsim_decode(data, pt, opt, arith, w, h, chunked=False, clean=False):
    """chunked=True forces the restart-free chunk-parallel path (jd_chunk.h) for scans without restart markers;
    clean=True un-stuffs each restart segment first and decodes it with the CLEAN bit reader (the GPU default)."""
    oh, pitch = tight_shape(w, h, pt, opt)
    if chunked:
        opt |= 0x20000
    if clean:
        opt |= 0x40000
    out = np.zeros((oh, pitch), dtype=np.uint8)
    v = [C.c_int() for _ in range(4)]
    rc = hostsim().hostsim_decode(data, len(data), pt, opt, arith, out.ctypes.data, pitch, *[C.byref(x) for x in v])
    return rc, out, v[2].value
