"""CPU tier: single 8x8 blocks through (a) the reference's own JPEGIDCT (static function, reachable inside
oracle/ref_shim.c's TU; its outputs recorded as digests in tests/golden/reference/idct_blocks.json), (b) the C restatement, (c) the per-thread code the CUDA kernel executes (tests/hostsim) --
random sparse blocks including extreme coefficient x quant products that exercise the int16 wrap-around of the SSE2
build and the two corner cases the kernel's unified column pass patches."""
import ctypes as C
import os

import numpy as np
import pytest

from tests import common as T

ZZ = [0, 1, 8, 16, 9, 2, 3, 10, 17, 24, 32, 25, 18, 11, 4, 5, 12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13, 6, 7, 14, 21, 28,
      35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63]


def _flags(coef):
    f = 0
    for n in range(1, 64):
        if coef[n] != 0:
            f |= (1 << (n & 7)) | (n << 8)
    return f & 0xFFFF


def _blocks(rng, n):
    for it in range(n):
        kind = it % 6
        coef = np.zeros(64, np.int16)
        quant = np.ones(64, np.int16)
        if kind == 5:  # corner cases of the unified column pass: s2(d3) == -32768, |d2| >= 8192, rows 4-7 empty
            c = int(rng.integers(0, 8))
            coef[0] = int(rng.integers(-500, 500)); quant[0] = int(rng.integers(1, 100))
            d3 = 0x2000 + int(rng.integers(-3, 4)) * 0x4000
            coef[24 + c] = np.int16(((d3 + 32768) % 65536) - 32768)
            coef[16 + c] = np.int16(int(rng.integers(-2047, 2048)) or 1); quant[16 + c] = np.int16(int(rng.integers(1, 32767)))
            coef[8 + c] = np.int16(int(rng.integers(-2047, 2048)) or 1); quant[8 + c] = np.int16(int(rng.integers(1, 2000)))
        else:
            nnz = int(rng.integers(1, 20)) if kind < 3 else int(rng.integers(1, 64))
            maxk = int(rng.integers(2, 64)) if kind != 1 else int(rng.integers(2, 12))
            amp = [30, 200, 1023, 1023, 2047][kind]
            for k in rng.choice(np.arange(1, maxk + 1), size=min(nnz, maxk), replace=False):
                coef[ZZ[k]] = int(rng.integers(-amp, amp + 1)) or 1
            coef[0] = int(rng.integers(-1024, 1024))
            qmax = [40, 255, 255, 4000, 32767][kind]
            quant = rng.integers(1, qmax + 1, size=64).astype(np.int16)
            if kind == 4:
                quant = rng.integers(-32768, 32767, size=64).astype(np.int16)
        fl = _flags(coef)
        if fl:
            yield coef, quant, fl


def record_idct_blocks(refs):
    """digest of the reference's JPEGIDCT output for every block of the test's seeded sequence, per arithmetic build"""
    libs = [C.CDLL(os.path.join(T.ROOT, "oracle", "_ref", "libjpegdec_ref_%s.so" % m)) for m in ("sse", "scalar")]
    outs = ([], [])
    for coef, quant, fl in _blocks(np.random.default_rng(11), 12000):
        for arith in (0, 1):
            o_ref = np.zeros(64, np.uint8)
            libs[arith].ref_idct(coef.ctypes.data, quant.ctypes.data, fl, 0, o_ref.ctypes.data)
            outs[arith].append(o_ref)
    return {"sse": T.sha(np.concatenate(outs[0])), "scalar": T.sha(np.concatenate(outs[1]))}


def test_idct_blocks_reference_restatement_kernelcode():
    orc = T.oracle()
    sim = T.hostsim()
    want = T.reference_calls("idct_blocks")
    outs = ([], [])
    rng = np.random.default_rng(11)
    n = 0
    for coef, quant, fl in _blocks(rng, 12000):
        for arith in (0, 1):
            o_or = np.zeros(64, np.uint8); o_sim = np.zeros(64, np.uint8)
            orc.oracle_idct(coef.ctypes.data, quant.ctypes.data, fl, arith, 0, o_or.ctypes.data)
            sim.hostsim_idct(coef.ctypes.data, quant.ctypes.data, fl, arith, o_sim.ctypes.data)
            assert np.array_equal(o_or, o_sim), (arith, hex(fl))
            if arith == 0:      # the packed thread-per-block code of jdk_idct_p, both instantiations
                o_p = np.zeros(64, np.uint8); o_g = np.zeros(64, np.uint8)
                sim.hostsim_idct_packed(coef.ctypes.data, quant.ctypes.data, fl, o_p.ctypes.data)
                sim.hostsim_idct_packed_general(coef.ctypes.data, quant.ctypes.data, fl, o_g.ctypes.data)
                assert np.array_equal(o_or, o_p), ("packed", hex(fl))
                assert np.array_equal(o_or, o_g), ("packed general", hex(fl))
            outs[arith].append(o_or)
            n += 1
    assert n > 20000
    # the restatement's blocks, in order, are the reference's (tests/golden/reference/idct_blocks.json)
    assert T.sha(np.concatenate(outs[0])) == want["sse"]
    assert T.sha(np.concatenate(outs[1])) == want["scalar"]
