"""Helpers of the LMMSE tests: the reference's lines (oracle/_ref, compiled without OpenMP), the oracle in its two modes, cases."""
import ctypes as C

import numpy as np

import util

CASES = {"rggb": (300, 260, "RGGB"), "bggr_odd": (263, 151, "BGGR"), "grbg_one_tile": (128, 128, "GRBG"), "gbrg_small": (40, 33, "GBRG"), "rggb_wide": (500, 70, "RGGB")}
PMAX = (1.0, 0.9, 1.1)


def case(name, seed=7):
    w, h, pat = CASES[name]
    m = util.frame_natural(w, h, seed, filters=util.BAYER[pat])
    if h > 60:
        m[20, 8] = 0.0
        m[30:42, 30:42] = 0.25
        m[50:56, 10:22] = 1.4          # beyond the table: calc_gamma clips
        m[5, 5] = -0.1
    return np.ascontiguousarray(m, np.float32), util.BAYER[pat]


def _run(lib, fn, m, filters, mode, extra=()):
    h, w = m.shape
    out, src = util.aligned_empty((h, w, 4)), util.aligned_empty(m.shape)
    out[...] = -7.0
    src[...] = m
    f = getattr(lib, fn)
    f.restype = None
    f.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_uint32, C.c_int, C.POINTER(C.c_float)] + [C.c_int] * len(extra)
    f(out.ctypes.data, src.ctypes.data, w, h, filters, mode, (C.c_float * 3)(*PMAX), *extra)
    return np.array(out)


def oracle(m, filters, mode, carry=0):
    return _run(util.oracle(), "orc_lmmse", m, filters, mode, (carry,))


@util.recorded(lambda m, filters, mode, kind="strict": oracle(m, filters, mode, carry=1))
def ref(m, filters, mode, kind="strict"):
    lib = util.ref(kind)
    return None if lib is None else _run(lib, "ref_lmmse", m, filters, mode)


_EMUL = None


def emul(m, filters, mode, nthreads=96, ascending=0):
    """ansel_b200/csrc/lmmse.cu compiled with g++ (tests/emul/emul_lmmse.cpp): the stages thread by thread, tile after tile"""
    global _EMUL
    if _EMUL is None:
        import os
        import subprocess
        here = os.path.join(os.path.dirname(os.path.abspath(__file__)), "emul")
        so = os.path.join(here, "libemul_lmmse.so")
        srcs = [os.path.join(here, "emul_lmmse.cpp"), os.path.join(here, "cuda_on_cpu.h"), os.path.join(here, "..", "..", "ansel_b200", "csrc", "lmmse.cu")]
        if not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in srcs):
            subprocess.run(["g++", "-O1", "-std=c++17", "-fno-fast-math", "-ffp-contract=off", "-I", here, "-shared", "-fPIC", "-o", so, srcs[0]], check=True)
        _EMUL = C.CDLL(so)
    h, w = m.shape
    out, src = util.aligned_empty((h, w, 4)), util.aligned_empty(m.shape)
    out[...] = -7.0
    src[...] = m
    f = _EMUL.emul_lmmse
    f.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_uint32, C.c_int, C.POINTER(C.c_float), C.c_int, C.c_int]
    assert f(out.ctypes.data, src.ctypes.data, w, h, filters, mode, (C.c_float * 3)(*PMAX), nthreads, ascending) == 0
    return np.array(out)
