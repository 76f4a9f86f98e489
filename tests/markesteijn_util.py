"""Helpers of the Markesteijn (X-Trans) tests: the reference's lines (oracle/_ref), the oracle, the CUDA path."""
import ctypes as C

import numpy as np

import util
from vng_util import XTRANS

CASES = {"origin": (300, 210, 0, 0), "roi": (131, 127, 1, 4), "roi2": (264, 148, 3, 2), "one_tile": (98, 98, 0, 0), "narrow": (40, 230, 5, 5),
         "small": (30, 17, 2, 3)}


def case(name, seed=6):
    w, h, x, y = CASES[name]
    m = util.frame_natural(w, h, seed)
    if h > 60 and w > 60:
        m[20, 8] = 0.0
        m[30:42, 30:42] = 0.25     # a flat patch
        m[50:60, 10:22] = 0.0      # a black patch: the maxima of green are 0.0f, the loop's marker of a new pair
    return np.ascontiguousarray(m, np.float32), x, y


def _call(lib, fn, m, x, y, passes):
    h, w = m.shape
    out, src = util.aligned_empty((h, w, 4)), util.aligned_empty(m.shape)
    out[...] = -7.0
    src[...] = m
    xt = np.ascontiguousarray(XTRANS)
    f = getattr(lib, fn)
    f.restype = None
    f.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int]
    f(out.ctypes.data, src.ctypes.data, w, h, x, y, xt.ctypes.data, passes)
    return np.array(out)


def oracle(m, x=0, y=0, passes=1):
    return _call(util.oracle(), "orc_markesteijn", m, x, y, passes)


@util.recorded(lambda m, x=0, y=0, passes=1, kind="strict": oracle(m, x, y, passes))
def ref(m, x=0, y=0, passes=1, kind="strict"):
    lib = util.ref(kind)
    return None if lib is None else _call(lib, "ref_markesteijn", m, x, y, passes)


_EMUL = None


def emul_lib():
    """ansel_b200/csrc/markesteijn.cu compiled with g++ (tests/emul/emul_markesteijn.cpp)"""
    global _EMUL
    if _EMUL is None:
        import os
        import subprocess
        here = os.path.join(os.path.dirname(os.path.abspath(__file__)), "emul")
        so = os.path.join(here, "libemul_markesteijn.so")
        srcs = [os.path.join(here, "emul_markesteijn.cpp"), os.path.join(here, "cuda_on_cpu.h"),
                os.path.join(here, "..", "..", "ansel_b200", "csrc", "markesteijn.cu")]
        if not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in srcs):
            subprocess.run(["g++", "-O1", "-std=c++17", "-fno-fast-math", "-ffp-contract=off", "-I", here, "-shared", "-fPIC", "-o", so, srcs[0]], check=True)
        _EMUL = C.CDLL(so)
    return _EMUL


def emul(m, x=0, y=0, nthreads=96, ascending=0, passes=1):
    """the kernel's stages run thread by thread on the CPU, the threads of a stage in descending (or ascending) order"""
    h, w = m.shape
    out, src = util.aligned_empty((h, w, 4)), util.aligned_empty(m.shape)
    out[...] = -7.0
    src[...] = m
    xt = np.ascontiguousarray(XTRANS)
    f = emul_lib().emul_markesteijn
    f.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int]
    assert f(out.ctypes.data, src.ctypes.data, w, h, x, y, xt.ctypes.data, nthreads, ascending, passes) == 0
    return np.array(out)


def emul_classes(w, h, x, y, xtrans=None, passes=1):
    xt = np.ascontiguousarray(XTRANS if xtrans is None else xtrans)
    f = emul_lib().emul_markesteijn_classes
    f.argtypes = [C.c_int] * 4 + [C.c_void_p, C.c_int]
    return f(w, h, x, y, xt.ctypes.data, passes)
