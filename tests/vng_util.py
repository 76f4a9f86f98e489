"""Helpers for the VNG4 / dual-demosaic tests: the oracle (oracle/restate/vng_oracle.c), the reference's own lines compiled
in place (oracle/_ref: ref_vng.c, a serial build -- see its header) and the product's kernels run on the CPU
(tests/emul/emul_vng.cpp).  Checkers only."""
import ctypes as C
import os
import subprocess

import numpy as np

import util

EMUL = os.path.join(os.path.dirname(os.path.abspath(__file__)), "emul")
WB = (2.0, 1.0, 1.5, 0.0)

CASES = {
    # name: (width, height, roi x, roi y, Bayer pattern)
    "rggb": (134, 78, 0, 0, "RGGB"),
    "bggr_roi": (131, 77, 1, 1, "BGGR"),
    "grbg_roi": (64, 48, 3, 2, "GRBG"),
    "gbrg_wide": (300, 17, 2, 5, "GBRG"),
    "smallest_dual": (16, 16, 0, 0, "RGGB"),
}


def case(name):
    w, h, x, y, pat = CASES[name]
    m = util.frame_natural(w, h, 6, filters=util.BAYER[pat])
    if h > 40:
        m[5, 5], m[20, 8] = np.nan, 0.0
        m[30:34, 30:34] = 0.25           # a flat patch: all gradients zero, the bilinear pixel stays
    return m, util.BAYER[pat], x, y


def _vng(lib, fn, m, filters, x, y, lin=0):
    h, w = m.shape
    out, src = util.aligned_empty((h, w, 4)), util.aligned_empty(m.shape)
    out[...] = -7.0
    src[...] = m
    f = getattr(lib, fn)
    f.restype = C.c_int
    f.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_uint32, C.c_int]
    assert f(out.ctypes.data, src.ctypes.data, w, h, x, y, filters, lin) == 0
    return np.array(out)


def oracle_vng(m, filters, x=0, y=0, lin=0):
    return _vng(util.oracle(), "orc_vng_interpolate", m, filters, x, y, lin)


@util.recorded(lambda m, filters, x=0, y=0, lin=0, kind="strict": oracle_vng(m, filters, x, y, lin))
def ref_vng(m, filters, x=0, y=0, lin=0, kind="strict"):
    lib = util.ref(kind)
    return None if lib is None else _vng(lib, "ref_vng_interpolate", m, filters, x, y, lin)


def _dual(lib, fn, rgb, m, filters, x, y, thr, mask=0):
    h, w = m.shape
    out, src = util.aligned_empty((h, w, 4)), util.aligned_empty(m.shape)
    out[...] = rgb
    src[...] = m
    f = getattr(lib, fn)
    f.restype = C.c_int
    f.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_uint32, C.c_void_p, C.c_float, C.c_int]
    assert f(out.ctypes.data, src.ctypes.data, w, h, x, y, filters, (C.c_float * 4)(*WB), thr, mask) == 0
    return np.array(out)


def oracle_dual(rgb, m, filters, x, y, thr, mask=0):
    return _dual(util.oracle(), "orc_dual_demosaic", rgb, m, filters, x, y, thr, mask)


@util.recorded(lambda rgb, m, filters, x, y, thr, mask=0, kind="strict": oracle_dual(rgb, m, filters, x, y, thr, mask))
def ref_dual(rgb, m, filters, x, y, thr, mask=0, kind="strict"):
    lib = util.ref(kind)
    return None if lib is None else _dual(lib, "ref_dual_demosaic", rgb, m, filters, x, y, thr, mask)


def sharp_frame(m, filters, x=0, y=0):
    """the frame the dual blend starts from: RCD of the mosaic (undefined RCD pixels zeroed so that every checker sees the same input)"""
    import ansel_b200 as ab
    rf = ab.lib().b200_roi_filters(C.c_uint32(filters), x, y)
    return np.nan_to_num(util.oracle_rcd(np.nan_to_num(m), rf))


def emul_lib():
    so = os.path.join(EMUL, "libemul_vng.so")
    srcs = [os.path.join(EMUL, "emul_vng.cpp"), os.path.join(EMUL, "cuda_on_cpu.h"), os.path.join(util.ROOT, "ansel_b200", "csrc", "vng.cu")]
    if not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in srcs):
        subprocess.run(["g++", "-O1", "-std=c++17", "-fno-fast-math", "-ffp-contract=off", "-I", EMUL, "-shared", "-fPIC", "-o", so, srcs[0]], check=True)
    return C.CDLL(so)


def emul_vng(m, filters, x=0, y=0, lin=0):
    return _vng(emul_lib(), "emul_vng", m, filters, x, y, lin)


_SMOOTH = C.CFUNCTYPE(None, C.c_void_p, C.c_int, C.c_int, C.c_int)


def emul_dual(rgb, m, filters, x, y, thr):
    h, w = m.shape
    out, src = util.aligned_empty((h, w, 4)), util.aligned_empty(m.shape)
    out[...] = rgb
    src[...] = m
    o = util.oracle()
    smooth = _SMOOTH(lambda p, ww, hh, n: o.orc_color_smoothing(C.c_void_p(p), ww, hh, n))
    f = emul_lib().emul_dual
    f.restype = C.c_int
    f.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_uint32, C.c_void_p, C.c_float, _SMOOTH]
    assert f(out.ctypes.data, src.ctypes.data, w, h, x, y, filters, (C.c_float * 4)(*WB), thr, smooth) == 0
    return np.array(out)


# ---- X-Trans (filters == 9): three colours, lane 3 is not a result ----------------------------------------------------------
XTRANS = np.array([[1, 1, 0, 1, 1, 2], [1, 1, 2, 1, 1, 0], [2, 0, 1, 0, 2, 1], [1, 1, 2, 1, 1, 0], [1, 1, 0, 1, 1, 2], [0, 2, 1, 2, 0, 1]], np.uint8)
XTRANS_CASES = {"origin": (134, 78, 0, 0), "roi": (131, 77, 1, 4), "roi2": (64, 48, 3, 2), "small": (30, 17, 5, 5)}


def xtrans_case(name):
    w, h, x, y = XTRANS_CASES[name]
    m = util.frame_natural(w, h, 6)
    if h > 40:
        m[5, 5], m[20, 8] = np.nan, 0.0
        m[30:36, 30:36] = 0.25
    return m, x, y


def _vng_xtrans(lib, fn, m, x, y, lin=0, extra=()):
    h, w = m.shape
    out, src = util.aligned_empty((h, w, 4)), util.aligned_empty(m.shape)
    out[...] = -7.0
    src[...] = m
    xt = np.ascontiguousarray(XTRANS)
    f = getattr(lib, fn)
    f.restype = C.c_int
    f.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int] + [C.c_uint32] * len(extra) + [C.c_void_p, C.c_int]
    assert f(out.ctypes.data, src.ctypes.data, w, h, x, y, *extra, xt.ctypes.data, lin) == 0
    return np.array(out)


def oracle_vng_xtrans(m, x=0, y=0, lin=0):
    return _vng_xtrans(util.oracle(), "orc_vng_interpolate_xtrans", m, x, y, lin)


@util.recorded(lambda m, x=0, y=0, lin=0, kind="strict": oracle_vng_xtrans(m, x, y, lin))
def ref_vng_xtrans(m, x=0, y=0, lin=0, kind="strict"):
    lib = util.ref(kind)
    return None if lib is None else _vng_xtrans(lib, "ref_vng_interpolate_xtrans", m, x, y, lin)


def emul_vng_xtrans(m, x=0, y=0, lin=0):
    return _vng_xtrans(emul_lib(), "emul_vng_cfa", m, x, y, lin, extra=(9,))
