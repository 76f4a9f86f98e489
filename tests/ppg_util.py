"""Helpers for the PPG demosaicer's tests: the oracle (oracle/restate/ppg_oracle.c), the reference's own lines compiled
in place (oracle/_ref: ref_ppg.c) and the product's kernels run on the CPU (tests/emul/emul_ppg.cpp).  Checkers only."""
import ctypes as C
import os
import subprocess

import numpy as np

import util

EMUL = os.path.join(os.path.dirname(os.path.abspath(__file__)), "emul")
ALPHA_FILL = -7.0      # the reference leaves the alpha of the outer three pixels as it finds it

CASES = {
    # name: (width, height, Bayer pattern, median threshold, special samples)
    "rggb": (206, 120, "RGGB", 0.0, True),
    "bggr_median": (117, 131, "BGGR", 0.05, True),
    "grbg_median_wide": (300, 40, "GRBG", 0.5, False),
    "gbrg": (134, 78, "GBRG", 0.0, False),
    "smallest": (8, 9, "RGGB", 0.05, False),
    "sixteen": (16, 16, "GBRG", 0.0, False),
}


def case(name):
    w, h, pat, thrs, special = CASES[name]
    m = util.frame_natural(w, h, 3, filters=util.BAYER[pat])
    if special:
        m[5, 5], m[20, 8], m[7, 30], m[40, 41] = np.nan, np.inf, -1.0, 0.0
    return m, util.BAYER[pat], thrs


def _run(lib, fn, mosaic, filters, thrs):
    h, w = mosaic.shape
    out, src = util.aligned_empty((h, w, 4)), util.aligned_empty(mosaic.shape)
    out[...] = ALPHA_FILL
    src[...] = mosaic
    f = getattr(lib, fn)
    f.restype = C.c_int
    f.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_uint32, C.c_float]
    assert f(out.ctypes.data, src.ctypes.data, w, h, filters, thrs) == 0
    return np.array(out)


def oracle_ppg(mosaic, filters, thrs=0.0):
    return _run(util.oracle(), "orc_demosaic_ppg", mosaic, filters, thrs)


@util.recorded(lambda mosaic, filters, thrs=0.0, kind="strict": oracle_ppg(mosaic, filters, thrs))
def ref_ppg(mosaic, filters, thrs=0.0, kind="strict"):
    lib = util.ref(kind)
    return None if lib is None else _run(lib, "ref_demosaic_ppg", mosaic, filters, thrs)


def emul_lib(name="ppg"):
    so = os.path.join(EMUL, "libemul_%s.so" % name)
    srcs = [os.path.join(EMUL, "emul_%s.cpp" % name), os.path.join(EMUL, "cuda_on_cpu.h"), os.path.join(util.ROOT, "ansel_b200", "csrc", "%s.cu" % name)]
    if not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in srcs):
        subprocess.run(["g++", "-O1", "-std=c++17", "-fno-fast-math", "-ffp-contract=off", "-I", EMUL, "-shared", "-fPIC", "-o", so, srcs[0]], check=True)
    return C.CDLL(so)


def emul_ppg(mosaic, filters, thrs=0.0):
    return _run(emul_lib(), "emul_demosaic_ppg", mosaic, filters, thrs)


XTRANS = np.array([[1, 1, 0, 1, 1, 2], [1, 1, 2, 1, 1, 0], [2, 0, 1, 0, 2, 1], [1, 1, 2, 1, 1, 0], [1, 1, 0, 1, 1, 2], [0, 2, 1, 2, 0, 1]], np.uint8)


def _passthrough(lib, fn, mosaic, filters, x, y, colour):
    h, w = mosaic.shape
    out, src = util.aligned_empty((h, w, 4)), util.aligned_empty(mosaic.shape)
    out[...] = ALPHA_FILL
    src[...] = mosaic
    xt = np.ascontiguousarray(XTRANS)
    f = getattr(lib, fn)
    f.restype = C.c_int
    f.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_uint32, C.c_void_p, C.c_int]
    assert f(out.ctypes.data, src.ctypes.data, w, h, x, y, filters, xt.ctypes.data, colour) == 0
    return np.array(out)


def oracle_passthrough(m, filters, x=0, y=0, colour=0):
    return _passthrough(util.oracle(), "orc_demosaic_passthrough", m, filters, x, y, colour)


@util.recorded(lambda m, filters, x=0, y=0, colour=0, kind="strict": oracle_passthrough(m, filters, x, y, colour))
def ref_passthrough(m, filters, x=0, y=0, colour=0, kind="strict"):
    lib = util.ref(kind)
    return None if lib is None else _passthrough(lib, "ref_demosaic_passthrough", m, filters, x, y, colour)


def emul_passthrough(m, filters, x=0, y=0, colour=0):
    return _passthrough(emul_lib(), "emul_demosaic_passthrough", m, filters, x, y, colour)


def _downsample(lib, fn, mosaic, filters):
    h, w = mosaic.shape
    out, src = util.aligned_empty(((h + 1) // 2, (w + 1) // 2, 4)), util.aligned_empty(mosaic.shape)
    out[...] = ALPHA_FILL
    src[...] = mosaic
    f = getattr(lib, fn)
    f.restype = C.c_int
    f.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_uint32]
    assert f(out.ctypes.data, src.ctypes.data, w, h, filters) == 0
    return np.array(out)


def oracle_downsample(m, filters):
    return _downsample(util.oracle(), "orc_demosaic_downsample", m, filters)


@util.recorded(lambda m, filters, kind="strict": oracle_downsample(m, filters))
def ref_downsample(m, filters, kind="strict"):
    lib = util.ref(kind)
    return None if lib is None else _downsample(lib, "ref_demosaic_downsample", m, filters)


def emul_downsample(m, filters):
    return _downsample(emul_lib(), "emul_demosaic_downsample", m, filters)


def _downsample_xtrans(lib, fn, mosaic, x, y, xtrans):
    h, w = mosaic.shape
    out, src = util.aligned_empty(((h + 1) // 2, (w + 1) // 2, 4)), util.aligned_empty(mosaic.shape)
    out[...] = ALPHA_FILL
    src[...] = mosaic
    xt = np.ascontiguousarray(xtrans, np.uint8)
    f = getattr(lib, fn)
    f.restype = C.c_int
    f.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]
    assert f(out.ctypes.data, src.ctypes.data, w, h, x, y, xt.ctypes.data) == 0
    return np.array(out)


def oracle_downsample_xtrans(m, x, y, xtrans):
    return _downsample_xtrans(util.oracle(), "orc_demosaic_downsample_xtrans", m, x, y, xtrans)


@util.recorded(lambda m, x, y, xtrans, kind="strict": oracle_downsample_xtrans(m, x, y, xtrans))
def ref_downsample_xtrans(m, x, y, xtrans, kind="strict"):
    lib = util.ref(kind)
    return None if lib is None else _downsample_xtrans(lib, "ref_demosaic_downsample_xtrans", m, x, y, xtrans)


def emul_downsample_xtrans(m, x, y, xtrans):
    return _downsample_xtrans(emul_lib(), "emul_demosaic_downsample_xtrans", m, x, y, xtrans)


def _postfilter(lib, fn, rgba, iterations):
    h, w = rgba.shape[:2]
    buf = util.aligned_empty((h, w, 4))
    buf[...] = rgba
    f = getattr(lib, fn)
    f.restype = C.c_int
    f.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int]
    util.oracle().orc_fp_fast_mode_all()  # FTZ|DAZ on every worker thread, as the pipe's have it
    assert f(buf.ctypes.data, w, h, iterations) == 0
    return np.array(buf)


def oracle_postfilter(rgba, iterations):
    return _postfilter(util.oracle(), "orc_demosaic_downsample_postfilter", rgba, iterations)


@util.recorded(lambda rgba, iterations, kind="strict": oracle_postfilter(rgba, iterations))
def ref_postfilter(rgba, iterations, kind="strict"):
    lib = util.ref(kind)
    return None if lib is None else _postfilter(lib, "ref_demosaic_downsample_postfilter", rgba, iterations)


def emul_postfilter(rgba, iterations):
    return _postfilter(emul_lib("demosaic_postfilter"), "emul_demosaic_downsample_postfilter", rgba, iterations)


CYGM_TO_RGB = np.array([[0.82, -1.27, 0.31, 1.14], [-0.35, 1.61, 0.48, -0.74], [1.03, -0.22, -0.67, 0.86]], np.float64) / 3.0


def _downsample4(lib, fn, mosaic, filters, cam_to_rgb):
    h, w = mosaic.shape
    out, src = util.aligned_empty(((h + 1) // 2, (w + 1) // 2, 4)), util.aligned_empty(mosaic.shape)
    out[...] = ALPHA_FILL
    src[...] = mosaic
    mat = np.ascontiguousarray(cam_to_rgb, np.float64)
    f = getattr(lib, fn)
    f.restype = C.c_int
    f.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_uint32, C.c_void_p]
    assert f(out.ctypes.data, src.ctypes.data, w, h, filters, mat.ctypes.data) == 0
    return np.array(out)


def oracle_downsample4(m, filters, cam_to_rgb=CYGM_TO_RGB):
    return _downsample4(util.oracle(), "orc_demosaic_downsample4", m, filters, cam_to_rgb)


@util.recorded(lambda m, filters, cam_to_rgb=CYGM_TO_RGB, kind="strict": oracle_downsample4(m, filters, cam_to_rgb))
def ref_downsample4(m, filters, cam_to_rgb=CYGM_TO_RGB, kind="strict"):
    lib = util.ref(kind)
    return None if lib is None else _downsample4(lib, "ref_demosaic_downsample4", m, filters, cam_to_rgb)


def emul_downsample4(m, filters, cam_to_rgb=CYGM_TO_RGB):
    return _downsample4(emul_lib(), "emul_demosaic_downsample4", m, filters, cam_to_rgb)
