"""Helpers for the bilateral-grid tests: the oracle (oracle/restate/bilateral_oracle.c), the reference's pixel/bilateral.c
compiled in place (oracle/_ref: ref_bilateral.c; the splat's slice count is a parameter) and the product's kernels run on the
CPU (tests/emul/emul_bilateral.cpp).  Checkers only."""
import ctypes as C
import os
import subprocess

import numpy as np

import util

EMUL = os.path.join(os.path.dirname(os.path.abspath(__file__)), "emul")

CASES = {
    # name: (width, height, sigma_s, sigma_r, detail)
    "default_like": (200, 150, 8.0, 5.0, 0.5),
    "coarse_smoothing": (333, 217, 20.0, 10.0, -1.0),
    "sub_pixel_sigma": (64, 48, 0.3, 50.0, 1.0),          # sigma_s is raised to 0.5: a grid finer than the frame
    "fine_range": (160, 120, 3.7, 2.0, 0.25),               # 51 range bins
    "few_cells": (200, 150, 50.0, 5.0, 0.6),                # 5 x 4 x 21 cells: every cell sees thousands of pixels
}


def case(name):
    w, h, ss, sr, detail = CASES[name]
    img = np.ascontiguousarray(util.lab_scene(w, h, 5))
    img[3, 3, 0], img[4, 4, 0], img[5, 5, 0] = np.nan, 150.0, -3.0
    return img, ss, sr, detail


def _run(lib, fn, img, ss, sr, detail, grid_after=None):
    """-> (rc, out, dims, grid or None); grid_after: None, "splat" or "blur" """
    h, w = img.shape[:2]
    src, out = util.aligned_empty(img.shape), util.aligned_empty(img.shape)
    src[...] = img
    out[...] = -7.0
    dims = (C.c_int * 3)()
    cap = 4_000_000
    grid = np.zeros(cap, np.float32) if grid_after else None
    f = getattr(lib, fn)
    f.restype = C.c_int
    f.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_float, C.c_float, C.c_float, C.c_void_p, C.c_int, C.c_void_p, C.c_int]
    rc = f(src.ctypes.data, out.ctypes.data, w, h, ss, sr, detail, grid.ctypes.data if grid_after else None, cap, dims, 1 if grid_after == "blur" else 0)
    n = dims[0] * dims[1] * dims[2]
    return rc, np.array(out), tuple(dims), (grid[:n].copy() if grid_after else None)


def oracle_bilateral(img, ss, sr, detail, grid_after=None):
    return _run(util.oracle(), "orc_bilateral", img, ss, sr, detail, grid_after)


def emul_lib():
    so = os.path.join(EMUL, "libemul_bilateral.so")
    srcs = [os.path.join(EMUL, "emul_bilateral.cpp"), os.path.join(EMUL, "cuda_on_cpu.h"), os.path.join(util.ROOT, "ansel_b200", "csrc", "bilateral.cu")]
    if not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in srcs):
        subprocess.run(["g++", "-O1", "-std=c++17", "-fno-fast-math", "-ffp-contract=off", "-I", EMUL, "-shared", "-fPIC", "-o", so, srcs[0]], check=True)
    return C.CDLL(so)


def emul_bilateral(img, ss, sr, detail, grid_after=None):
    return _run(emul_lib(), "emul_bilateral", img, ss, sr, detail, grid_after)


@util.recorded(lambda img, ss, sr, detail, threads=1, kind="strict": oracle_bilateral(img, ss, sr, detail)[1])
def ref_bilateral(img, ss, sr, detail, threads=1, kind="strict"):
    lib = util.ref(kind)
    if lib is None:
        return None
    h, w = img.shape[:2]
    src, out = util.aligned_empty(img.shape), util.aligned_empty(img.shape)
    src[...] = img
    out[...] = -7.0
    f = lib.ref_bilateral
    f.restype = C.c_int
    f.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_float, C.c_float, C.c_float, C.c_int]
    assert f(src.ctypes.data, out.ctypes.data, w, h, ss, sr, detail, threads) == 0
    return np.array(out)


@util.recorded(lambda img, ss, sr, blur, threads=1, kind="strict": oracle_bilateral(img, ss, sr, 0.0, "blur" if blur else "splat")[2:])
def ref_grid(img, ss, sr, blur, threads=1, kind="strict"):
    lib = util.ref(kind)
    h, w = img.shape[:2]
    src = util.aligned_empty(img.shape)
    src[...] = img
    cap = 4_000_000
    grid, dims = np.zeros(cap, np.float32), (C.c_int * 3)()
    f = lib.ref_bilateral_grid
    f.restype = C.c_int
    f.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_float, C.c_float, C.c_int, C.c_int]
    assert f(src.ctypes.data, grid.ctypes.data, cap, dims, w, h, ss, sr, blur, threads) == 0
    return tuple(dims), grid[:dims[0] * dims[1] * dims[2]].copy()
