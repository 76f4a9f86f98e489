"""highlights, mode "guided laplacians" (iop/highlights/laplacian.c) on the CPU: the restated oracle against the reference's lines compiled
in place, and the kernels of ansel_b200/csrc/highlights_laplacian.cu run thread by thread against the oracle."""
import ctypes as C
import numpy as np
import pytest
import util
import hl_laplacian_util as hu

RGGB, GBRG = util.BAYER["RGGB"], util.BAYER["GBRG"]


def same_bits(a, b):
    return a.view(np.int32) == b.view(np.int32)


CASES = [
    ("defaults", 400, 300, RGGB, {}),
    ("odd_size_noise", 401, 299, GBRG, dict(iterations=3, noise_level=0.2)),
    ("few_scales_solid", 203, 157, RGGB, dict(scales=4, solid_color=0.3, iterations=1)),
    ("zoomed_out_roi", 260, 180, RGGB, dict(roi_scale=0.5, x=13, y=7, iterations=2)),
    ("one_scale", 120, 90, RGGB, dict(scales=2, iterations=2, noise_level=0.05)),
]


@pytest.mark.parametrize("name,w,h,filters,kw", CASES, ids=[c[0] for c in CASES])
def test_oracle_is_the_reference(name, w, h, filters, kw):
    m = hu.clipped_mosaic(w, h, len(name))
    want, norm = hu.ref(m, filters, hu.clips_of(), **kw)
    got, _ = hu.oracle(m, filters, hu.clips_of(), norm=norm, **kw)
    assert same_bits(got, want).all()
    changed = got != m
    assert 0.02 < changed.mean() < 0.9 and np.isfinite(got).all()


def test_oracle_is_the_reference_on_rgba_input():
    img = hu.clipped_rgba(300, 200, 4)
    want, norm = hu.ref(img, 0, hu.clips_of(), iterations=2, noise_level=0.1)
    got, _ = hu.oracle(img, 0, hu.clips_of(), norm=norm, iterations=2, noise_level=0.1)
    assert same_bits(got, want).all()
    assert same_bits(got[..., 3], img[..., 3]).all() and (got[..., :3] != img[..., :3]).any()


XCASES = [("xtrans", 300, 200, dict(xtrans=hu.XTRANS)), ("xtrans_roi_noise", 251, 173, dict(xtrans=hu.XTRANS, x=5, y=2, iterations=2, noise_level=0.1))]


@pytest.mark.parametrize("name,w,h,kw", XCASES, ids=[c[0] for c in XCASES])
def test_oracle_is_the_reference_on_xtrans(name, w, h, kw):
    m = hu.clipped_mosaic(w, h, 3)
    want, norm = hu.ref(m, 9, hu.clips_of(), **kw)
    got, _ = hu.oracle(m, 9, hu.clips_of(), norm=norm, **kw)
    assert same_bits(got, want).all() and (got != m).mean() > 0.05


@pytest.mark.parametrize("name,w,h,kw", XCASES, ids=[c[0] for c in XCASES])
def test_kernels_thread_by_thread_xtrans(name, w, h, kw):
    m = hu.clipped_mosaic(w, h, 3)
    want, norm = hu.oracle(m, 9, hu.clips_of(), **kw)
    assert same_bits(hu.emul(m, 9, hu.clips_of(), norm, **kw), want).all()


def test_normalization_is_the_serial_sum_of_one_thread():
    """the reference's vector is an OpenMP float reduction: with one thread it is the oracle's row-order sum, bit for bit, and with many it is
    another value; the frames agree closely all the same (the vector divides the gathered frame and multiplies the result back)"""
    m = hu.clipped_mosaic(640, 480, 11)
    want, norm1 = hu.ref(m, RGGB, hu.clips_of(), threads=1)
    got, norm_o = hu.oracle(m, RGGB, hu.clips_of())
    assert same_bits(norm1, norm_o).all() and same_bits(got, want).all()
    many, norm8 = hu.ref(m, RGGB, hu.clips_of(), threads=8)
    exact = np.array([m[0::2, 0::2].sum(dtype=np.float64), m[0::2, 1::2].sum(dtype=np.float64) + m[1::2, 0::2].sum(dtype=np.float64),
                      m[1::2, 1::2].sum(dtype=np.float64)]) / m.size
    assert np.abs(norm8[:3] / exact - 1).max() < 1e-4 and np.abs(norm1[:3] / exact - 1).max() < 1e-3
    assert np.abs(many - want).max() < 2e-3


@pytest.mark.parametrize("name,w,h,filters,kw", CASES, ids=[c[0] for c in CASES])
def test_kernels_thread_by_thread(name, w, h, filters, kw):
    m = hu.clipped_mosaic(w, h, len(name))
    want, norm = hu.oracle(m, filters, hu.clips_of(), **kw)
    got = hu.emul(m, filters, hu.clips_of(), norm, **kw)
    assert same_bits(got, want).all()


def test_kernels_thread_by_thread_rgba():
    img = hu.clipped_rgba(220, 160, 5)
    want, norm = hu.oracle(img, 0, hu.clips_of(), iterations=2, noise_level=0.1)
    got = hu.emul(img, 0, hu.clips_of(), norm, iterations=2, noise_level=0.1)
    assert same_bits(got, want).all()


def test_scale_count():
    """laplacian.c:461-463 through the library's host code and the oracle's"""
    import ansel_b200  # noqa: F401  (the harness is built next to it)
    hu.emul(hu.clipped_mosaic(64, 48, 1), RGGB, hu.clips_of(), (0.1, 0.3, 0.1, 1.0), iterations=1)
    f, g = hu._EMUL.emul_hl_laplacian_scales, util.oracle().orc_hl_laplacian_scales
    for param in range(0, 13):
        for iscale, roi_scale in [(1.0, 1.0), (1.0, 0.5), (1.0, 0.13), (2.0, 1.0)]:
            a = f(param, C.c_float(iscale), C.c_float(roi_scale))
            assert a == g(param, C.c_float(iscale), C.c_float(roi_scale)) and 1 <= a <= 12


@pytest.mark.parametrize("name", list(hu.GOLDEN))
def test_oracle_against_the_committed_reference_output(name):
    """tests/golden/hl_laplacian.npz: what the reference's lines produced in the authoring container (make_golden_hl_laplacian.py)"""
    import os
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "hl_laplacian.npz"))
    w, h, f, kw = hu.GOLDEN[name]
    img = hu.clipped_mosaic(w, h, len(name)) if f else hu.clipped_rgba(w, h, len(name))
    got, _ = hu.oracle(img, f, hu.clips_of(), norm=g[name + "_norm"], **kw)
    assert same_bits(got, g[name]).all()
    assert same_bits(hu.emul(img, f, hu.clips_of(), g[name + "_norm"], **kw), g[name]).all()


def test_random_frames_and_parameters_reference_oracle_and_kernels_agree():
    """frames from 8 px a side, the three layouts, ROI origins, zoom, the scale parameter from 0, noise and solid colour, clip levels"""
    rng = np.random.default_rng(7)
    for trial in range(40):
        w, h, kind = int(rng.integers(8, 180)), int(rng.integers(8, 140)), int(rng.integers(3))
        f = [RGGB, GBRG, util.BAYER["BGGR"]][rng.integers(3)] if kind == 0 else (9 if kind == 1 else 0)
        kw = dict(iterations=int(rng.integers(1, 4)), scales=int(rng.integers(0, 10)), noise_level=float(rng.choice([0, 0.1, 0.5])),
                  solid_color=float(rng.choice([0, 0.3, 1.0])), roi_scale=float(rng.choice([1.0, 0.5, 0.33])), iscale=float(rng.choice([1.0, 2.0])))
        if f:
            kw.update(x=int(rng.integers(0, 7)), y=int(rng.integers(0, 7)))
        if f == 9:
            kw["xtrans"] = hu.XTRANS
        img = hu.clipped_mosaic(w, h, int(rng.integers(100)), blobs=3) if f else hu.clipped_rgba(w, h, int(rng.integers(100)))
        clips = hu.clips_of(float(rng.choice([1.0, 0.8])), (float(rng.choice([1.0, 2.0])), 1.0, float(rng.choice([1.0, 1.5]))))
        want, norm = hu.ref(img, f, clips, **kw)
        got, _ = hu.oracle(img, f, clips, norm=norm, **kw)
        assert same_bits(got, want).all(), (trial, w, h, f, kw)
        assert same_bits(hu.emul(img, f, clips, norm, **kw), got).all(), (trial, w, h, f, kw)
