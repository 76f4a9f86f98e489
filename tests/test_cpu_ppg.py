"""CPU: the PPG demosaicer's oracle pinned bit for bit to iop/demosaic/ppg.c + basic.c pre_median compiled in place, to
the golden vectors those builds produced, and the product's fused kernel (one pass instead of the reference's three)
run on the CPU against the oracle."""
import os
import subprocess

import numpy as np
import pytest

import ppg_util as pu
import util


def same_bits(a, b):
    return (a.view(np.uint32) == b.view(np.uint32)) | (np.isnan(a) & np.isnan(b))


@pytest.fixture(scope="module", autouse=True)
def _build():
    subprocess.run(["make", "-s", "-C", util.ORACLE_DIR, "oracle"], check=True)
    if util.ref("strict") is None and os.path.isdir("/root/reference/src"):
        util.build_oracle()




@pytest.mark.parametrize("name", list(pu.CASES))
def test_ppg_oracle_equals_reference(name):
    m, filters, thrs = pu.case(name)
    want = pu.ref_ppg(m, filters, thrs)
    assert same_bits(pu.oracle_ppg(m, filters, thrs), want).all()
    h, w = m.shape
    assert (want[3:h - 3, 3:w - 3, 3] == 0.0).all() and (want[0, :, 3] == pu.ALPHA_FILL).all() and (want[:, 2, 3] == pu.ALPHA_FILL).all()


def test_pre_median_changes_the_result():
    m, filters, _ = pu.case("rggb")
    assert not same_bits(pu.ref_ppg(m, filters, 0.0), pu.ref_ppg(m, filters, 0.05)).all()


def test_ppg_oracle_equals_golden():
    g = np.load(os.path.join(util.GOLDEN_DIR, "ppg.npz"))
    for name in pu.CASES:
        assert same_bits(pu.oracle_ppg(*pu.case(name)), g[name]).all(), name


@pytest.mark.parametrize("name", list(pu.CASES))
def test_fused_ppg_kernel_equals_oracle(name):
    """ansel_b200/csrc/ppg.cu: pre_median_kernel + ppg_kernel, thread by thread on the CPU"""
    m, filters, thrs = pu.case(name)
    assert same_bits(pu.emul_ppg(m, filters, thrs), pu.oracle_ppg(m, filters, thrs)).all()


@pytest.mark.parametrize("pattern", list(util.BAYER))
def test_fused_ppg_kernel_every_phase_and_ragged_size(pattern):
    for w, h in ((33, 20), (64, 47), (9, 8)):
        m = util.frame_natural(w, h, 9, filters=util.BAYER[pattern])
        for thrs in (0.0, 0.1):
            assert same_bits(pu.emul_ppg(m, util.BAYER[pattern], thrs), pu.oracle_ppg(m, util.BAYER[pattern], thrs)).all()


PASSTHROUGH = [(util.BAYER["RGGB"], 0, 0), (util.BAYER["GBRG"], 3, 1), (9, 0, 0), (9, 4, 5)]


@pytest.mark.parametrize("filters,x,y", PASSTHROUGH)
def test_passthrough_oracle_equals_reference(filters, x, y):
    m = util.frame_natural(77, 50, 2)
    for colour in (0, 1):
        want = pu.ref_passthrough(m, filters, x, y, colour)
        assert same_bits(pu.oracle_passthrough(m, filters, x, y, colour), want).all()
        assert (want[..., 3] == pu.ALPHA_FILL).all()


@pytest.mark.parametrize("filters,x,y", PASSTHROUGH)
def test_passthrough_kernel_equals_oracle(filters, x, y):
    m = util.frame_natural(77, 50, 2)
    for colour in (0, 1):
        assert same_bits(pu.emul_passthrough(m, filters, x, y, colour), pu.oracle_passthrough(m, filters, x, y, colour)).all()


@pytest.mark.parametrize("pattern", list(util.BAYER))
def test_downsample_oracle_reference_and_kernel(pattern):
    """the half-size method (demosaic.c:480-532) on even and odd frame sizes"""
    f = util.BAYER[pattern]
    for w, h in ((64, 48), (77, 51), (9, 8)):
        m = util.frame_natural(w, h, 4, filters=f)
        want = pu.oracle_downsample(m, f)
        assert same_bits(want, pu.ref_downsample(m, f)).all()
        assert same_bits(pu.emul_downsample(m, f), want).all()


@pytest.mark.parametrize("case", ["origin", "roi", "roi2", "small", "sliver", "column"])
def test_downsample_xtrans_oracle_reference_and_kernel(case):
    """the half-size method on an X-Trans sensor (demosaic.c:543-666): missing colours from the quadrant search, ROI origins that
    rotate the pattern, odd sizes, NaN and flat patches, and frames so thin that quadrants are hidden by the edge"""
    import vng_util as vu
    if case in vu.XTRANS_CASES:
        m, x, y = vu.xtrans_case(case)
    else:
        w, h, x, y = {"sliver": (41, 2, 2, 3), "column": (1, 9, 4, 1)}[case]
        m = util.frame_natural(w, h, 8)
    want = pu.oracle_downsample_xtrans(m, x, y, vu.XTRANS)
    assert want.shape == ((m.shape[0] + 1) // 2, (m.shape[1] + 1) // 2, 4) and (want[..., 3] == 0).all()
    assert same_bits(want, pu.ref_downsample_xtrans(m, x, y, vu.XTRANS)).all()
    assert same_bits(pu.emul_downsample_xtrans(m, x, y, vu.XTRANS), want).all()


def test_downsample_xtrans_random_tables():
    """any 6x6 table with values 0..2 (not only Fuji's): a colour absent from the whole window resolves to 0"""
    import vng_util as vu
    rng = np.random.default_rng(77)
    for k in range(12):
        xt = rng.integers(0, 3, (6, 6)).astype(np.uint8)
        if k == 0:
            xt[...] = 1
        w, h, x, y = int(rng.integers(1, 40)), int(rng.integers(1, 40)), int(rng.integers(0, 12)), int(rng.integers(0, 12))
        m = util.frame_natural(w, h, 20 + k)
        want = pu.oracle_downsample_xtrans(m, x, y, xt)
        assert same_bits(want, pu.ref_downsample_xtrans(m, x, y, xt)).all(), k
        assert same_bits(pu.emul_downsample_xtrans(m, x, y, xt), want).all(), k


@pytest.mark.parametrize("size,iterations", [((64, 48), 1), ((33, 21), 3), ((5, 4), 2), ((1, 1), 1), ((2, 7), 1), ((300, 3), 2)])
def test_downsample_postfilter_oracle_reference_and_kernels(size, iterations):
    """the guided-Laplacian post-filter of the half-size method (demosaic.c:681-926) on half-size frames with NaN, inf, zero
    and flat patches; one to three iterations; frames thinner than the 5x5 patch"""
    w, h = size
    f = util.BAYER["RGGB"]
    half = pu.oracle_downsample(util.frame_natural(2 * w, 2 * h, 11 + w, filters=f), f)
    if w >= 40 and h >= 40:
        half[5, 5, 0] = np.nan
        half[10:14, 10:14, :3] = 0.25
        half[20, 20, :3] = 0
        half[30, 30, 1] = np.inf
    want = pu.oracle_postfilter(half, iterations)
    assert (want[..., 3] == 0).all() and not same_bits(want, half).all() or w == 1
    assert same_bits(want, pu.ref_postfilter(half, iterations)).all()
    assert same_bits(pu.emul_postfilter(half, iterations), want).all()


@pytest.mark.parametrize("filters", [0xb4b4b4b4, 0x1e4e1e4e, 0xe1e4e1e4])
def test_downsample_four_colour_oracle_reference_and_kernel(filters):
    """four-colour Bayer sensors (CYGM / RGBE words) through CAM_to_RGB, demosaic.c:514-521: double products, float accumulator"""
    for w, h in ((64, 48), (77, 51), (3, 1)):
        m = util.frame_natural(w, h, 31)
        if w > 10:
            m[7, 9], m[20, 21] = np.nan, 1e30
        want = pu.oracle_downsample4(m, filters)
        assert same_bits(want, pu.ref_downsample4(m, filters)).all()
        assert same_bits(pu.emul_downsample4(m, filters), want).all()
