"""CPU: the VNG4 demosaicer and the dual-demosaic blend: oracle pinned bit for bit to iop/demosaic/vng.c, basic.c
lin_interpolate, dual.c and develop/masks/detail.c compiled in place, to the golden vectors those builds produced, and the
product's kernels (VNG as a function of the bilinear image, the detail mask as stencils at clamped coordinates) run on the
CPU against the oracle."""
import os
import subprocess

import numpy as np
import pytest

import util
import vng_util as vu


def same_bits(a, b):
    return (a.view(np.uint32) == b.view(np.uint32)) | (np.isnan(a) & np.isnan(b))


@pytest.fixture(scope="module", autouse=True)
def _build():
    subprocess.run(["make", "-s", "-C", util.ORACLE_DIR, "oracle"], check=True)
    if util.ref("strict") is None and os.path.isdir("/root/reference/src"):
        util.build_oracle()


THRESHOLDS = (0.2, 0.05, 1.0)


@pytest.mark.parametrize("name", list(vu.CASES))
def test_vng_oracle_equals_reference(name):
    m, filters, x, y = vu.case(name)
    for lin in (1, 0):
        assert same_bits(vu.oracle_vng(m, filters, x, y, lin), vu.ref_vng(m, filters, x, y, lin)).all(), lin


@pytest.mark.parametrize("name", list(vu.CASES))
def test_dual_oracle_equals_reference(name):
    m, filters, x, y = vu.case(name)
    rgb = vu.sharp_frame(m, filters, x, y)
    for thr in THRESHOLDS:
        want = vu.ref_dual(rgb, m, filters, x, y, thr)
        assert same_bits(vu.oracle_dual(rgb, m, filters, x, y, thr), want).all(), thr
        assert m.shape[0] <= 16 or not same_bits(want, rgb).all()
    assert same_bits(vu.oracle_dual(rgb, m, filters, x, y, 0.3, mask=1), vu.ref_dual(rgb, m, filters, x, y, 0.3, mask=1)).all()
    assert same_bits(vu.ref_dual(rgb, m, filters, x, y, 0.0), rgb).all()          # threshold 0: untouched (dual.c:52)


def test_vng_and_dual_oracle_equal_golden():
    g = np.load(os.path.join(util.GOLDEN_DIR, "vng.npz"))
    for name in vu.CASES:
        m, filters, x, y = vu.case(name)
        assert same_bits(vu.oracle_vng(m, filters, x, y), g["vng_" + name]).all(), name
        assert same_bits(vu.oracle_dual(vu.sharp_frame(m, filters, x, y), m, filters, x, y, 0.2), g["dual_" + name]).all(), name


@pytest.mark.parametrize("name", list(vu.CASES))
def test_vng_kernels_equal_oracle(name):
    m, filters, x, y = vu.case(name)
    for lin in (1, 0):
        assert same_bits(vu.emul_vng(m, filters, x, y, lin), vu.oracle_vng(m, filters, x, y, lin)).all(), lin


@pytest.mark.parametrize("name", list(vu.CASES))
def test_dual_kernels_equal_oracle(name):
    m, filters, x, y = vu.case(name)
    rgb = vu.sharp_frame(m, filters, x, y)
    for thr in THRESHOLDS:
        assert same_bits(vu.emul_dual(rgb, m, filters, x, y, thr), vu.oracle_dual(rgb, m, filters, x, y, thr)).all(), thr


@pytest.mark.parametrize("name", list(vu.XTRANS_CASES))
def test_vng_xtrans_oracle_equals_reference(name):
    """the X-Trans branch of vng_interpolate (three colours, 6x6 periods); lane 3 is uninitialised memory in the reference"""
    m, x, y = vu.xtrans_case(name)
    for lin in (1, 0):
        assert same_bits(vu.oracle_vng_xtrans(m, x, y, lin)[..., :3], vu.ref_vng_xtrans(m, x, y, lin)[..., :3]).all(), lin


@pytest.mark.parametrize("name", list(vu.XTRANS_CASES))
def test_vng_xtrans_kernels_equal_oracle(name):
    m, x, y = vu.xtrans_case(name)
    g = np.load(os.path.join(util.GOLDEN_DIR, "vng.npz"))
    for lin in (1, 0):
        got = vu.emul_vng_xtrans(m, x, y, lin)
        assert same_bits(got[..., :3], vu.oracle_vng_xtrans(m, x, y, lin)[..., :3]).all(), lin
    assert same_bits(got[..., :3], g["xtrans_" + name][..., :3]).all() and (got[..., 3] == -7.0).all()
