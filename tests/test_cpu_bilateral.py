"""CPU: the bilateral grid (local contrast's other mode): oracle pinned bit for bit to pixel/bilateral.c compiled in place
with one splat slice, the thread-count dependence of the reference measured, golden vectors, and the product's kernels (a
gather per grid column instead of the reference's scatter) run on the CPU against the oracle."""
import os
import subprocess

import numpy as np
import pytest

import bilateral_util as bu
import util


def same_bits(a, b):
    return (a.view(np.uint32) == b.view(np.uint32)) | (np.isnan(a) & np.isnan(b))


@pytest.fixture(scope="module", autouse=True)
def _build():
    subprocess.run(["make", "-s", "-C", util.ORACLE_DIR, "oracle"], check=True)
    if util.ref("strict") is None and os.path.isdir("/root/reference/src"):
        util.build_oracle()




@pytest.mark.parametrize("name", list(bu.CASES))
def test_bilateral_oracle_equals_one_slice_reference(name):
    img, ss, sr, detail = bu.case(name)
    rc, got, dims, grid = bu.oracle_bilateral(img, ss, sr, detail, "splat")
    assert rc == 0 and same_bits(got, bu.ref_bilateral(img, ss, sr, detail, threads=1)).all()
    rdims, rgrid = bu.ref_grid(img, ss, sr, blur=0, threads=1)
    assert dims == rdims and same_bits(grid, rgrid).all()
    assert same_bits(bu.oracle_bilateral(img, ss, sr, detail, "blur")[3], bu.ref_grid(img, ss, sr, blur=1, threads=1)[1]).all()


def test_reference_splat_depends_on_the_thread_count():
    """the partial grids of the slices are added after the fact: cells fed by two slices round differently"""
    img, ss, sr, detail = bu.case("coarse_smoothing")
    one, eight = bu.ref_bilateral(img, ss, sr, detail, threads=1), bu.ref_bilateral(img, ss, sr, detail, threads=8)
    differ = ~same_bits(one, eight)
    assert differ.any() and util.ulp_distance(one[..., 0], eight[..., 0]).max() < 64


def test_bilateral_oracle_equals_golden():
    g = np.load(os.path.join(util.GOLDEN_DIR, "bilateral.npz"))
    for name in bu.CASES:
        assert same_bits(bu.oracle_bilateral(*bu.case(name))[1], g[name]).all(), name


@pytest.mark.parametrize("name", list(bu.CASES))
def test_bilateral_kernels_equal_oracle(name):
    """splat (grid compared cell for cell), the three blurs, the slice"""
    img, ss, sr, detail = bu.case(name)
    for stage in ("splat", "blur"):
        rc, got, dims, grid = bu.emul_bilateral(img, ss, sr, detail, stage)
        _, want, odims, ogrid = bu.oracle_bilateral(img, ss, sr, detail, stage)
        assert rc == 0 and dims == odims and same_bits(grid, ogrid).all(), stage
        assert same_bits(got, want).all()


def test_bilateral_kernels_ragged_sizes():
    for w, h, ss in ((97, 61, 4.3), (40, 200, 7.0), (500, 31, 2.2)):
        img = np.ascontiguousarray(util.lab_scene(w, h, 9))
        rc, got, _, _ = bu.emul_bilateral(img, ss, 6.0, 0.4)
        assert rc == 0 and same_bits(got, bu.oracle_bilateral(img, ss, 6.0, 0.4)[1]).all()
