"""CPU: the LMMSE demosaicer.  The oracle with the tile planes carried through the serial walk of the tiles is pinned bit for bit to
iop/demosaic/lmmse.c compiled in place without OpenMP (and to the golden vectors of that build), every refinement mode; with the planes zeroed
in front of every tile it is what the product's kernel computes: its stages, compiled with g++ and run thread by thread in either order, equal
it.  The distance between the two modes -- what in the reference depends on the order a thread met its tiles -- is measured."""
import os
import subprocess

import numpy as np
import pytest

import util
import lmmse_util as lu


def same_bits(a, b):
    return (a.view(np.uint32) == b.view(np.uint32)) | (np.isnan(a) & np.isnan(b))


@pytest.fixture(scope="module", autouse=True)
def _build():
    subprocess.run(["make", "-s", "-C", util.ORACLE_DIR, "oracle"], check=True)
    if util.ref("strict") is None and os.path.isdir("/root/reference/src"):
        util.build_oracle()




@pytest.mark.parametrize("mode", [0, 1, 2, 3, 4])
@pytest.mark.parametrize("name", list(lu.CASES))
def test_oracle_with_carried_planes_equals_reference(name, mode):
    m, f = lu.case(name)
    assert same_bits(lu.oracle(m, f, mode, carry=1), lu.ref(m, f, mode)).all()


@pytest.mark.parametrize("name", list(lu.CASES))
def test_oracle_equals_golden(name):
    g = np.load(os.path.join(util.GOLDEN_DIR, "lmmse.npz"))
    m, f = lu.case(name)
    for mode in (0, 1, 4):
        if f"m{mode}_{name}" in g:
            assert same_bits(lu.oracle(m, f, mode, carry=1), g[f"m{mode}_{name}"]).all(), mode


@pytest.mark.parametrize("mode", [0, 1, 2, 3, 4])
@pytest.mark.parametrize("name", list(lu.CASES))
def test_kernel_stages_equal_oracle_with_fresh_planes(name, mode):
    m, f = lu.case(name)
    want = lu.oracle(m, f, mode, carry=0)
    for ascending in (0, 1):
        assert same_bits(lu.emul(m, f, mode, 96, ascending), want).all(), ascending


def test_what_the_carried_planes_change():
    """a frame of one tile has nothing to carry; in a frame of several, what differs lies on the tile seams and the frame's rim: within 20 px of a
    seam column / row (a multiple of 112 + 8) or of the frame's edge"""
    m, f = lu.case("grbg_one_tile")
    for mode in (0, 4):
        assert same_bits(lu.oracle(m, f, mode, carry=0), lu.oracle(m, f, mode, carry=1)).all()
    m, f = lu.case("rggb")
    h, w = m.shape
    for mode in (1, 4):
        bad = (~same_bits(lu.oracle(m, f, mode, carry=0), lu.oracle(m, f, mode, carry=1))).any(axis=2)
        assert 0.02 < bad.mean() < 0.25
        ys, xs = np.nonzero(bad)
        near_rim = (ys < 20) | (xs < 20) | (ys >= h - 20) | (xs >= w - 20)
        seam = lambda v: np.minimum(np.abs((v - 8) % 112), 112 - np.abs((v - 8) % 112)) <= 20   # noqa: E731
        assert (near_rim | seam(ys) | seam(xs)).all()


def test_kernel_stages_on_random_frame_sizes_and_modes():
    """sizes from 12 px, the four Bayer phases, the five refinement modes, three thread counts and both thread orders"""
    rng = np.random.default_rng(5)
    pats = ["RGGB", "BGGR", "GRBG", "GBRG"]
    for trial in range(8):
        w, h, mode, pat = int(rng.integers(12, 420)), int(rng.integers(12, 330)), int(rng.integers(0, 5)), pats[rng.integers(4)]
        m = np.ascontiguousarray(util.frame_natural(w, h, int(rng.integers(50)), filters=util.BAYER[pat]), np.float32)
        want = lu.oracle(m, util.BAYER[pat], mode, carry=0)
        got = lu.emul(m, util.BAYER[pat], mode, nthreads=int(rng.choice([32, 96, 128])), ascending=int(rng.integers(2)))
        assert same_bits(got, want).all(), (trial, w, h, mode, pat)
