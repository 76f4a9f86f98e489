"""CPU: Markesteijn's X-Trans demosaicer.  The oracle is pinned bit for bit to iop/demosaic/markesteijn.c :25-523 compiled in place
(one and three passes) and to the golden vectors that build produced; the stages of the product's kernel (one and three passes), compiled with g++
and run thread by thread in either order, equal the oracle; the classes of tiles the product ships one record of the loop
:199-246 for are checked against a walk of every tile on its own."""
import os
import subprocess

import numpy as np
import pytest

import util
import markesteijn_util as mu
from vng_util import XTRANS


def same_bits(a, b):
    return (a.view(np.uint32) == b.view(np.uint32)) | (np.isnan(a) & np.isnan(b))


@pytest.fixture(scope="module", autouse=True)
def _build():
    subprocess.run(["make", "-s", "-C", util.ORACLE_DIR, "oracle"], check=True)
    if util.ref("strict") is None and os.path.isdir("/root/reference/src"):
        util.build_oracle()




@pytest.mark.parametrize("passes", [1, 3])
@pytest.mark.parametrize("name", list(mu.CASES))
def test_oracle_equals_reference(name, passes):
    m, x, y = mu.case(name)
    if min(m.shape) <= (12 if passes == 1 else 17):
        pytest.skip("the reference mirrors out of its input on frames this small (TRANSLATE, markesteijn.c:158): undefined")
    got, want = mu.oracle(m, x, y, passes), mu.ref(m, x, y, passes)
    assert same_bits(got, want).all()
    assert (got[..., 3] == -7.0).all()          # lane 3 is not written


@pytest.mark.parametrize("name", list(mu.CASES))
def test_oracle_equals_golden(name):
    g = np.load(os.path.join(util.GOLDEN_DIR, "markesteijn.npz"))
    m, x, y = mu.case(name)
    for passes in (1, 3):
        if min(m.shape) > (12 if passes == 1 else 17):
            assert same_bits(mu.oracle(m, x, y, passes)[..., :3], g[f"p{passes}_{name}"][..., :3]).all(), passes


def test_oracle_equals_reference_on_other_seeds_and_a_dark_frame():
    for seed in (1, 2):
        m, x, y = mu.case("roi2", seed)
        assert same_bits(mu.oracle(m, x, y, 1), mu.ref(m, x, y, 1)).all()
    m = np.zeros((150, 140), np.float32)         # every maximum of green is the loop's "new pair" marker
    m[70:80, 60:90] = 0.5
    assert same_bits(mu.oracle(m, 2, 1, 1), mu.ref(m, 2, 1, 1)).all()


@pytest.mark.parametrize("passes", [1, 3])
@pytest.mark.parametrize("ascending", [0, 1])
@pytest.mark.parametrize("name", list(mu.CASES))
def test_kernel_stages_equal_oracle(name, ascending, passes):
    """no stage reads what another thread of the same stage writes: both thread orders give the oracle's bits"""
    m, x, y = mu.case(name)
    if min(m.shape) <= (12 if passes == 1 else 17):
        pytest.skip("undefined in the reference (out-of-bounds mirror); the product refuses the frame")
    assert same_bits(mu.emul(m, x, y, 96, ascending, passes), mu.oracle(m, x, y, passes)).all()


def test_kernel_stages_on_a_dark_frame_and_other_thread_counts():
    m = np.zeros((150, 140), np.float32)
    m[70:80, 60:90] = 0.5
    for passes in (1, 3):
        want = mu.oracle(m, 2, 1, passes)
        for nt in (1, 37, 1024):
            assert same_bits(mu.emul(m, 2, 1, nt, 0, passes), want).all(), (passes, nt)


@pytest.mark.parametrize("geom", [(8256, 5504, 0, 0), (6000, 4000, 3, 5), (4896, 3264, 1, 2), (98, 98, 0, 0), (99, 197, 4, 1), (300, 210, 0, 0), (30, 17, 2, 3)])
def test_tile_classes_walk_like_every_tile_on_its_own(geom):
    """-1: two tiles of a class walk differently; -2: too many classes; -3: a red/blue pixel the walk never writes (the reference would read
    what the previous tile left there)"""
    for passes in (1, 3):
        n = mu.emul_classes(*geom, passes=passes)
        assert 1 <= n <= 20, (passes, n)


def test_tile_classes_with_a_permuted_pattern():
    xt = np.roll(np.roll(XTRANS, 2, axis=0), 1, axis=1)
    assert 1 <= mu.emul_classes(1000, 700, 0, 0, xt) <= 20


def test_kernel_stages_on_random_frame_sizes_and_origins():
    """frame sizes, ROI origins (the phase of the 6x6 pattern and of the hexagon walk), one and three passes, both thread orders"""
    rng = np.random.default_rng(6)
    for trial in range(5):
        w, h, x, y = int(rng.integers(40, 400)), int(rng.integers(40, 300)), int(rng.integers(0, 12)), int(rng.integers(0, 12))
        passes = int(rng.choice([1, 3]))
        m = np.ascontiguousarray(util.frame_natural(w, h, int(rng.integers(50))), np.float32)
        want = mu.oracle(m, x, y, passes)
        got = mu.emul(m, x, y, nthreads=int(rng.choice([64, 96])), ascending=int(rng.integers(2)), passes=passes)
        assert same_bits(got, want).all(), (trial, w, h, x, y, passes)
