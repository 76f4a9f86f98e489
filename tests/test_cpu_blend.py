"""CPU: blending in the scene-referred RGB space.  The oracle is pinned bit for bit to develop/blend.c and develop/blends/blendif_rgb_jzczhz.c
compiled in place (oracle/_ref: ref_blend.c) on every blend operator, mask source, combination and the mask tone curve; the product's
plan and kernel, compiled with g++ and run thread by thread, equal the oracle."""
import os
import subprocess

import numpy as np
import pytest

import util
import blend_util as bu


def same_bits(a, b):
    return (a.view(np.uint32) == b.view(np.uint32)) | (np.isnan(a) & np.isnan(b))


@pytest.fixture(scope="module", autouse=True)
def _build():
    subprocess.run(["make", "-s", "-C", util.ORACLE_DIR, "oracle"], check=True)
    if util.ref("strict") is None and os.path.isdir("/root/reference/src"):
        util.build_oracle()


IDS = [c[0] for c in bu.CONFIGS]


@pytest.mark.parametrize("cfg", bu.CONFIGS, ids=IDS)
def test_oracle_equals_reference(cfg):
    name, kw, uses_form = cfg
    a, b, form = bu.frames()
    p = bu.params(**kw)
    rc_r, out_r, mask_r = bu.ref(a, b, p, form if uses_form else None)
    rc_o, out_o, mask_o = bu.oracle(a, b, p, form if uses_form else None)
    assert rc_r == rc_o == 0
    assert same_bits(out_o, out_r).all() and same_bits(mask_o, mask_r).all()
    assert (name == "disabled") == np.array_equal(out_r, b)      # every other configuration changes the output


def test_oracle_equals_reference_with_roi_out_inside_roi_in():
    a, b, form = bu.frames(100, 80, 2, xoffs=7, yoffs=5)
    for name, kw, uses_form in bu.CONFIGS[::3]:
        p = bu.params(**kw)
        r, o = bu.ref(a, b, p, form if uses_form else None, 7, 5), bu.oracle(a, b, p, form if uses_form else None, 7, 5)
        assert same_bits(o[1], r[1]).all() and same_bits(o[2], r[2]).all(), name


@pytest.mark.parametrize("cfg", bu.CONFIGS, ids=IDS)
def test_kernel_equals_oracle(cfg):
    name, kw, uses_form = cfg
    a, b, form = bu.frames(301, 77, 3)
    p = bu.params(**kw)
    rc_e, out_e, mask_e = bu.emul(a, b, p, form if uses_form else None)
    rc_o, out_o, mask_o = bu.oracle(a, b, p, form if uses_form else None)
    assert rc_e == rc_o == 0
    assert same_bits(out_e, out_o).all() and same_bits(mask_e, mask_o).all()


def test_kernel_with_offsets_and_what_is_refused():
    a, b, form = bu.frames(100, 80, 2, xoffs=7, yoffs=5)
    p = bu.params(mask_mode=bu.MASK_ENABLED | bu.MASK_SHAPE | bu.MASK_PARAMETRIC, drawn=1, channels={0: (0.1, 0.3, 0.7, 0.9), 6: (0.0, 0.0, 0.6, 0.9)})
    e, o = bu.emul(a, b, p, form, 7, 5), bu.oracle(a, b, p, form, 7, 5)
    assert same_bits(e[1], o[1]).all() and same_bits(e[2], o[2]).all()
    a, b, form = bu.frames(64, 48, 4)
    for kw in (dict(feathering_radius=5.0), dict(blur_radius=2.0), dict(details=0.5), dict(blend_cst=0), dict(profile_nonlinear=1)):
        p = bu.params(**kw)
        assert bu.emul(a, b, p)[0] == -1 and bu.oracle(a, b, p)[0] == -1, kw


# ---- the Lab space (develop/blends/blendif_lab.c) ----------------------------------------------------------------------------------------
LAB_IDS = [c[0] for c in bu.LAB_CONFIGS]


@pytest.mark.parametrize("cfg", bu.LAB_CONFIGS, ids=LAB_IDS)
def test_lab_oracle_equals_reference(cfg):
    """every operator of the Lab space, the L / a / b / C / h channels of the parametric mask, the other mask sources"""
    name, kw, uses_form = cfg
    a, b, form = bu.frames_lab()
    p = bu.params(**kw)
    rc_r, out_r, mask_r = bu.ref(a, b, p, form if uses_form else None)
    rc_o, out_o, mask_o = bu.oracle(a, b, p, form if uses_form else None)
    assert rc_r == rc_o == 0
    assert same_bits(out_o, out_r).all() and same_bits(mask_o, mask_r).all()
    assert not np.array_equal(out_r[..., :3], b[..., :3])


def test_lab_oracle_equals_reference_with_roi_out_inside_roi_in():
    a, b, form = bu.frames_lab(100, 80, 2, xoffs=7, yoffs=5)
    for name, kw, uses_form in bu.LAB_CONFIGS[::4]:
        p = bu.params(**kw)
        r, o = bu.ref(a, b, p, form if uses_form else None, 7, 5), bu.oracle(a, b, p, form if uses_form else None, 7, 5)
        assert same_bits(o[1], r[1]).all() and same_bits(o[2], r[2]).all(), name


@pytest.mark.parametrize("cfg", bu.LAB_CONFIGS, ids=LAB_IDS)
def test_lab_kernel_equals_oracle(cfg):
    """the kernel thread by thread; what goes through LCh is refused by the plan (the oracle follows the reference there too)"""
    name, kw, uses_form = cfg
    a, b, form = bu.frames_lab(301, 77, 3)
    p = bu.params(**kw)
    rc_e, out_e, mask_e = bu.emul(a, b, p, form if uses_form else None)
    rc_o, out_o, mask_o = bu.oracle(a, b, p, form if uses_form else None)
    assert rc_o == 0
    if not bu.lab_on_device(cfg):
        assert rc_e == -1 and np.array_equal(out_e, b)
        return
    assert rc_e == 0 and same_bits(out_e, out_o).all() and same_bits(mask_e, mask_o).all()


@pytest.mark.parametrize("cfg", bu.golden_configs(), ids=[c[0] for c in bu.golden_configs()])
def test_oracle_and_kernel_against_the_committed_reference_output(cfg):
    """tests/golden/blend.npz: what the reference's lines produced in the authoring container (tests/golden/make_golden_blend.py)"""
    name, kw, uses_form = cfg
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "blend.npz"))
    a, b, form = bu.golden_frames(kw)
    p = bu.params(**kw)
    for run in (bu.oracle, bu.emul):
        rc, out, mask = run(a, b, p, form if uses_form else None)
        assert rc == 0 and same_bits(out, g[name]).all() and same_bits(mask, g[name + "_mask"]).all(), run.__name__


# ---- the display-referred RGB space (develop/blends/blendif_rgb_hsl.c) ----------------------------------------------------------------------
DISPLAY_IDS = [c[0] for c in bu.DISPLAY_CONFIGS]


@pytest.mark.parametrize("cfg", bu.DISPLAY_CONFIGS, ids=DISPLAY_IDS)
def test_display_oracle_equals_reference(cfg):
    """every operator of the display-referred space, the gray / R / G / B / H / S / L channels of the parametric mask, the other mask sources"""
    name, kw, uses_form = cfg
    a, b, form = bu.frames_display()
    p = bu.params(**kw)
    rc_r, out_r, mask_r = bu.ref(a, b, p, form if uses_form else None)
    rc_o, out_o, mask_o = bu.oracle(a, b, p, form if uses_form else None)
    assert rc_r == rc_o == 0
    assert same_bits(out_o, out_r).all() and same_bits(mask_o, mask_r).all()
    assert not np.array_equal(out_r[..., :3], b[..., :3])


@pytest.mark.parametrize("cfg", bu.DISPLAY_CONFIGS, ids=DISPLAY_IDS)
def test_display_kernel_equals_oracle(cfg):
    name, kw, uses_form = cfg
    a, b, form = bu.frames_display(301, 77, 3)
    p = bu.params(**kw)
    rc_e, out_e, mask_e = bu.emul(a, b, p, form if uses_form else None)
    rc_o, out_o, mask_o = bu.oracle(a, b, p, form if uses_form else None)
    assert rc_e == rc_o == 0 and same_bits(out_e, out_o).all() and same_bits(mask_e, mask_o).all()


# ---- the raw space (develop/blends/blendif_raw.c): one float per site ------------------------------------------------------------------------
@pytest.mark.parametrize("cfg", bu.RAW_CONFIGS, ids=[c[0] for c in bu.RAW_CONFIGS])
def test_raw_reference_oracle_and_kernel(cfg):
    name, kw, uses_form = cfg
    a, b, form = bu.frames_raw(203, 77, 3)
    p, f = bu.params(**kw), None
    if uses_form:
        f = form
    r, o, e = bu.ref(a, b, p, f), bu.oracle(a, b, p, f), bu.emul(a, b, p, f)
    assert r[0] == o[0] == e[0] == 0
    assert same_bits(o[1], r[1]).all() and same_bits(o[2], r[2]).all() and same_bits(e[1], o[1]).all() and same_bits(e[2], o[2]).all()
    assert not np.array_equal(r[1], b)


def test_raw_kernel_with_roi_out_inside_roi_in():
    a, b, form = bu.frames_raw(100, 80, 2, xoffs=7, yoffs=5)
    p = bu.params(cst=bu.CS_RAW, mode="screen", mask_mode=bu.MASK_ENABLED | bu.MASK_SHAPE, drawn=1, opacity=80.0)
    e, o = bu.emul(a, b, p, form, 7, 5), bu.oracle(a, b, p, form, 7, 5)
    assert e[0] == o[0] == 0 and same_bits(e[1], o[1]).all() and same_bits(e[2], o[2]).all()


def random_parameter_block(rng):
    """a parameter block drawn at random in either colour space: operator, opacity, reverse, mask sources, up to three parametric channels with
    random limits, inversions and boosts, the combination mode, the mask tone curve, an earlier module's mask"""
    cst = (bu.CS_RGB_SCENE, bu.CS_LAB, bu.CS_RGB_DISPLAY, bu.CS_RAW)[rng.integers(4)]
    lab = cst == bu.CS_LAB
    modes = list({bu.CS_LAB: bu.LAB_MODES, bu.CS_RGB_DISPLAY: bu.DISPLAY_MODES, bu.CS_RAW: bu.RAW_MODES}.get(cst, bu.MODES).keys())
    kw = dict(mode=modes[rng.integers(len(modes))], opacity=float(rng.choice([0, 35, 70, 100, 140])), reverse=bool(rng.random() < 0.3),
              blend_parameter=float(rng.choice([0, -1.5, 2.0])), combine=int(rng.integers(0, 4)))
    kw["cst"] = cst
    scene = cst == bu.CS_RGB_SCENE
    mask_mode, uses_form, r = bu.MASK_ENABLED, False, rng.random()
    if r < 0.3:
        mask_mode, kw["drawn"], uses_form = mask_mode | bu.MASK_SHAPE, 1, True
    elif r < 0.45:
        mask_mode, kw["raster"], uses_form = mask_mode | bu.MASK_RASTER, 1, True
    if rng.random() < 0.6:
        mask_mode |= bu.MASK_PARAMETRIC
        allowed = [0, 1, 2, 4, 5, 6, 8, 9, 12, 13] if lab else [0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 12, 13, 14]
        channels, blendif = {}, 0
        for c in rng.choice(allowed, size=rng.integers(1, 4), replace=False):
            v = np.sort(rng.random(4)).astype(float)
            if scene and c in (8, 12):
                v = v * 0.02          # Jz of scene-referred pixels around 1 is about 0.01
            if scene and c in (9, 13):
                v = v * 0.01
            if rng.random() < 0.2:
                v[0] = v[1] = 0.0     # open at the bottom
            if rng.random() < 0.2:
                v[2] = v[3] = 1.0     # open at the top
            channels[int(c)] = tuple(v)
            if rng.random() < 0.3:
                blendif |= 1 << (16 + int(c))
        kw["channels"], kw["blendif"] = channels, blendif
        if rng.random() < 0.3:
            kw["boosts"] = {list(channels)[0]: float(rng.choice([-1.0, 0.5, 2.0]))}
    if rng.random() < 0.3:
        kw["contrast"], kw["brightness"] = float(rng.uniform(-0.8, 0.8)), float(rng.uniform(-1.0, 1.0))
    if rng.random() < 0.15:
        kw["mask_display"] = 1
    kw["mask_mode"] = mask_mode
    return cst, kw, uses_form


def test_random_parameter_blocks_reference_oracle_and_kernel_agree():
    """the four colour spaces"""
    rng = np.random.default_rng(123)
    for trial in range(240):
        cst, kw, uses_form = random_parameter_block(rng)
        a, b, form = bu.frames_of(cst)(64, 40, int(rng.integers(1000)))
        if rng.random() < 0.2:
            a[5, 5, ...], b[6, 6, ...] = np.nan, np.inf
        p, f = bu.params(**kw), (form if uses_form else None)
        r, o, e = bu.ref(a, b, p, f), bu.oracle(a, b, p, f), bu.emul(a, b, p, f)
        assert r[0] == o[0] == e[0] == 0, (trial, kw)
        assert same_bits(o[1], r[1]).all() and same_bits(o[2], r[2]).all() and same_bits(e[1], o[1]).all() and same_bits(e[2], o[2]).all(), (trial, kw)
