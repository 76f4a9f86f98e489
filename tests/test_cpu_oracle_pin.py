"""CPU tests: the oracle against (a) the reference's own sources compiled here (oracle/_ref, when
present) and (b) the committed golden vectors those sources produced (tests/golden, always)."""
import ctypes as C
import os

import numpy as np
import pytest

import util


def same_bits(a, b):
    return (a.view(np.uint32) == b.view(np.uint32)) | (np.isnan(a) & np.isnan(b))


@pytest.fixture(scope="module", autouse=True)
def _build():
    util.build_oracle()




@pytest.mark.parametrize("name", list(util.BAYER))
@pytest.mark.parametrize("size", [(16, 16), (117, 131), (206, 206), (207, 113), (1024, 768)])
def test_rcd_oracle_equals_reference_strict(name, size):
    w, h = size
    m = util.frame_uniform(w, h, 1)
    m[::7, ::5] = 0.0
    m[3::11, 2::9] = -0.02
    got = util.oracle_rcd(m, util.BAYER[name])
    want = util.ref_rcd(m, util.BAYER[name], kind="strict")
    mask = util.oracle_rcd_mask(m, util.BAYER[name])
    bad = (~same_bits(got[..., :3], want[..., :3])).any(axis=2) & ((mask & 1) == 0)
    assert not bad.any()
    assert (mask & 1).sum() < 4 * (w + h)


def test_rcd_reference_undefined_pixels_are_real():
    """The masked set is where the reference itself is not a function of its input: poisoning its
    uninitialised scratch moves (some of) those pixels and nothing else."""
    m = util.frame_uniform(1024, 768, 2)
    f = util.BAYER["RGGB"]
    a = util.ref_rcd(m, f, kind="strict", poison=0.0)
    b = util.ref_rcd(m, f, kind="strict", poison=0.37)
    moved = (~same_bits(a[..., :3], b[..., :3])).any(axis=2)
    mask = util.oracle_rcd_mask(m, f)
    assert moved.any()
    assert not (moved & ((mask & 1) == 0)).any()


@pytest.mark.skipif(util.ref("fast") is None, reason="compares the reference's release build with its strict build: needs oracle/_ref")
def test_rcd_fast_build_distance_is_what_design_md_says():
    """The release (-ffast-math) build of the SAME reference source is not within 1 ulp of its own
    strict build; record the distribution the parity statement in DESIGN.md quotes."""
    m = util.frame_natural(1024, 768, util.SEEDS[0])
    f = util.BAYER["RGGB"]
    s = util.ref_rcd.__wrapped__(m, f, kind="strict")
    q = util.ref_rcd.__wrapped__(m, f, kind="fast")
    mask = util.oracle_rcd_mask(m, f)
    u = util.ulp_distance(s[..., :3], q[..., :3])[(mask & 1) == 0]
    assert (u > 1).mean() > 0.01          # the release build is NOT within 1 ulp of the source semantics
    assert np.abs(s[..., :3] - q[..., :3])[(mask & 1) == 0].max() < 1e-3


@pytest.mark.parametrize("kind,fp", [("strict", util.FP_STRICT), ("fast", util.FP_CONTRACT)])
def test_colour_oracle_equals_reference(kind, fp):
    enc, dec = util.srgb_encode_lut(), util.srgb_decode_lut()
    co_t, co_s = util.fit_unbounded_coeffs(enc), util.fit_unbounded_coeffs(dec)
    img = util.rgba_test_image(512, 384, 4)
    for kw in (dict(matrix=util.MATRIX_CAM_TO_REC2020),
               dict(matrix=util.MATRIX_CAM_TO_REC2020, clip=util.MATRIX_CLIP_IN),
               dict(matrix=util.MATRIX_CAM_TO_REC2020, lut_s=dec, co_s=co_s),
               dict(matrix=util.MATRIX_REC2020_TO_SRGB, lut_t=enc, co_t=co_t),
               dict(matrix=util.MATRIX_REC2020_TO_SRGB, clip=util.MATRIX_CLIP_IN, lut_s=dec, co_s=co_s, lut_t=enc, co_t=co_t)):
        r = util.ref_convert(img, kind=kind, **kw)
        o = util.oracle_convert(img, fp=fp, **kw)
        assert same_bits(r, o).all()


@pytest.mark.parametrize("scale", [0, 2, 5])
def test_eaw_oracle_equals_reference_strict(scale):
    rng = np.random.default_rng(scale)
    img = rng.normal(10, 1, (203, 301, 4)).astype(np.float32)
    oc, od, osum = util.oracle_eaw_decompose(img, scale, 1.7)
    rc, rd, rsum = util.ref_eaw_decompose(img, scale, 1.7)
    assert same_bits(oc, rc).all() and same_bits(od, rd).all()
    assert np.allclose(osum, rsum, rtol=2e-6)     # the reference sums in float, the oracle in double
    thr = (0.3, 0.2, 0.1, 0.0)
    assert same_bits(util.oracle_eaw_synthesize(img, od, thr), util.ref_eaw_synthesize(img, od, thr)).all()


# ---- golden vectors: produced by tests/golden/make_golden.py from oracle/_ref, committed ----------
def _golden(name):
    return np.load(os.path.join(util.GOLDEN_DIR, name))


@pytest.mark.parametrize("name", list(util.BAYER))
def test_rcd_oracle_equals_golden(name):
    g = _golden(f"rcd_{name}.npz")
    got = util.oracle_rcd(g["mosaic"], util.BAYER[name], tuple(g["pm"]))
    mask = util.oracle_rcd_mask(g["mosaic"], util.BAYER[name], tuple(g["pm"]))
    bad = (~same_bits(got[..., :3], g["rgb_strict"][..., :3])).any(axis=2) & ((mask & 1) == 0)
    assert not bad.any()


@pytest.mark.parametrize("case", ["colorin_matrix", "colorin_clip", "colorout_trc"])
def test_colour_oracle_equals_golden(case):
    g = _golden(f"color_{case}.npz")
    kw = dict(matrix=g["matrix"])
    if "clip" in g.files:
        kw["clip"] = g["clip"]
    if "lut_t_row" in g.files:
        kw["lut_t"] = np.ascontiguousarray(np.tile(g["lut_t_row"], (3, 1)))
        kw["co_t"] = g["co_t"]
    assert same_bits(util.oracle_convert(g["rgba"], fp=util.FP_STRICT, **kw), g["out_strict"]).all()
    assert same_bits(util.oracle_convert(g["rgba"], fp=util.FP_CONTRACT, **kw), g["out_fast"]).all()


def test_eaw_oracle_equals_golden():
    g = _golden("eaw.npz")
    for scale in (0, 3):
        oc, od, _ = util.oracle_eaw_decompose(g["img"], scale, float(g["inv_sigma2"]))
        assert same_bits(oc, g[f"coarse_{scale}"]).all() and same_bits(od, g[f"detail_{scale}"]).all()
    assert same_bits(util.oracle_eaw_synthesize(g["img"], g["detail_0"], tuple(g["thr"])), g["synth"]).all()


@util.recorded(lambda color_mode, new_vst, img, fwd, plan, oracle_back: (fwd, oracle_back))
def _ref_dn_vst(color_mode, new_vst, img, fwd, plan, oracle_back):
    """the reference's forward and inverse transforms of `img` / `fwd` with the parameters of the oracle's plan (the oracle's
    results, `fwd` and `oracle_back`, are what a recording is stored against)"""
    R, f4 = util.ref("strict"), (lambda v: (C.c_float * 4)(*v))
    h, w = img.shape[:2]
    wb, p, a_eff, b, bias = plan[1:5], plan[5:9], plan[9], plan[10], plan[11]
    toY, toRGB, aa, bb = plan[12:24].copy(), plan[24:36].copy(), plan[36:40], plan[40:44]
    rf, rb = np.zeros_like(img), fwd.copy()
    if not new_vst:
        R.ref_dn_precondition(util.fptr(img), util.fptr(rf), w, h, f4(aa), f4(bb))
        R.ref_dn_backtransform(util.fptr(rb), w, h, f4(aa), f4(bb))
    elif color_mode == 0:
        R.ref_dn_precondition_v2(util.fptr(img), util.fptr(rf), w, h, C.c_float(a_eff), f4(p), C.c_float(b), f4(wb))
        R.ref_dn_backtransform_v2(util.fptr(rb), w, h, C.c_float(a_eff), f4(p), C.c_float(b), C.c_float(bias), f4(wb))
    else:
        R.ref_dn_precondition_Y0U0V0(util.fptr(img), util.fptr(rf), w, h, C.c_float(a_eff), f4(p), C.c_float(b), util.fptr(toY))
        R.ref_dn_backtransform_Y0U0V0(util.fptr(rb), w, h, C.c_float(a_eff), f4(p), C.c_float(b), C.c_float(bias), f4(wb), util.fptr(toRGB))
    return rf, rb


@util.recorded()
def _ref_dn_call(fn, out_sizes, *args):
    """one of the reference's denoise helpers: float32 outputs of `out_sizes` first, then `args` (4-tuples become float[4],
    float32 arrays pointers)"""
    outs = [np.zeros(n, np.float32) for n in out_sizes]
    conv = [(C.c_float * 4)(*a) if isinstance(a, tuple) else util.fptr(a) if isinstance(a, np.ndarray) else a for a in args]
    getattr(util.ref("strict"), fn)(*[util.fptr(o) for o in outs], *conv)
    return tuple(outs)


@pytest.mark.parametrize("color_mode,new_vst", [(1, True), (0, True), (0, False)])
def test_denoise_vst_oracle_equals_reference(color_mode, new_vst):
    """precondition/backtransform{,_v2,_Y0U0V0} cut verbatim from iop/denoiseprofile.c:852-1089."""
    import ctypes as C
    import ansel_b200 as ab
    O = util.oracle()
    f4 = lambda v: (C.c_float * 4)(*v)  # noqa: E731
    wbc, pm = (2.0, 1.0, 1.5, 0.0), (1.0, 1.0, 1.0, 1.0)
    img = util.rgba_scene(300, 200, 1)
    img[..., 3] = 0.3
    npx = 300 * 200
    d = ab.denoiseprofile_data(ab.DENOISE_WAVELETS, color_mode=color_mode, use_new_vst=new_vst, b=(0.0, 1e-6, 0.0))
    plan = np.zeros(51, np.float32)
    O.orc_dn_plan_export(C.byref(d), C.c_float(1.0), 6000, 4000, f4(wbc), f4(pm), util.fptr(plan))
    fwd, back = np.zeros_like(img), np.zeros_like(img)
    O.orc_dn_vst(1, C.byref(d), C.c_float(1.0), 6000, 4000, f4(wbc), f4(pm), util.fptr(img), util.fptr(fwd), C.c_size_t(npx))
    O.orc_dn_vst(0, C.byref(d), C.c_float(1.0), 6000, 4000, f4(wbc), f4(pm), util.fptr(fwd), util.fptr(back), C.c_size_t(npx))
    rf, rb = _ref_dn_vst(color_mode, new_vst, img, fwd, plan, back)
    assert same_bits(fwd, rf).all() and same_bits(back, rb).all()
    assert np.abs(back[..., :3] - img[..., :3]).max() < 1e-3  # the pair is (nearly) an inverse


def test_denoise_plan_pieces_equal_reference():
    """compute_wb_factors, set_up_conversion_matrices, variance_stabilizing_xform (denoiseprofile.c:1098-1286)."""
    import ctypes as C
    import ansel_b200 as ab
    O = util.oracle()
    f4 = lambda v: (C.c_float * 4)(*v)  # noqa: E731
    wbc, pm = (2.0, 1.0, 1.5, 0.0), (1.0, 1.0, 1.0, 1.0)
    d = ab.denoiseprofile_data(ab.DENOISE_WAVELETS)
    a = np.zeros(4, np.float32)
    O.orc_dn_wb_factors(util.fptr(a), C.byref(d), f4(wbc), f4(pm), f4((2, 1, 2, 0)))
    assert same_bits(a, _ref_dn_call("ref_dn_wb_factors", (4,), 1, 1, wbc, pm, (2, 1, 2, 0))[0]).all()
    tY, tR = _ref_dn_call("ref_dn_conversion_matrices", (12, 12), a)
    plan = np.zeros(51, np.float32)
    O.orc_dn_plan_export(C.byref(d), C.c_float(1.0), 6000, 4000, f4(wbc), f4(pm), util.fptr(plan))
    k = np.float32(d.strength) * np.float32(2.5) * np.float32(1.0)
    assert same_bits((tY / k).astype(np.float32), plan[12:24]).all() and same_bits((tR * k).astype(np.float32), plan[24:36]).all()
    assert plan[0] == 7
    force = np.ascontiguousarray(np.array(d.force, np.float32))
    for cm in (0, 1):
        d.wavelet_color_mode = cm
        t1 = np.zeros(4, np.float32)
        sums = (3e7, 2.5e7, 2.8e7, 1.0)
        O.orc_wavelet_thresholds(util.fptr(t1), 2, 7, C.c_size_t(45441024), f4(sums), C.c_float(plan[46]), C.byref(d))
        assert same_bits(t1, _ref_dn_call("ref_dn_thresholds", (4,), 2, 7, C.c_size_t(45441024), sums, cm, force)[0]).all()


FILMIC_CASES = {"default_v8": {}, "no_bleach": dict(version=5), "high_bleach_hue": dict(version=8, saturation=60.0),
                "poly_curves": dict(shadows=0, highlights=1), "rational_curves": dict(shadows=2, highlights=2, contrast=1.5),
                "wide_dr_gamma22": dict(white_point_source=6.0, black_point_source=-10.0, output_power=2.2)}


@pytest.mark.parametrize("name", list(FILMIC_CASES))
def test_filmic_oracle_equals_reference(name):
    """filmic_agx and everything under it, cut verbatim from iop/filmicrgb.c:948-2649; piece->data from the
    reference's own commit_params (:4005-4113)."""
    work, export = util.profile_pair(util.REC2020_TO_XYZ_D50), util.profile_pair(util.SRGB_TO_XYZ_D50)
    img = util.hdr_rgba(400, 300, 5)
    blob = util.ref_filmic_commit(util.filmic_default_params(**FILMIC_CASES[name]))
    for e in (export, None):
        assert same_bits(util.ref_filmic_agx(img, blob, work, e), util.oracle_filmic_agx(img, blob, work, e)).all()
    for v in (5, 6, 7, 8, 9):
        assert same_bits(util.ref_filmic_prepare(v, work, export),
                         util.filmic_prepare(util.oracle(), "orc_filmic_prepare", v, work, export)).all()


def test_filmic_oracle_equals_golden():
    g = _golden("filmic_agx.npz")
    blob = _golden("filmic_data.npz")["default_v8"]
    work, export = util.profile_pair(util.REC2020_TO_XYZ_D50), util.profile_pair(util.SRGB_TO_XYZ_D50)
    assert same_bits(util.oracle_filmic_agx(g["img"], blob, work, export), g["out_export"]).all()
    assert same_bits(util.oracle_filmic_agx(g["img"], blob, work, None), g["out_work"]).all()
    assert same_bits(util.filmic_prepare(util.oracle(), "orc_filmic_prepare", 7, work, export), g["prepare"]).all()


def test_filmic_abi_layout_matches_reference():
    import ctypes as C
    import ansel_b200 as ab
    assert C.sizeof(ab.FilmicPiece) == 1088
    for fn, want in (("ref_filmic_sizeof_data", 832), ("ref_filmic_offsetof_spline", 128), ("ref_filmic_sizeof_spline", 144),
                     ("ref_filmic_offsetof_noise_distribution", 272), ("ref_filmic_sizeof_params", 112)):
        assert util.ref_size_t(fn) == want


NLM_CONFIGS = [dict(), dict(P=2, K=4, scattering=0.5), dict(center_weight=-1.0, sharpness=0.01, luma=0.8, chroma=0.6, K=3, P=3),
               dict(K=2, P=1, scattering=1.0, scale=0.7), dict(P=4, K=2), dict(P=0, K=3), dict(K=5, decimate=1)]


@pytest.mark.parametrize("cfg", range(len(NLM_CONFIGS)))
def test_nlmeans_oracle_equals_reference(cfg):
    """pixel/nlmeans_core.c compiled in place; chunked, order-dependent float accumulation."""
    for (w, h) in ((200, 150), (73, 61), (301, 203)):
        img = (util.rgba_scene(w, h, 2, noise=0.02) * 60).astype(np.float32)
        assert same_bits(util.oracle_nlmeans(img, **NLM_CONFIGS[cfg]), util.ref_nlmeans(img, **NLM_CONFIGS[cfg])).all()


def test_nlmeans_oracle_equals_golden():
    g = _golden("nlmeans.npz")
    assert same_bits(util.oracle_nlmeans(g["img"]), g["out_profiled"]).all()
    assert same_bits(util.oracle_nlmeans(g["img"], center_weight=-1.0, sharpness=0.01, luma=0.8, chroma=0.6, K=3, P=2), g["out_lab"]).all()


LL_PARAMS = [dict(), dict(sigma=0.2, shadows=1.5, highlights=0.1, clarity=1.0), dict(sigma=0.8, shadows=-0.5, highlights=1.8, clarity=-0.6)]


@pytest.mark.parametrize("p", range(len(LL_PARAMS)))
def test_local_laplacian_oracle_equals_reference(p):
    """pixel/locallaplacian.c compiled in place; channel 0 is the filter output, 1,2 copies, 3 untouched."""
    for (w, h) in ((200, 150), (257, 129), (64, 48), (33, 17), (9, 4), (4, 4)):
        img = util.lab_scene(w, h, 5)
        assert same_bits(util.oracle_local_laplacian(img, **LL_PARAMS[p]), util.ref_local_laplacian(img, **LL_PARAMS[p])).all()


def test_local_laplacian_oracle_equals_golden():
    g = _golden("ll.npz")
    assert same_bits(util.oracle_local_laplacian(g["img"]), g["out_default"]).all()
    assert same_bits(util.oracle_local_laplacian(g["img"], **LL_PARAMS[1]), g["out_strong"]).all()


def _diffuse_cases():
    import ansel_b200 as ab
    out = {}
    for name, kw in ab.DIFFUSE_PRESETS.items():
        kw = dict(kw)
        kw["iterations"] = min(kw.get("iterations", 1), 3)       # the stock counts (up to 32) only repeat the same step
        out[name] = kw
    out["gradient_sharpen"] = dict(iterations=2, radius=16, radius_center=4, sharpness=0.3, regularization=3.0, variance_threshold=-1.0,
                                   anisotropy_first=-3.0, anisotropy_second=2.0, anisotropy_third=-0.5, anisotropy_fourth=5.0,
                                   first=0.3, second=-0.6, third=0.8, fourth=-1.0)
    out["masked_all_orders"] = dict(iterations=2, radius=8, threshold=0.5, regularization=1.5, anisotropy_first=1.0, anisotropy_second=-1.0,
                                    anisotropy_third=-2.0, anisotropy_fourth=3.0, first=0.5, second=0.3, third=-0.2, fourth=0.1)
    return out


@pytest.mark.parametrize("name", list(_diffuse_cases()))
def test_diffuse_oracle_equals_reference(name):
    """iop/diffuse.c process() cut verbatim + pixel/bspline.h; NaN/inf/negative input included (hdr_rgba)."""
    import ansel_b200 as ab
    d = ab.diffuse_data(**_diffuse_cases()[name])
    for (w, h), zoom in (((160, 120), 1.0), ((97, 61), 1.0), ((120, 90), 2.0), ((40, 7), 0.5)):
        img = util.hdr_rgba(w, h, 3)
        assert same_bits(util.oracle_diffuse(img, d, iscale=zoom), util.ref_diffuse(img, d, iscale=zoom)).all()


def test_diffuse_oracle_equals_golden():
    import ansel_b200 as ab
    g = _golden("diffuse.npz")
    for name in ("sharpen_demosaic_aa", "gradient_sharpen", "inpaint_highlights"):
        assert same_bits(util.oracle_diffuse(g["img"], ab.diffuse_data(**_diffuse_cases()[name])), g[name]).all()


def test_libm_sinf_cosf_restatement_equals_system_libm():
    """glibc sinf/cosf as iop/noise_generator.h:93-96 reaches them: EVERY argument the Box-Muller call can produce,
    (float)(2*pi*k/2^24), plus a stride through all floats below 120."""
    L = util.oracle()
    FP = C.POINTER(C.c_float)

    def run(fn, x):
        out = np.empty_like(x)
        getattr(L, fn)(x.ctypes.data_as(FP), out.ctypes.data_as(FP), C.c_size_t(x.size))
        return out
    k = np.arange(1 << 24, dtype=np.float64)
    u = np.arange(0, 0x42F00000, 211, dtype=np.uint32)
    for x in (((2.0 * np.pi) * (k * 2.0 ** -24)).astype(np.float32), np.concatenate([u.view(np.float32), (u | 0x80000000).view(np.float32)])):
        for f in ("sinf", "cosf"):
            assert (run(f"orc_{f}_array", x).view(np.uint32) == run(f"sys_{f}_array", x).view(np.uint32)).all(), f


WORK_PROFILE = util.profile_pair(util.REC2020_TO_XYZ_D50)


def test_lab_glue_oracle_equals_reference():
    """colorprofiles/iop_profile.c _transform_rgb_to_lab_matrix / _transform_lab_to_rgb_matrix cut verbatim."""
    rgb = util.hdr_rgba(333, 217, 6)                     # negatives, zeros, NaN, inf, > 1
    assert same_bits(util.oracle_rgb_to_lab(rgb, WORK_PROFILE), util.ref_rgb_to_lab(rgb, WORK_PROFILE)).all()
    lab = util.lab_scene(333, 217, 6)
    lab[5, 5, :3] = (0.0, 0.0, 0.0)
    lab[6, 6, :3] = (7.9, -300.0, 250.0)                 # both branches of lab_f_inv
    lab[7, 7, 0] = np.nan
    assert same_bits(util.oracle_lab_to_rgb(lab, WORK_PROFILE), util.ref_lab_to_rgb(lab, WORK_PROFILE)).all()


def test_lab_glue_oracle_equals_golden():
    g = _golden("labglue.npz")
    assert same_bits(util.oracle_rgb_to_lab(g["rgb"], WORK_PROFILE), g["lab_of_rgb"]).all()
    assert same_bits(util.oracle_lab_to_rgb(g["lab"], WORK_PROFILE), g["rgb_of_lab"]).all()
    d, cd, e, ce = _srgb_curves(False)
    assert same_bits(util.oracle_rgb_to_lab_trc(g["rgb"], SRGB_PROFILE, d, cd), g["lab_of_rgb_trc"]).all()
    assert same_bits(util.oracle_lab_to_rgb_trc(g["lab"], SRGB_PROFILE, e, ce), g["rgb_of_lab_trc"]).all()


SRGB_PROFILE = util.profile_pair(util.SRGB_TO_XYZ_D50)


def _srgb_curves(partial):
    """the sRGB TRC as lut_in (decode) / lut_out (encode); partial: one channel of each marked linear"""
    d, e = util.srgb_decode_lut(), util.srgb_encode_lut()
    if partial:
        d[1, 0] = -1.0
        e[2, 0] = -1.0
    return d, util.fit_unbounded_coeffs(d), e, util.fit_unbounded_coeffs(e)


@pytest.mark.parametrize("partial", [False, True])
def test_lab_glue_with_tone_curves_oracle_equals_reference(partial):
    """_apply_tonecurves + the two matrix loops cut verbatim, for a profile with tone curves (sRGB)"""
    d, cd, e, ce = _srgb_curves(partial)
    rgb, lab = util.hdr_rgba(333, 217, 6), util.lab_scene(333, 217, 6)
    assert same_bits(util.oracle_rgb_to_lab_trc(rgb, SRGB_PROFILE, d, cd), util.ref_rgb_to_lab_trc(rgb, SRGB_PROFILE, d, cd, e, ce)).all()
    assert same_bits(util.oracle_lab_to_rgb_trc(lab, SRGB_PROFILE, e, ce), util.ref_lab_to_rgb_trc(lab, SRGB_PROFILE, d, cd, e, ce)).all()
    # the flag comes from the input curves alone: three linear lut_in switch the output curves off as well
    d[:, 0] = -1.0
    cd = util.fit_unbounded_coeffs(d)
    assert same_bits(util.ref_lab_to_rgb_trc(lab, SRGB_PROFILE, d, cd, e, ce), util.ref_lab_to_rgb(lab, SRGB_PROFILE)).all()
    assert same_bits(util.ref_rgb_to_lab_trc(rgb, SRGB_PROFILE, d, cd, e, ce), util.ref_rgb_to_lab(rgb, SRGB_PROFILE)).all()


@pytest.mark.parametrize("scale,pipe,prev", [(1.0, 1, 0), (0.5, 1, 0), (2.5, 2, 0), (0.3, 4, 0), (0.4, 3, 1)])
def test_nlmeans_iop_oracle_equals_reference(scale, pipe, prev):
    """iop/nlmeans.c process_cpu cut verbatim: P, K, sharpness, Lab norms, decimation, mask alpha copy."""
    import ansel_b200 as ab
    img = util.lab_scene(150, 110, 3)
    for d in (ab.nlmeans_data(), ab.nlmeans_data(radius=1.0, strength=120.0, luma=1.0, chroma=1.0)):
        dec = 1 if (pipe == 4 or prev) else 0
        for mask in (0, 1):
            got = util.oracle_nlmeans_iop(img, d, scale, dec, mask)
            want = util.ref_nlmeans_iop(img, d, scale, pipe, prev, mask)
            assert same_bits(got, want).all()


@pytest.mark.parametrize("passes", [1, 3, 5])
def test_color_smoothing_oracle_equals_reference(passes):
    """iop/demosaic/basic.c color_smoothing cut verbatim (median network, alpha lane as scratch)."""
    for (w, h) in ((200, 150), (33, 17), (3, 3), (2, 5)):
        img = util.hdr_rgba(w, h, 4) if w > 8 else util.rgba_test_image(w, h, 4)
        assert same_bits(util.oracle_color_smoothing(img, passes), util.ref_color_smoothing(img, passes)).all()


@pytest.mark.parametrize("name", list(util.BAYER))
@pytest.mark.parametrize("mode", [1, 2, 3])
def test_green_eq_oracle_equals_reference(name, mode):
    """green_equilibration_lavg / _favg cut verbatim; ROI phases; the reference called with one thread so that its
    reduction order is the raster order the oracle uses."""
    os.environ["OMP_NUM_THREADS"] = "1"
    for (w, h), (x, y), iso in (((214, 135), (0, 0), 100.0), ((101, 77), (1, 0), 800.0), ((64, 48), (1, 1), 6400.0), ((5, 4), (0, 1), 100.0)):
        m = util.frame_natural(w, h, 9, filters=util.BAYER[name], iso=iso)
        got, want = util.oracle_green_eq(m, util.BAYER[name], mode, x, y, iso), util.ref_green_eq(m, util.BAYER[name], mode, x, y, iso)
        if mode == 1:
            assert same_bits(got, want).all()
        else:  # the full average's sums are an OpenMP reduction: order-dependent in the last bits of a double
            assert util.ulp_distance(got, want).max() <= 1 and (~same_bits(got, want)).mean() < 1e-3


def test_demosaic_extras_oracle_equals_golden():
    g = _golden("demosaic_extra.npz")
    assert same_bits(util.oracle_color_smoothing(g["rgba"], 2), g["smoothed2"]).all()
    assert same_bits(util.oracle_green_eq(g["mosaic"], util.BAYER["RGGB"], 1, iso=400.0), g["geq_local"]).all()
    assert util.ulp_distance(util.oracle_green_eq(g["mosaic"], util.BAYER["RGGB"], 3, iso=400.0), g["geq_both"]).max() <= 1


LEGACY_EXTRA = [{}, dict(saturation=20.0), dict(saturation=-15.0, shadows=0, highlights=2, contrast=1.4)]


@pytest.mark.parametrize("version", [0, 1, 2, 3, 4])
def test_filmic_legacy_oracle_equals_reference(version):
    """filmic_split/chroma_v1, _v2_v3, _v4 and filmic_v5 cut verbatim from filmicrgb.c, every norm, with/without an
    export profile; piece->data from the reference's own commit_params()."""
    work, export = util.profile_pair(util.REC2020_TO_XYZ_D50), util.profile_pair(util.SRGB_TO_XYZ_D50)
    img = util.hdr_rgba(160, 100, 7)
    for pc in range(6):
        for extra in LEGACY_EXTRA:
            blob = util.ref_filmic_commit(util.filmic_default_params(version=version, preserve_color=pc, **extra))
            for ex in (export, None):
                assert same_bits(util.oracle_filmic_legacy(img, blob, work, ex), util.ref_filmic_legacy(img, blob, work, ex)).all(), (pc, extra)


def test_filmic_legacy_oracle_equals_golden():
    g = _golden("filmic_legacy.npz")
    work, export = util.profile_pair(util.REC2020_TO_XYZ_D50), util.profile_pair(util.SRGB_TO_XYZ_D50)
    for key in [k for k in g.files if k.startswith("out_")]:
        tag = key[4:]
        assert same_bits(util.oracle_filmic_legacy(g["img"], g["data_" + tag], work, export), g[key]).all(), tag


@pytest.mark.parametrize("name", list(util.BAYER))
def test_amaze_oracle_equals_reference(name):
    """iop/demosaic/amaze.cc compiled in place, one thread (its scratch is carried from tile to tile in raster order:
    oracle scratch_mode 0); several tiles, ragged edges, clip points above and below the data."""
    f = util.BAYER[name]
    for (w, h), pm, gain in (((320, 240), (1.0, 1.0, 1.0), 1.0), ((501, 333), (0.8, 1.0, 0.9), 1.3), ((129, 161), (2.0, 2.0, 2.0), 1.0), ((33, 34), (1.0, 1.0, 1.0), 1.0)):
        m = (util.frame_natural(w, h, 5, filters=f) * gain).astype(np.float32)
        assert same_bits(util.oracle_amaze(m, f, pm, 0), util.ref_amaze(m, f, pm)).all()


def test_amaze_edge_inputs_and_scratch_modes():
    f = util.BAYER["RGGB"]
    for kind in ("zeros", "ones", "impulses", "negative", "tiny"):
        m = util.frame_edge(300, 200, kind)
        assert same_bits(util.oracle_amaze(m, f, scratch_mode=0), util.ref_amaze(m, f)).all(), kind
    # the reference is thread-count dependent through its carried scratch; zeroing it per tile moves only a few pixels
    m = util.frame_natural(1300, 900, 6)
    a0, a1 = util.oracle_amaze(m, f, scratch_mode=0), util.oracle_amaze(m, f, scratch_mode=1)
    moved = (~same_bits(a0, a1)).any(axis=2).mean()
    assert 0 < moved < 1e-3
    r8 = util.ref_amaze(m, f, threads=8)
    assert (~same_bits(r8, a0)).any(axis=2).mean() < 1e-3      # ... as many as the reference moves by itself


def test_amaze_oracle_equals_golden():
    g = _golden("amaze.npz")
    assert same_bits(util.oracle_amaze(g["mosaic"], util.BAYER["RGGB"], scratch_mode=0)[..., :3], g["rgb_carried"][..., :3]).all()


# ---- filmic's highlight reconstruction (a16) ------------------------------------------------------------------------
RECONSTRUCT_CASES = {
    "rgb_only_gaussian": dict(reconstruct_threshold=0.0, reconstruct_feather=3.0, reconstruct_bloom_vs_details=40.0, reconstruct_grey_vs_color=-30.0,
                              reconstruct_structure_vs_texture=20.0, noise_level=0.2, high_quality_reconstruction=0, noise_distribution=1),
    "default_poisson": dict(reconstruct_threshold=-1.0, noise_level=0.1),                      # hq 1, poissonian, sliders at +100 %
    "two_passes_uniform_v3": dict(reconstruct_threshold=-0.5, reconstruct_feather=1.5, reconstruct_bloom_vs_details=-50.0, reconstruct_grey_vs_color=10.0,
                                  reconstruct_structure_vs_texture=-70.0, noise_level=0.5, high_quality_reconstruction=2, noise_distribution=0, version=2),
}


def _reconstruct_frames():
    return {"scene": (util.rgba_scene(333, 217, 4) * 2.0).astype(np.float32), "hdr": util.hdr_rgba(200, 150, 3),
            "dark": (util.rgba_scene(100, 80, 4) * 0.01).astype(np.float32), "tiny": (util.rgba_scene(7, 5, 4) * 3).astype(np.float32)}


@pytest.mark.parametrize("name", list(RECONSTRUCT_CASES))
def test_filmic_reconstruct_oracle_equals_reference(name):
    """process() :2729-2838 replayed on mask_clipped_pixels / inpaint_noise / reconstruct_highlights / compute_ratios /
    restore_ratios cut verbatim; every noise distribution, 0-2 ratio passes, zoomed pipes, a frame with nothing to recover"""
    d = util.ref_filmic_commit(util.filmic_default_params(**RECONSTRUCT_CASES[name]))
    assert d[84:88].view(np.int32)[0] == 0                   # hl_deprecated off: the path is live
    for fname, img in _reconstruct_frames().items():
        for kw in ({}, dict(iscale=2.0, roi_scale=0.3, buf=(4000, 3000))):
            r, o = util.ref_filmic_reconstruct(img, d, **kw), util.oracle_filmic_reconstruct(img, d, **kw)
            assert r[0] == o[0] == (0 if fname == "dark" else 1), fname
            assert same_bits(r[2], o[2]).all() and same_bits(r[1], o[1]).all(), (fname, kw)


def test_filmic_reconstruct_oracle_equals_golden():
    g = _golden("filmic_reconstruct.npz")
    for name in RECONSTRUCT_CASES:
        rc, frame, mask = util.oracle_filmic_reconstruct(g["img"], g["data_" + name])
        assert rc == 1 and same_bits(frame, g["frame_" + name]).all() and same_bits(mask, g["mask_" + name]).all()


@util.recorded(lambda img, plan, center_weight, oracle_out: oracle_out)
def _ref_dn_nlmeans_module(img, plan, center_weight, oracle_out):
    """precondition_v2 -> nlmeans_denoise -> backtransform_v2 of the reference, with the parameters of the oracle's plan (the
    oracle's module output `oracle_out` is what a recording is stored against)"""
    R, f4 = util.ref("strict"), (lambda v: (C.c_float * 4)(*v))
    h, w = img.shape[:2]
    wb, p, a_eff, b, bias = plan[1:5], plan[5:9], plan[9], plan[10], plan[11]
    pre = np.zeros_like(img)
    R.ref_dn_precondition_v2(util.fptr(img), util.fptr(pre), w, h, C.c_float(a_eff), f4(p), C.c_float(b), f4(wb))
    nlm = util.ref_nlmeans(pre, kind="strict", sharpness=float(np.float32(0.045) / np.float32(9)), center_weight=center_weight, P=1, K=7)
    buf = np.ascontiguousarray(nlm)
    R.ref_dn_backtransform_v2(util.fptr(buf), w, h, C.c_float(a_eff), f4(p), C.c_float(b), C.c_float(bias), f4(wb))
    return buf


def test_denoiseprofile_nlmeans_module_is_the_reference_pieces_in_order():
    """process_nlmeans_cpu(), denoiseprofile.c:1599-1648, composed from the reference's own precondition_v2, nlmeans_denoise and
    backtransform_v2 with the parameters nlmeans_precondition() :1500-1533 derives (exported by the oracle's NLM plan): what
    bench.py's CPU arm runs for the denoise node of the C3 chain, and what the oracle's module-level entry point restates"""
    import ctypes as C
    import ansel_b200 as ab
    O = util.oracle()
    f4 = lambda v: (C.c_float * 4)(*v)  # noqa: E731
    w, h = 300, 200
    img = util.rgba_scene(w, h, 5)
    d = ab.denoiseprofile_data(ab.DENOISE_NLMEANS, radius=1, nbhood=7)
    wbc, pm = (2.0, 1.0, 1.5, 0.0), (1.0, 1.0, 1.0, 1.0)
    plan = np.zeros(51, np.float32)
    O.orc_dn_plan_export_nlm(C.byref(d), C.c_float(1.0), w, h, f4(wbc), f4(pm), util.fptr(plan))
    f = O.orc_denoiseprofile_nlmeans
    f.restype = C.c_int
    want = np.zeros_like(img)
    assert f(util.fptr(img), util.fptr(want), w, h, C.byref(d), C.c_float(1.0), 1, f4(wbc), f4(pm)) == 0
    buf = _ref_dn_nlmeans_module(img, plan, float(np.float32(d.central_pixel_weight)), want)
    assert same_bits(buf, want).all()
