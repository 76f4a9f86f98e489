"""CPU: the oracle of the modules either side of the demosaic .. colorout path (rawprepare, temperature, highlights' clip
mode and bypass, exposure, gamma, the export's float -> integer conversions) pinned bit for bit against the reference's
own lines compiled in place (oracle/_ref, strict build), and against the golden vectors those builds produced
(tests/golden/pipe_ends.npz), which travel to the GPU box."""
import os

import numpy as np
import pytest

import ansel_b200 as ab
import pipe_ends_util as pe
import util


def same_bits(a, b):
    return (a.view(np.uint32) == b.view(np.uint32)) | (np.isnan(a) & np.isnan(b))


@pytest.fixture(scope="module", autouse=True)
def _build():
    import subprocess
    subprocess.run(["make", "-s", "-C", util.ORACLE_DIR, "oracle"], check=True)   # dependency-tracked; oracle/_ref comes from build()
    if util.ref("strict") is None and os.path.isdir("/root/reference/src"):
        util.build_oracle()



SUB = (512.0, 520.0, 508.0, 515.0)
DIV = (15871.0, 15863.0, 15875.0, 15868.0)


def gain_maps(mw=9, mh=7, seed=3):
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:mh, 0:mw]
    r2 = ((xx / (mw - 1) - 0.5) ** 2 + (yy / (mh - 1) - 0.5) ** 2)
    return np.stack([(1.0 + (0.6 + 0.1 * f) * r2 + rng.normal(0, 0.01, r2.shape)).astype(np.float32) for f in range(4)])


RAWPREPARE_CASES = {
    "uint16": dict(),
    "uint16_crop": dict(x=3, y=5),
    "uint16_odd_sizes": dict(size=(131, 77), x=1, y=0),
    "uint16_roi": dict(x=2, y=2, out=(7, 4, 90, 50)),
    "float_mosaic": dict(datatype=ab.TYPE_FLOAT, x=4, y=1),
    "uint16_scaled": dict(x=8, y=6, scale=0.5),
    "uint16_gainmaps": dict(x=2, y=4, gain=True),
    "rgba_predownsampled": dict(datatype=ab.TYPE_FLOAT, filters=0, channels=4, x=2, y=3),
    "mono_unknown_type": dict(datatype=ab.TYPE_UNKNOWN, filters=0, channels=1),
}


def rawprepare_case(name, size=(134, 78)):
    kw = dict(RAWPREPARE_CASES[name])
    w, h = kw.pop("size", size)
    gain = gain_maps() if kw.pop("gain", False) else None
    spacing, origin = (1.0 / 8, 1.0 / 6), (0.01, -0.02)
    d = ab.rawprepare_data(SUB, DIV, kw.pop("x", 0), kw.pop("y", 0), gain=gain, spacing=spacing, origin=origin)
    ch, datatype = kw.get("channels", 1), kw.get("datatype", ab.TYPE_UINT16)
    raw = pe.sensor_frame(w * ch, h, 11)
    src = raw if datatype == ab.TYPE_UINT16 else raw.astype(np.float32)
    piece = pe.rawprepare_piece(w, h, d, **kw)
    return piece, src, dict(gain=gain, spacing=spacing, origin=origin)


@pytest.mark.parametrize("name", list(RAWPREPARE_CASES))
def test_rawprepare_oracle_equals_reference(name):
    piece, src, g = rawprepare_case(name)
    want = pe.ref_rawprepare(piece, src, **g)
    assert same_bits(pe.oracle_rawprepare(piece, src), want).all()
    assert np.isfinite(want).all() and want.std() > 0


TEMPERATURE_CASES = {
    "bayer": dict(),
    "bayer_roi_odd": dict(x=3, y=1, size=(131, 77)),
    "bayer_gbrg": dict(filters=util.BAYER["GBRG"], x=1, y=2),
    "xtrans": dict(filters=9, xtrans=pe.XTRANS, x=4, y=5, size=(133, 70)),
    "rgba": dict(filters=0, channels=4),
    "rgba_mask": dict(filters=0, channels=4, mask_display=1),
}
COEFFS = (2.13, 1.0, 1.57, 1.02)


def temperature_case(name):
    kw = dict(TEMPERATURE_CASES[name])
    w, h = kw.pop("size", (134, 78))
    piece = pe.mosaic_piece(w, h, ab.temperature_data(COEFFS), **kw)
    img = util.rgba_test_image(w, h, 5) if piece.channels == 4 else util.frame_natural(w, h, 5)
    return piece, img


@pytest.mark.parametrize("name", list(TEMPERATURE_CASES))
def test_temperature_oracle_equals_reference(name):
    piece, img = temperature_case(name)
    assert same_bits(pe.oracle_temperature(piece, img), pe.ref_temperature(piece, img)).all()


HIGHLIGHTS_CASES = {
    "clip_mosaic": dict(),
    "clip_mosaic_wb_maximum": dict(pm=(2.13, 1.0, 1.57, 0.0), clip=0.9),
    "clip_mosaic_24_clipped": dict(n_clipped=24),          # one short of DT_HL_MIN_CLIPPED_PIXELS: copied through
    "clip_mosaic_25_clipped": dict(n_clipped=25),
    "clip_rgba": dict(filters=0, channels=4),
    "clip_rgba_mask_zero_maximum": dict(filters=0, channels=4, mask_display=1, pm=(0.0, 0.0, 0.0, 0.0)),
    "lch_on_rgba_is_clip": dict(filters=0, channels=4, mode=ab.HIGHLIGHTS_LCH),
    "harmonic_bypass": dict(mode=ab.HIGHLIGHTS_HARMONIC, n_clipped=3),   # the default mode on a frame with nothing to reconstruct
    "inpaint_bypass_rgba": dict(filters=0, channels=4, mode=ab.HIGHLIGHTS_INPAINT, n_clipped=10),
    "inpaint_mosaic": dict(mode=ab.HIGHLIGHTS_INPAINT, clip=0.95),                    # colour inpainting along rows and columns
    "inpaint_mosaic_wb_roi": dict(mode=ab.HIGHLIGHTS_INPAINT, clip=0.9, pm=(2.13, 1.0, 1.57, 0.0), x=3, y=1, filters=util.BAYER["GBRG"]),
    "inpaint_mosaic_bypass": dict(mode=ab.HIGHLIGHTS_INPAINT, n_clipped=5),
    "lch_mosaic": dict(mode=ab.HIGHLIGHTS_LCH, clip=0.95),                            # 2x2 blocks rebuilt in LCh, long double constants
    "lch_mosaic_wb_roi": dict(mode=ab.HIGHLIGHTS_LCH, clip=0.9, pm=(2.13, 1.0, 1.57, 0.0), x=3, y=1, filters=util.BAYER["GRBG"]),
    "lch_mosaic_bypass": dict(mode=ab.HIGHLIGHTS_LCH, n_clipped=12),
    "lch_xtrans": dict(mode=ab.HIGHLIGHTS_LCH, clip=0.95, filters=9, xtrans=pe.XTRANS, x=1, y=4),
    "inpaint_xtrans_wb": dict(mode=ab.HIGHLIGHTS_INPAINT, clip=0.9, filters=9, xtrans=pe.XTRANS, x=3, y=2, pm=(2.13, 1.0, 1.57, 0.0)),
    "clip_xtrans": dict(filters=9, xtrans=pe.XTRANS),
}


def highlights_case(name, size=(134, 78)):
    kw = dict(HIGHLIGHTS_CASES[name])
    w, h = size
    mode, clip, n = kw.pop("mode", ab.HIGHLIGHTS_CLIP), kw.pop("clip", 1.0), kw.pop("n_clipped", None)
    piece = pe.mosaic_piece(w, h, ab.highlights_data(mode, clip), **kw)
    rng = np.random.default_rng(8)
    if piece.channels == 4:
        img = util.rgba_test_image(w, h, 6, lo=0.0, hi=0.8 if n is not None else 1.3)
        if n is not None:
            ys, xs = rng.choice(h * w, n, replace=False) // w, rng.choice(h * w, n, replace=False) % w
            img[ys[:n], xs[:n], rng.integers(0, 3, n)] = 1.5
    else:
        img = np.minimum(util.frame_natural(w, h, 6) * (0.7 if n is not None else 1.6), 3.0).astype(np.float32)
        if n is not None:
            img = np.minimum(img, 0.8)
            k = rng.choice(h * w, n, replace=False)
            img.reshape(-1)[k] = 1.25
    img.reshape(-1)[7] = np.nan
    return piece, img


@pytest.mark.parametrize("name", list(HIGHLIGHTS_CASES))
def test_highlights_oracle_equals_reference(name):
    piece, img = highlights_case(name)
    rc, got, n = pe.oracle_highlights(piece, img)
    assert rc == 0
    want = pe.ref_highlights(piece, img)
    assert same_bits(got, want).all()
    if "bypass" in name or "24" in name:
        assert n < 25 and same_bits(want, img).all()
    else:
        assert n >= 25 and not same_bits(want, img).all()


def test_highlights_oracle_refuses_reconstruction_modes():
    piece, img = highlights_case("clip_mosaic")
    for mode in (ab.HIGHLIGHTS_LAPLACIAN, ab.HIGHLIGHTS_HARMONIC):
        p = pe.mosaic_piece(134, 78, ab.highlights_data(mode, 1.0))
        assert pe.oracle_highlights(p, img)[0] == -1


EXPOSURE_CASES = {"rgba": dict(channels=4), "rgba_mask": dict(channels=4, mask_display=1), "mono": dict(channels=1)}


def exposure_case(name):
    kw = EXPOSURE_CASES[name]
    w, h = 131, 75
    piece = pe.mosaic_piece(w, h, ab.exposure_data(-0.00024, 0.7), filters=0, **kw)
    img = util.rgba_test_image(w, h, 4) if kw["channels"] == 4 else util.frame_natural(w, h, 4)
    return piece, img


@pytest.mark.parametrize("name", list(EXPOSURE_CASES))
def test_exposure_oracle_equals_reference(name):
    piece, img = exposure_case(name)
    assert same_bits(pe.oracle_exposure(piece, img), pe.ref_exposure(piece, img)).all()


def test_exposure_data_layout_is_the_reference_struct():
    import ctypes as C
    assert util.ref_size_t("ref_exposure_sizeof_data") == C.sizeof(ab.ExposureData)
    assert util.ref_size_t("ref_exposure_offsetof_black") == ab.ExposureData.black.offset
    assert util.ref_size_t("ref_rawprepare_sizeof_data") == C.sizeof(ab.RawprepareData)
    assert util.ref_size_t("ref_highlights_sizeof_data") == C.sizeof(ab.HighlightsData)


def test_float_to_integer_ends_oracle_equals_reference():
    img = pe.awkward_rgba(141, 67, 12)
    got, want = pe.oracle_gamma(img), pe.ref_gamma(img)
    assert (got == want).all() and (want[..., 3] == 0x5A).all()      # the fourth byte is never written
    for fmt in (ab.EXPORT_UINT8, ab.EXPORT_UINT8_SWAP, ab.EXPORT_UINT16):
        assert (pe.oracle_export(img, fmt) == pe.ref_export(img, fmt)).all()


FINALSCALE_CASES = {
    # name: (input w, h, input scale, output scale, interpolator); output size = round(input * out / in) as modify_roi_in implies
    "export_half_mitchell": (161, 97, 1.0, 0.5, ab.INTERPOLATION_MITCHELL),
    "export_third_bicubic": (173, 101, 1.0, 0.3333, ab.INTERPOLATION_BICUBIC),
    "export_0p77_bilinear": (150, 90, 1.0, 0.77, ab.INTERPOLATION_BILINEAR),
    "tiny_thumbnail_mitchell": (160, 120, 1.0, 0.06, ab.INTERPOLATION_MITCHELL),
    "darkroom_upscale_mitchell": (90, 60, 1.0, 1.7, ab.INTERPOLATION_MITCHELL),
    "darkroom_upscale_bicubic": (70, 50, 1.0, 2.0, ab.INTERPOLATION_BICUBIC),
    "upscale_bilinear": (64, 48, 1.0, 1.25, ab.INTERPOLATION_BILINEAR),
    "same_scale_is_a_copy": (80, 60, 0.5, 0.5, ab.INTERPOLATION_MITCHELL),
}


def finalscale_case(name):
    w, h, si, so, itor = FINALSCALE_CASES[name]
    img = util.rgba_test_image(w, h, 17, lo=-0.2, hi=1.5)
    img[3, 3, 1] = np.nan
    img[h // 2, w // 2, 0] = np.inf
    ow, oh = (w - 10, h - 7) if si == so else (int(round(w * so / si)), int(round(h * so / si)))
    return img, ow, oh, si, so, itor


@pytest.mark.parametrize("itor", [ab.INTERPOLATION_BILINEAR, ab.INTERPOLATION_BICUBIC, ab.INTERPOLATION_MITCHELL])
@pytest.mark.parametrize("scale", [0.5, 0.3333, 0.77, 0.06, 0.999, 1.001, 1.7, 2.0, 3.3])
def test_resampling_plan_oracle_equals_reference(itor, scale):
    """_prepare_resampling_plan cut verbatim: lengths, normalised taps (bit for bit) and clipped indexes of one axis"""
    n_in = 400
    for x0_in, x0_out in ((0, 0), (13, 7)):
        n_out = max(int(n_in * scale) - x0_out, 4)
        n, l, k, i = pe.oracle_plan(itor, n_in, x0_in, n_out, x0_out, scale)
        rn, rl, rk, ri = pe.ref_plan(itor, n_in, x0_in, n_out, x0_out, scale)
        assert n == rn and n > 0 and (l == rl).all() and (i == ri).all() and same_bits(k, rk).all()
    assert pe.oracle_plan(itor, n_in, 0, n_in, 0, 1.0)[0] == -1 == pe.ref_plan(itor, n_in, 0, n_in, 0, 1.0)[0]


@pytest.mark.parametrize("name", list(FINALSCALE_CASES))
def test_finalscale_oracle_equals_reference(name):
    args = finalscale_case(name)
    want = pe.ref_finalscale(*args)
    assert same_bits(pe.oracle_finalscale(*args), want).all()
    if "copy" not in name:       # resampled pixels are clipped at 0 and never non-finite; copied rows are what they were
        assert (want >= 0).all() and np.isfinite(want).all() and want.std() > 0


WORK = util.profile_pair(util.REC2020_TO_XYZ_D50)
MIX = [[1.1, -0.05, -0.05], [0.02, 0.95, 0.03], [-0.1, 0.0, 1.1]]
CHANNELMIXER_CASES = {
    # the module's default (CAT16, version 3, clip, gamut compression 1) and one case per branch of loop_switch
    "cat16_v3_default": dict(adaptation=ab.ADAPTATION_CAT16, illuminant=(0.93, 1.02, 0.71)),
    "cat16_v3_tuned": dict(adaptation=ab.ADAPTATION_CAT16, illuminant=(0.93, 1.02, 0.71), mix=MIX, saturation=(0.1, -0.2, 0.05), lightness=(0.05, 0.1, -0.1)),
    "bradford_full_v2_noclip": dict(adaptation=ab.ADAPTATION_FULL_BRADFORD, version=1, clip=0, illuminant=(1.05, 1.0, 0.6), mix=MIX, p=0.8, gamut=2.5),
    "bradford_linear_v1": dict(adaptation=ab.ADAPTATION_LINEAR_BRADFORD, version=0, illuminant=(1.05, 1.0, 0.6), saturation=(0.3, 0.1, -0.2)),
    "xyz_no_gamut": dict(adaptation=ab.ADAPTATION_XYZ, illuminant=(0.9, 1.0, 0.7), gamut=0.0, mix=MIX),
    "rgb_bypass_mix_only": dict(adaptation=ab.ADAPTATION_RGB, mix=MIX, clip=0, lightness=(0.2, 0.2, 0.2)),
    "grey_output": dict(adaptation=ab.ADAPTATION_CAT16, illuminant=(0.93, 1.02, 0.71), apply_grey=1, grey=(0.3, 0.5, 0.2)),
    "unhandled_adaptation_writes_nothing": dict(adaptation=5),
}


def channelmixer_case(name):
    img = util.hdr_rgba(131, 75, 3)
    img[3, 3, :3] = np.nan
    img[4, 4, 0] = np.inf
    img[5, 5, :3] = (-0.5, 0.2, 0.1)
    img[6, 6, :3] = 0.0
    img[7, 7, :3] = 1e-7
    return img, ab.channelmixer_piece(WORK, **CHANNELMIXER_CASES[name])


@pytest.mark.parametrize("name", list(CHANNELMIXER_CASES))
def test_channelmixerrgb_oracle_equals_reference(name):
    img, cp = channelmixer_case(name)
    want = pe.ref_channelmixerrgb(img, cp)
    assert same_bits(pe.oracle_channelmixerrgb(img, cp), want).all()
    assert same_bits(want[..., 3], img[..., 3]).all() != ("unhandled" in name)


def test_channelmixerrgb_oracle_every_branch_combination():
    img = channelmixer_case("cat16_v3_default")[0]
    for ad in range(5):
        for ver in range(3):
            for clip in (0, 1):
                cp = ab.channelmixer_piece(WORK, adaptation=ad, version=ver, clip=clip, illuminant=(0.93, 1.02, 0.71), mix=MIX, saturation=(0.1, -0.2, 0.05),
                                           lightness=(0.05, 0.1, -0.1), p=0.85, gamut=1.5)
                assert same_bits(pe.oracle_channelmixerrgb(img, cp), pe.ref_channelmixerrgb(img, cp)).all(), (ad, ver, clip)


def test_channelmixerrgb_data_layout_is_the_reference_struct():
    import ctypes as C
    P = ab.ChannelmixerPiece
    assert util.ref_size_t("ref_channelmixerrgb_sizeof_data") == P.work_in.offset == 192
    assert [util.ref_size_t("ref_channelmixerrgb_offsetof", i) for i in range(5)] == [P.saturation.offset, P.illuminant.offset, P.p.offset, P.adaptation.offset,
                                                                                      P.version.offset]


INITIALSCALE_CASES = {
    # name: (full image w, h; roi_in (x, y, w, h, scale); roi_out (x, y, w, h, scale); interpolator): what the darkroom asks of the module
    "zoomed_out_region": ((40, 30, 160, 110, 1.0), (12, 9, 48, 33, 0.3), ab.INTERPOLATION_MITCHELL),
    "half_size_bicubic": ((0, 0, 151, 97, 1.0), (0, 0, 75, 48, 0.5), ab.INTERPOLATION_BICUBIC),
    "crop_at_equal_scale": ((10, 20, 120, 90, 1.0), (25, 31, 60, 40, 1.0), ab.INTERPOLATION_MITCHELL),
    "upscaled_region_bilinear": ((30, 20, 60, 50, 1.0), (45, 30, 80, 60, 1.5), ab.INTERPOLATION_BILINEAR),
}


def initialscale_case(name):
    roi_in, roi_out, itor = INITIALSCALE_CASES[name]
    img = util.rgba_test_image(roi_in[2], roi_in[3], 19, lo=-0.2, hi=1.5)
    return img, roi_in, roi_out, itor


@pytest.mark.parametrize("name", list(INITIALSCALE_CASES))
def test_initialscale_oracle_equals_reference(name):
    args = initialscale_case(name)
    assert same_bits(pe.oracle_clip_and_zoom(*args), pe.ref_clip_and_zoom(*args)).all()


@pytest.mark.parametrize("orientation", range(8))
def test_flip_oracle_equals_reference(orientation):
    for img in (util.rgba_test_image(37, 23, 3), util.frame_natural(41, 19, 3)):
        want = pe.ref_flip(img, orientation)
        assert same_bits(pe.oracle_flip(img, orientation), want).all() and (want != -7.0).all()


def _golden():
    return np.load(os.path.join(util.GOLDEN_DIR, "pipe_ends.npz"))


def test_pipe_ends_oracle_equals_golden():
    """the same cases as above against the outputs the reference builds gave in the authoring container"""
    g = _golden()
    for name in RAWPREPARE_CASES:
        piece, src, _ = rawprepare_case(name)
        assert same_bits(pe.oracle_rawprepare(piece, src), g["rawprepare_" + name]).all()
    for name in TEMPERATURE_CASES:
        assert same_bits(pe.oracle_temperature(*temperature_case(name)), g["temperature_" + name]).all()
    for name in HIGHLIGHTS_CASES:
        assert same_bits(pe.oracle_highlights(*highlights_case(name))[1], g["highlights_" + name]).all()
    for name in EXPOSURE_CASES:
        assert same_bits(pe.oracle_exposure(*exposure_case(name)), g["exposure_" + name]).all()
    for name in FINALSCALE_CASES:
        assert same_bits(pe.oracle_finalscale(*finalscale_case(name)), g["finalscale_" + name]).all()
    for name in CHANNELMIXER_CASES:
        assert same_bits(pe.oracle_channelmixerrgb(*channelmixer_case(name)), g["channelmixerrgb_" + name]).all()
    for name in INITIALSCALE_CASES:
        assert same_bits(pe.oracle_clip_and_zoom(*initialscale_case(name)), g["initialscale_" + name]).all()
    for orientation in range(8):
        assert same_bits(pe.oracle_flip(util.rgba_test_image(37, 23, 3), orientation), g[f"flip_{orientation}"]).all()
    img = pe.awkward_rgba(141, 67, 12)
    assert (pe.oracle_gamma(img) == g["gamma"]).all()
    for fmt in (ab.EXPORT_UINT8, ab.EXPORT_UINT8_SWAP, ab.EXPORT_UINT16):
        assert (pe.oracle_export(img, fmt) == g[f"export_{fmt}"]).all()
