"""Helpers of the blending tests: the parameter block (same layout for the reference wrapper, the oracle and the product), cases."""
import ctypes as C

import numpy as np

import util

MASK_ENABLED, MASK_SHAPE, MASK_PARAMETRIC, MASK_RASTER = 1, 2, 4, 8
COMBINE_INV, COMBINE_INCL = 1, 2
CS_RAW, CS_LAB, CS_RGB_DISPLAY, CS_RGB_SCENE = 1, 2, 3, 4
REVERSE = 0x80000000
MODES = {"normal": 0x18, "multiply": 0x04, "average": 0x05, "add": 0x06, "subtract": 0x07, "subtract_inverse": 0x25, "difference": 0x17,
         "divide": 0x26, "divide_inverse": 0x27, "geometric_mean": 0x28, "harmonic_mean": 0x29, "luminance": 0x10, "chromaticity": 0x11,
         "rgb_r": 0x21, "rgb_g": 0x22, "rgb_b": 0x23}
# the operators of the Lab space (develop/blends/blendif_lab.c _choose_blend_func :1070-1162)
LAB_MODES = {"normal": 0x18, "bounded": 0x19, "lighten": 0x02, "darken": 0x03, "multiply": 0x04, "average": 0x05, "add": 0x06, "subtract": 0x07,
             "difference_old": 0x08, "difference": 0x17, "screen": 0x09, "overlay": 0x0A, "softlight": 0x0B, "hardlight": 0x0C, "vividlight": 0x0D,
             "linearlight": 0x0E, "pinlight": 0x0F, "lightness": 0x10, "chromaticity": 0x11, "hue": 0x12, "color": 0x13, "coloradjust": 0x16,
             "lab_lightness": 0x1A, "lab_l": 0x1E, "lab_a": 0x1F, "lab_b": 0x20, "lab_color": 0x1B}
# the operators of the display-referred RGB space (develop/blends/blendif_rgb_hsl.c _choose_blend_func :915-1007)
DISPLAY_MODES = {"normal": 0x18, "bounded": 0x19, "lighten": 0x02, "darken": 0x03, "multiply": 0x04, "average": 0x05, "add": 0x06, "subtract": 0x07,
                 "difference": 0x17, "screen": 0x09, "overlay": 0x0A, "softlight": 0x0B, "hardlight": 0x0C, "vividlight": 0x0D, "linearlight": 0x0E,
                 "pinlight": 0x0F, "lightness": 0x10, "chromaticity": 0x11, "hue": 0x12, "color": 0x13, "coloradjust": 0x16, "hsv_value": 0x1C,
                 "hsv_color": 0x1D, "rgb_r": 0x21, "rgb_g": 0x22, "rgb_b": 0x23}
# the operators of the raw space (develop/blends/blendif_raw.c _choose_blend_func :290-352); any other mode is the unbounded normal blend there
RAW_MODES = {k: v for k, v in DISPLAY_MODES.items() if v <= 0x0F or v in (0x17, 0x18, 0x19)}
RAW_MODES["lightness_is_normal_here"] = 0x10
LAB_LCH_MODES = ("chromaticity", "hue", "color", "coloradjust")      # through atan2f / hypotf / cosf / sinf (ansel_b200/csrc/flt32_math.cuh)
# linear Rec2020 -> XYZ (D50), the work profile's matrix_in, row by row; its middle row is what the gray channel of the parametric mask weighs with
MATRIX_IN = (0.6734241, 0.1656411, 0.1251286, 0.2790177, 0.6753402, 0.0456377, -0.0019300, 0.0299784, 0.7973330)
LUMINANCE = MATRIX_IN[3:6]


class BlendParams(C.Structure):
    _fields_ = [("mask_mode", C.c_uint32), ("blend_cst", C.c_int32), ("blend_mode", C.c_uint32), ("blend_parameter", C.c_float), ("opacity", C.c_float),
                ("mask_combine", C.c_uint32), ("blendif", C.c_uint32), ("feathering_radius", C.c_float), ("feathering_guide", C.c_uint32),
                ("blur_radius", C.c_float), ("contrast", C.c_float), ("brightness", C.c_float), ("details", C.c_float),
                ("blendif_parameters", C.c_float * 64), ("blendif_boost_factors", C.c_float * 16), ("raster_used", C.c_int32), ("drawn_used", C.c_int32),
                ("luminance", C.c_float * 3), ("profile_nonlinear", C.c_int32), ("mask_display", C.c_uint32), ("matrix_in", C.c_float * 9)]


def params(mode="normal", opacity=65.0, mask_mode=MASK_ENABLED, reverse=False, blend_parameter=0.0, combine=0, blendif=0, channels=None, boosts=None,
           contrast=0.0, brightness=0.0, raster=0, drawn=0, mask_display=0, **extra):
    """channels: {bit: (p0, p1, p2, p3)} of the parametric mask (bits 0..3 gray/R/G/B of the input, 4..7 of the output; bit + 16 in `blendif`
    inverts a channel)"""
    p = BlendParams()
    cst = extra.pop("cst", CS_RGB_SCENE)
    p.mask_mode, p.blend_cst = mask_mode, cst
    p.blend_mode = {CS_LAB: LAB_MODES, CS_RGB_DISPLAY: DISPLAY_MODES, CS_RAW: RAW_MODES}.get(cst, MODES)[mode] | (REVERSE if reverse else 0)
    p.blend_parameter, p.opacity, p.mask_combine, p.blendif = blend_parameter, opacity, combine, blendif
    p.contrast, p.brightness = contrast, brightness
    for i in range(16):
        p.blendif_parameters[4 * i:4 * i + 4] = (0.0, 0.0, 1.0, 1.0)
    for bit, v in (channels or {}).items():
        p.blendif_parameters[4 * bit:4 * bit + 4] = v
        p.blendif |= 1 << bit
    for bit, v in (boosts or {}).items():
        p.blendif_boost_factors[bit] = v
    p.raster_used, p.drawn_used, p.mask_display = raster, drawn, mask_display
    p.luminance[:] = LUMINANCE
    p.matrix_in[:] = MATRIX_IN
    for k, v in extra.items():
        setattr(p, k, v)
    return p


def frames(w=160, h=120, seed=1, xoffs=0, yoffs=0, iw=None, ih=None):
    """a module's input (scene-referred, some values beyond 1, a few non-positive) and output, and a smooth form mask"""
    rng = np.random.default_rng(seed)
    iw, ih = iw or w + xoffs, ih or h + yoffs
    a = (util.rgba_scene(iw, ih, seed, noise=0.02) * 1.8).astype(np.float32)
    a[..., 3] = rng.random((ih, iw), dtype=np.float32)
    a[3, 5, :3] = 0.0
    a[7, 2, 1] = -0.01
    b = (a[yoffs:yoffs + h, xoffs:xoffs + w] * rng.uniform(0.6, 1.5, (h, w, 1)) + rng.normal(0, 0.03, (h, w, 4))).astype(np.float32)
    b[11, 4, :3] = 0.0
    yy, xx = np.mgrid[0:h, 0:w]
    form = np.clip(1.2 - np.hypot(yy - h * 0.4, xx - w * 0.55) / (0.5 * w), 0.0, 1.0).astype(np.float32)
    return np.ascontiguousarray(a), np.ascontiguousarray(b), np.ascontiguousarray(form)


def frames_lab(w=160, h=120, seed=1, xoffs=0, yoffs=0):
    """the same for a Lab module: L in 0 .. 100 and a little beyond, a and b within +-90"""
    a, b, form = frames(w, h, seed, xoffs, yoffs)
    rng = np.random.default_rng(seed + 100)

    def to_lab(x, shape):
        lab = np.empty_like(x)
        lab[..., 0] = x[..., 1] * np.float32(62.0) - np.float32(3.0)
        lab[..., 1] = (x[..., 0] - x[..., 1]) * np.float32(140.0) + rng.normal(0, 6, shape).astype(np.float32)
        lab[..., 2] = (x[..., 1] - x[..., 2]) * np.float32(140.0) + rng.normal(0, 6, shape).astype(np.float32)
        lab[..., 3] = x[..., 3]
        return np.ascontiguousarray(lab)

    a, b = to_lab(a, a.shape[:2]), to_lab(b, b.shape[:2])
    a[3, 5, 1:3] = 0.0                  # a grey pixel: atan2f(0, 0)
    b[11, 4, 1:3] = (0.0, -4.0)
    return a, b, form


def _run(lib, fn, a, b, p, form=None, xoffs=0, yoffs=0, want_mask=True):
    ih, iw = a.shape[:2]
    oh, ow = b.shape[:2]
    out = util.aligned_empty(b.shape)
    out[...] = b
    src = util.aligned_empty(a.shape)
    src[...] = a
    mask = util.aligned_empty((oh, ow)) if want_mask else None
    if mask is not None:
        mask[...] = -3.0
    f = getattr(lib, fn)
    f.restype = C.c_int
    f.argtypes = [C.c_void_p, C.c_void_p] + [C.c_int] * 6 + [C.POINTER(BlendParams), C.c_void_p, C.c_void_p]
    fm = None
    if form is not None:
        fm = util.aligned_empty(form.shape)
        fm[...] = form
    rc = f(src.ctypes.data, out.ctypes.data, iw, ih, ow, oh, xoffs, yoffs, C.byref(p), None if fm is None else fm.ctypes.data,
           None if mask is None else mask.ctypes.data)
    return rc, np.array(out), (None if mask is None else np.array(mask))


def oracle(a, b, p, form=None, xoffs=0, yoffs=0):
    return _run(util.oracle(), "orc_blend_process", a, b, p, form, xoffs, yoffs)


@util.recorded(lambda a, b, p, form=None, xoffs=0, yoffs=0, kind="strict": oracle(a, b, p, form, xoffs, yoffs))
def ref(a, b, p, form=None, xoffs=0, yoffs=0, kind="strict"):
    lib = util.ref(kind)
    fn = {CS_LAB: "ref_blend_lab_process", CS_RGB_DISPLAY: "ref_blend_rgb_hsl_process", CS_RAW: "ref_blend_raw_process"}.get(p.blend_cst, "ref_blend_process")
    return None if lib is None else _run(lib, fn, a, b, p, form, xoffs, yoffs)


# the configurations every layer is checked on: (name, params kwargs, uses the form mask)
CONFIGS = [(m, dict(mode=m), False) for m in MODES] + [
    ("normal_reverse", dict(mode="normal", reverse=True, opacity=40.0), False),
    ("multiply_param", dict(mode="multiply", blend_parameter=1.5), False),
    ("divide_reverse", dict(mode="divide", reverse=True, blend_parameter=-0.5), False),
    ("opacity_0", dict(opacity=0.0), False),
    ("opacity_over", dict(opacity=130.0), False),
    ("raster_only", dict(mask_mode=MASK_ENABLED | MASK_RASTER, raster=1), True),
    ("drawn_only", dict(mask_mode=MASK_ENABLED | MASK_SHAPE, drawn=1), True),
    ("drawn_inverted", dict(mask_mode=MASK_ENABLED | MASK_SHAPE, drawn=1, combine=COMBINE_INV), True),
    ("parametric_gray_in", dict(mask_mode=MASK_ENABLED | MASK_PARAMETRIC, channels={0: (0.1, 0.3, 0.7, 0.9)}), False),
    ("parametric_rgb_out", dict(mask_mode=MASK_ENABLED | MASK_PARAMETRIC, channels={5: (0.0, 0.0, 0.5, 0.8), 6: (0.2, 0.4, 1.0, 1.0), 3: (0.05, 0.2, 0.6, 0.7)}), False),
    ("parametric_inverted_channel", dict(mask_mode=MASK_ENABLED | MASK_PARAMETRIC, channels={1: (0.2, 0.5, 0.8, 0.95)}, blendif=1 << 17), False),
    ("parametric_inclusive", dict(mask_mode=MASK_ENABLED | MASK_PARAMETRIC, combine=COMBINE_INCL, channels={0: (0.1, 0.3, 0.7, 0.9), 7: (0.0, 0.1, 0.4, 0.6)}), False),
    ("parametric_inclusive_inverted", dict(mask_mode=MASK_ENABLED | MASK_PARAMETRIC, combine=COMBINE_INCL | COMBINE_INV, channels={2: (0.1, 0.3, 0.7, 0.9)}), False),
    ("parametric_boost", dict(mask_mode=MASK_ENABLED | MASK_PARAMETRIC, channels={0: (0.1, 0.3, 0.7, 0.9)}, boosts={0: 1.5}), False),
    ("parametric_canceling", dict(mask_mode=MASK_ENABLED | MASK_PARAMETRIC, channels={1: (0.2, 0.5, 0.8, 0.95)}, blendif=(1 << 18)), False),
    ("drawn_and_parametric", dict(mask_mode=MASK_ENABLED | MASK_SHAPE | MASK_PARAMETRIC, drawn=1, channels={0: (0.1, 0.3, 0.7, 0.9)}), True),
    ("drawn_and_parametric_inv", dict(mask_mode=MASK_ENABLED | MASK_SHAPE | MASK_PARAMETRIC, drawn=1, combine=COMBINE_INV, channels={4: (0.1, 0.3, 0.7, 0.9)}), True),
    ("raster_and_parametric_incl", dict(mask_mode=MASK_ENABLED | MASK_RASTER | MASK_PARAMETRIC, raster=1, combine=COMBINE_INCL, channels={0: (0.1, 0.3, 0.7, 0.9)}), True),
    ("tone_curve", dict(mask_mode=MASK_ENABLED | MASK_SHAPE, drawn=1, contrast=0.4, brightness=0.2), True),
    ("tone_curve_dark", dict(mask_mode=MASK_ENABLED | MASK_SHAPE, drawn=1, contrast=-0.3, brightness=-0.35), True),
    ("tone_curve_extremes", dict(mask_mode=MASK_ENABLED | MASK_SHAPE, drawn=1, contrast=0.1, brightness=1.0), True),
    ("tone_curve_extremes2", dict(mask_mode=MASK_ENABLED | MASK_SHAPE, drawn=1, contrast=0.1, brightness=-1.0), True),
    ("mask_display", dict(mode="add", mask_display=1), False),
    ("disabled", dict(mask_mode=0), False),
    # the Jz / Cz / hz channels (bits 8..10 of the input, 12..14 of the output): XYZ D65 through the masking profile, the PQ curve, atan2f / hypotf
    ("parametric_jz_in", dict(mask_mode=MASK_ENABLED | MASK_PARAMETRIC, channels={8: (0.002, 0.006, 0.015, 0.02)}), False),
    ("parametric_cz_hz_out", dict(mask_mode=MASK_ENABLED | MASK_PARAMETRIC, channels={13: (0.0, 0.0, 0.004, 0.008), 14: (0.1, 0.2, 0.7, 0.85)}), False),
    ("parametric_jz_inverted_and_gray", dict(mask_mode=MASK_ENABLED | MASK_PARAMETRIC, channels={8: (0.001, 0.004, 0.012, 0.018), 0: (0.05, 0.2, 0.8, 1.0)}, blendif=1 << 24), False),
    ("drawn_and_parametric_hz_boost", dict(mask_mode=MASK_ENABLED | MASK_SHAPE | MASK_PARAMETRIC, drawn=1, channels={10: (0.2, 0.3, 0.6, 0.7), 12: (0.002, 0.006, 1.0, 1.0)},
                                           boosts={12: 1.0}), True),
]

# Lab: every operator, then the mask sources and combinations on the Lab channels (bits 0..2 L/a/b and 8..9 C/h of the input, 4..6 and 12..13 of the output)
_PAR = MASK_ENABLED | MASK_PARAMETRIC
LAB_CONFIGS = [("lab_" + m, dict(cst=CS_LAB, mode=m), False) for m in LAB_MODES] + [
    ("lab_overlay_reverse", dict(cst=CS_LAB, mode="overlay", reverse=True, opacity=40.0), False),
    ("lab_multiply_drawn", dict(cst=CS_LAB, mode="multiply", mask_mode=MASK_ENABLED | MASK_SHAPE, drawn=1), True),
    ("lab_vividlight_raster", dict(cst=CS_LAB, mode="vividlight", mask_mode=MASK_ENABLED | MASK_RASTER, raster=1, opacity=90.0), True),
    ("lab_parametric_L_in", dict(cst=CS_LAB, mask_mode=_PAR, channels={0: (0.1, 0.3, 0.6, 0.8)}), False),
    ("lab_parametric_ab_out", dict(cst=CS_LAB, mask_mode=_PAR, channels={5: (0.3, 0.45, 0.6, 0.7), 6: (0.2, 0.4, 1.0, 1.0), 2: (0.0, 0.0, 0.55, 0.65)}), False),
    ("lab_parametric_inverted_a", dict(cst=CS_LAB, mask_mode=_PAR, channels={1: (0.35, 0.45, 0.55, 0.7)}, blendif=1 << 17), False),
    ("lab_parametric_inclusive", dict(cst=CS_LAB, mask_mode=_PAR, combine=COMBINE_INCL, channels={0: (0.1, 0.3, 0.7, 0.9), 6: (0.4, 0.5, 0.6, 0.8)}), False),
    ("lab_parametric_boost_L", dict(cst=CS_LAB, mask_mode=_PAR, channels={4: (0.1, 0.3, 0.7, 0.9)}, boosts={4: -0.5}), False),
    ("lab_parametric_canceling", dict(cst=CS_LAB, mask_mode=_PAR, channels={2: (0.4, 0.5, 0.8, 0.95)}, blendif=(1 << 16)), False),
    ("lab_parametric_chroma_hue_in", dict(cst=CS_LAB, mask_mode=_PAR, channels={8: (0.05, 0.15, 0.5, 0.7), 9: (0.1, 0.2, 0.6, 0.75)}), False),
    ("lab_parametric_hue_out_inverted", dict(cst=CS_LAB, mask_mode=_PAR, channels={13: (0.3, 0.4, 0.7, 0.8), 0: (0.0, 0.0, 0.7, 0.9)}, blendif=1 << 29), False),
    ("lab_drawn_and_parametric", dict(cst=CS_LAB, mode="softlight", mask_mode=MASK_ENABLED | MASK_SHAPE | MASK_PARAMETRIC, drawn=1, channels={0: (0.1, 0.3, 0.7, 0.9)}), True),
    ("lab_tone_curve", dict(cst=CS_LAB, mask_mode=MASK_ENABLED | MASK_SHAPE, drawn=1, contrast=0.4, brightness=0.2), True),
    ("lab_mask_display", dict(cst=CS_LAB, mode="add", mask_display=1), False),
]


# display-referred RGB: every operator, then the mask sources and combinations on its channels (bits 0..3 gray/R/G/B and 8..10 H/S/L of the input,
# 4..7 and 12..14 of the output)
_D = dict(cst=CS_RGB_DISPLAY)
DISPLAY_CONFIGS = [("display_" + m, dict(_D, mode=m), False) for m in DISPLAY_MODES] + [
    ("display_overlay_reverse", dict(_D, mode="overlay", reverse=True, opacity=40.0), False),
    ("display_hsv_color_drawn", dict(_D, mode="hsv_color", mask_mode=MASK_ENABLED | MASK_SHAPE, drawn=1), True),
    ("display_vividlight_raster", dict(_D, mode="vividlight", mask_mode=MASK_ENABLED | MASK_RASTER, raster=1, opacity=90.0), True),
    ("display_parametric_gray_in", dict(_D, mask_mode=_PAR, channels={0: (0.1, 0.3, 0.6, 0.8)}), False),
    ("display_parametric_rgb_out", dict(_D, mask_mode=_PAR, channels={5: (0.0, 0.0, 0.5, 0.8), 6: (0.2, 0.4, 1.0, 1.0), 3: (0.05, 0.2, 0.6, 0.7)}), False),
    ("display_parametric_hsl_in", dict(_D, mask_mode=_PAR, channels={8: (0.05, 0.15, 0.5, 0.7), 9: (0.1, 0.2, 0.8, 0.95), 10: (0.1, 0.3, 0.7, 0.9)}), False),
    ("display_parametric_hue_out_inverted", dict(_D, mask_mode=_PAR, channels={12: (0.3, 0.4, 0.7, 0.8), 0: (0.0, 0.0, 0.7, 0.9)}, blendif=1 << 28), False),
    ("display_parametric_inclusive", dict(_D, mask_mode=_PAR, combine=COMBINE_INCL, channels={0: (0.1, 0.3, 0.7, 0.9), 13: (0.1, 0.2, 0.6, 0.8)}), False),
    ("display_drawn_and_parametric", dict(_D, mode="softlight", mask_mode=MASK_ENABLED | MASK_SHAPE | MASK_PARAMETRIC, drawn=1, channels={10: (0.1, 0.3, 0.7, 0.9)}), True),
    ("display_tone_curve", dict(_D, mask_mode=MASK_ENABLED | MASK_SHAPE, drawn=1, contrast=0.4, brightness=0.2), True),
    ("display_mask_display", dict(_D, mode="add", mask_display=1), False),
]


def frames_display(w=160, h=120, seed=1, xoffs=0, yoffs=0):
    """the same for a display-referred module: most values in 0 .. 1, some beyond on either side, a grey and a black pixel"""
    a, b, form = frames(w, h, seed, xoffs, yoffs)
    a[..., :3] = a[..., :3] * np.float32(0.62) - np.float32(0.03)
    b[..., :3] = b[..., :3] * np.float32(0.62) - np.float32(0.03)
    a[4, 6, :3] = 0.4
    b[4, 6, :3] = (0.2, 0.2, 0.7)
    a[9, 9, :3] = 0.0
    return a, b, form


# raw: every operator, then the mask sources; the parametric mask has no channels here, a block that asks for one only takes the seeded path
_R = dict(cst=CS_RAW)
RAW_CONFIGS = [("raw_" + m, dict(_R, mode=m), False) for m in RAW_MODES] + [
    ("raw_overlay_reverse", dict(_R, mode="overlay", reverse=True, opacity=40.0), False),
    ("raw_multiply_drawn_inverted", dict(_R, mode="multiply", mask_mode=MASK_ENABLED | MASK_SHAPE, drawn=1, combine=COMBINE_INV), True),
    ("raw_vividlight_raster", dict(_R, mode="vividlight", mask_mode=MASK_ENABLED | MASK_RASTER, raster=1, opacity=90.0), True),
    ("raw_parametric_asked_for", dict(_R, mask_mode=_PAR, channels={0: (0.1, 0.3, 0.6, 0.8)}, combine=COMBINE_INCL), False),
    ("raw_drawn_tone_curve", dict(_R, mode="softlight", mask_mode=MASK_ENABLED | MASK_SHAPE, drawn=1, contrast=0.4, brightness=0.2), True),
]


def frames_raw(w=160, h=120, seed=1, xoffs=0, yoffs=0):
    """a mosaic-like pair: one float per site, most values in 0 .. 1, some beyond on either side"""
    a, b, form = frames_display(w, h, seed, xoffs, yoffs)
    return np.ascontiguousarray(a[..., 1]), np.ascontiguousarray(b[..., 1]), form


def golden_configs():
    """the configurations of tests/golden/blend.npz: every third one of each space, and everything that goes through powf / atan2f / hypotf"""
    rgb = [c for k, c in enumerate(CONFIGS) if c[0] != "disabled" and (k % 3 == 0 or any(ch >= 8 for ch in c[1].get("channels", {})))]
    lab = [c for k, c in enumerate(LAB_CONFIGS) if k % 3 == 0 or c[1].get("mode") in LAB_LCH_MODES or any(ch >= 8 for ch in c[1].get("channels", {}))]
    display = [c for k, c in enumerate(DISPLAY_CONFIGS) if k % 3 == 0 or c[1].get("mode") in ("hsv_color", "hue", "color") or any(ch >= 8 for ch in c[1].get("channels", {}))]
    return rgb + lab + display + RAW_CONFIGS[::3]


def frames_of(cst):
    return {CS_LAB: frames_lab, CS_RGB_DISPLAY: frames_display, CS_RAW: frames_raw}.get(cst, frames)


def golden_frames(kw):
    return frames_of(kw.get("cst"))(96, 64, 7)


def lab_on_device(cfg):
    """what the library builds of a Lab configuration: all of it since the LCh operators and the C / h channels went in"""
    return True


_EMUL = None


def emul(a, b, p, form=None, xoffs=0, yoffs=0):
    """ansel_b200/csrc/blend.cu compiled with g++ (tests/emul/emul_blend.cpp): the host-side plan and the kernel, thread by thread"""
    global _EMUL
    if _EMUL is None:
        import os
        import subprocess
        here = os.path.join(os.path.dirname(os.path.abspath(__file__)), "emul")
        so = os.path.join(here, "libemul_blend.so")
        srcs = [os.path.join(here, "emul_blend.cpp"), os.path.join(here, "cuda_on_cpu.h"), os.path.join(here, "..", "..", "ansel_b200", "csrc", "blend.cu"),
                os.path.join(here, "..", "..", "include", "b200iop.h")]
        if not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in srcs):
            subprocess.run(["g++", "-O1", "-std=c++17", "-fno-fast-math", "-ffp-contract=off", "-I", here, "-shared", "-fPIC", "-o", so, srcs[0]], check=True)
        _EMUL = C.CDLL(so)
    return _run(_EMUL, "emul_blend_process", a, b, p, form, xoffs, yoffs)
