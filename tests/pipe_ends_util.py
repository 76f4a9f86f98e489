"""Helpers for the modules either side of the demosaic .. colorout path (rawprepare, temperature, highlights, exposure,
gamma, export conversions): calls into the oracle (oracle/restate/pipe_ends_oracle.c) and into the reference's own
lines compiled in place (oracle/_ref).  Checkers only."""
from __future__ import annotations

import ctypes as C

import numpy as np

import ansel_b200 as ab
import util

VP = C.c_void_p


def vp(a: np.ndarray):
    assert a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(VP)


def sensor_frame(w: int, h: int, seed: int, black: int = 512, white: int = 16383, clipped: int = 60, level: float = 0.9) -> np.ndarray:
    """uint16 RGGB sensor data: the natural test scene scaled into [black, white] with `clipped` blown samples"""
    m = util.frame_natural(w, h, seed)
    rng = np.random.default_rng(seed + 5)
    raw = np.clip(np.rint(m * (white - black) * level + black + rng.normal(0, 3, m.shape)), 0, 65535)
    if clipped:
        ys, xs = rng.integers(0, h, clipped), rng.integers(0, w, clipped)
        raw[ys, xs] = white + rng.integers(0, 40, clipped)
    return raw.astype(np.uint16)


def rawprepare_piece(in_w, in_h, d, *, out=None, datatype=ab.TYPE_UINT16, filters=util.BAYER["RGGB"], channels=1, scale=1.0,
                     buf=None, devid=-1):
    """roi_in = the whole (in_w x in_h) buffer; out = (x, y, w, h) of roi_out, default: the input minus the crop"""
    csx, csy = int(np.round(np.float32(d.x * scale))), int(np.round(np.float32(d.y * scale)))
    x, y, w, h = out if out else (0, 0, in_w - csx, in_h - csy)
    p = ab.make_piece(in_w, in_h, filters=filters, channels=channels, data=d, out_width=w, out_height=h, scale=scale, devid=devid)
    p.roi_out.x, p.roi_out.y = x, y
    p.datatype = datatype
    p.buf_in_width, p.buf_in_height = buf if buf else (in_w, in_h)
    return p


def oracle_rawprepare(piece, src: np.ndarray) -> np.ndarray:
    ch = piece.channels
    out = np.zeros((piece.roi_out.height, piece.roi_out.width) + ((ch,) if ch > 1 else ()), np.float32)
    f = util.oracle().orc_rawprepare
    f.restype = C.c_int
    assert f(C.byref(piece), vp(src), vp(out)) == 0
    return out


@util.recorded(lambda piece, src, gain=None, spacing=(0.0, 0.0), origin=(0.0, 0.0), kind="strict": oracle_rawprepare(piece, src))
def ref_rawprepare(piece, src: np.ndarray, gain=None, spacing=(0.0, 0.0), origin=(0.0, 0.0), kind="strict"):
    lib = util.ref(kind)
    if lib is None:
        return None
    d = C.cast(piece.data, C.POINTER(ab.RawprepareData)).contents
    ch = piece.channels
    out = util.aligned_empty((piece.roi_out.height, piece.roi_out.width) + ((ch,) if ch > 1 else ()))
    out[...] = 0
    g = None if gain is None else np.ascontiguousarray(gain, np.float32)
    mw, mh = (g.shape[2], g.shape[1]) if g is not None else (0, 0)
    f = lib.ref_rawprepare
    f.restype = C.c_int
    f.argtypes = [VP, VP] + [C.c_int] * 6 + [C.c_double, C.c_int, C.c_int, VP, VP, C.c_uint32, C.c_int, C.c_int, C.c_int, C.c_int, VP,
                             C.c_int, C.c_int] + [C.c_double] * 4
    assert f(vp(src), vp(out), piece.roi_in.width, piece.roi_in.height, piece.roi_out.x, piece.roi_out.y, piece.roi_out.width,
             piece.roi_out.height, piece.roi_in.scale, d.x, d.y, C.cast(d.sub, VP), C.cast(d.div, VP), piece.filters, ch, piece.datatype,
             piece.buf_in_width, piece.buf_in_height, None if g is None else vp(g), mw, mh, spacing[0], spacing[1], origin[0],
             origin[1]) == 0
    return np.array(out)


def mosaic_piece(w, h, data, *, filters=util.BAYER["RGGB"], x=0, y=0, channels=1, pm=(1.0, 1.0, 1.0, 1.0), mask_display=0,
                 xtrans=None, devid=-1):
    p = ab.make_piece(w, h, filters=filters, channels=channels, data=data, processed_maximum=pm, devid=devid)
    p.roi_in.x = p.roi_out.x = x
    p.roi_in.y = p.roi_out.y = y
    p.mask_display = mask_display
    p.datatype = ab.TYPE_FLOAT
    if xtrans is not None:
        for i in range(6):
            for j in range(6):
                p.xtrans[i][j] = int(xtrans[i][j])
    return p


XTRANS = np.array([[1, 1, 0, 1, 1, 2], [1, 1, 2, 1, 1, 0], [2, 0, 1, 0, 2, 1], [1, 1, 2, 1, 1, 0], [1, 1, 0, 1, 1, 2],
                   [0, 2, 1, 2, 0, 1]], np.uint8)


def oracle_temperature(piece, img: np.ndarray) -> np.ndarray:
    out = np.full_like(img, -7.0)
    f = util.oracle().orc_temperature
    f.restype = C.c_int
    assert f(C.byref(piece), vp(img), vp(out)) == 0
    return out


@util.recorded(lambda piece, img, kind="strict": oracle_temperature(piece, img))
def ref_temperature(piece, img: np.ndarray, kind="strict"):
    lib = util.ref(kind)
    if lib is None:
        return None
    d = C.cast(piece.data, C.POINTER(ab.TemperatureData)).contents
    src, out = util.aligned_empty(img.shape), util.aligned_empty(img.shape)
    src[...] = img
    out[...] = -7.0
    xt = np.ascontiguousarray(np.array([[piece.xtrans[i][j] for j in range(6)] for i in range(6)], np.uint8))
    f = lib.ref_temperature
    f.restype = C.c_int
    assert f(vp(src), vp(out), piece.roi_out.x, piece.roi_out.y, piece.roi_out.width, piece.roi_out.height, C.c_uint32(piece.filters),
             vp(xt), piece.channels, C.cast(d.coeffs, VP), piece.mask_display) == 0
    return np.array(out)


def oracle_highlights(piece, img: np.ndarray):
    """-> (rc, out, n_clipped)"""
    out = np.full_like(img, -7.0)
    n = C.c_size_t(0)
    f = util.oracle().orc_highlights
    f.restype = C.c_int
    rc = f(C.byref(piece), vp(img), vp(out), C.byref(n))
    return rc, out, n.value


@util.recorded(lambda piece, img, kind="strict": oracle_highlights(piece, img)[1])
def ref_highlights(piece, img: np.ndarray, kind="strict"):
    lib = util.ref(kind)
    if lib is None:
        return None
    d = C.cast(piece.data, C.POINTER(ab.HighlightsData)).contents
    src, out = util.aligned_empty(img.shape), util.aligned_empty(img.shape)
    src[...] = img
    out[...] = -7.0
    xt = np.ascontiguousarray(np.array([[piece.xtrans[i][j] for j in range(6)] for i in range(6)], np.uint8))
    lib.ref_highlights_set_xtrans(vp(xt))
    f = lib.ref_highlights
    f.restype = C.c_int
    pm = (C.c_float * 4)(*piece.processed_maximum)
    assert f(vp(src), vp(out), piece.roi_out.x, piece.roi_out.y, piece.roi_out.width, piece.roi_out.height, C.c_uint32(piece.filters),
             piece.channels, d.mode, C.c_float(d.clip), pm, piece.mask_display) == 0
    return np.array(out)


def oracle_exposure(piece, img: np.ndarray) -> np.ndarray:
    out = np.full_like(img, -7.0)
    f = util.oracle().orc_exposure
    f.restype = C.c_int
    assert f(C.byref(piece), vp(img), vp(out)) == 0
    return out


@util.recorded(lambda piece, img, kind="strict": oracle_exposure(piece, img))
def ref_exposure(piece, img: np.ndarray, kind="strict"):
    lib = util.ref(kind)
    if lib is None:
        return None
    d = C.cast(piece.data, C.POINTER(ab.ExposureData)).contents
    src, out = util.aligned_empty(img.shape), util.aligned_empty(img.shape)
    src[...] = img
    out[...] = -7.0
    f = lib.ref_exposure
    f.restype = C.c_int
    assert f(vp(src), vp(out), piece.roi_out.width, piece.roi_out.height, piece.channels, C.c_float(d.black), C.c_float(d.scale),
             piece.mask_display) == 0
    return np.array(out)


def oracle_gamma(img: np.ndarray, fill: int = 0x5A) -> np.ndarray:
    out = np.full(img.shape, fill, np.uint8)
    util.oracle().orc_gamma_copy_output(vp(img), vp(out), C.c_size_t(img.shape[0] * img.shape[1]))
    return out


@util.recorded(lambda img, fill=0x5A, kind="strict": oracle_gamma(img, fill))
def ref_gamma(img: np.ndarray, fill: int = 0x5A, kind="strict"):
    lib = util.ref(kind)
    if lib is None:
        return None
    src = util.aligned_empty(img.shape)
    src[...] = img
    out = util.aligned_empty(img.shape, np.uint8)
    out[...] = fill
    lib.ref_gamma_copy_output(vp(src), vp(out), C.c_size_t(img.shape[0] * img.shape[1]))
    return np.array(out)


EXPORT_DTYPE = {ab.EXPORT_UINT8: np.uint8, ab.EXPORT_UINT8_SWAP: np.uint8, ab.EXPORT_UINT16: np.uint16}
_REF_EXPORT = {ab.EXPORT_UINT8: "ref_clamp_float_to_uint8", ab.EXPORT_UINT8_SWAP: "ref_swap_byteorder_float_to_uint8",
               ab.EXPORT_UINT16: "ref_export_final_buffer_to_uint16"}


def oracle_export(img: np.ndarray, fmt: int) -> np.ndarray:
    out = np.zeros(img.shape, EXPORT_DTYPE[fmt])
    util.oracle().orc_export_convert(vp(img), vp(out), C.c_size_t(img.shape[0] * img.shape[1]), fmt)
    return out


@util.recorded(lambda img, fmt, kind="strict": oracle_export(img, fmt))
def ref_export(img: np.ndarray, fmt: int, kind="strict"):
    lib = util.ref(kind)
    if lib is None:
        return None
    src = util.aligned_empty(img.shape)
    src[...] = img
    out = np.zeros(img.shape, EXPORT_DTYPE[fmt])
    getattr(lib, _REF_EXPORT[fmt])(vp(src), vp(out), C.c_size_t(img.shape[1]), C.c_size_t(img.shape[0]))
    return out


def awkward_rgba(w: int, h: int, seed: int) -> np.ndarray:
    """RGBA floats with everything the float -> integer ends must survive: negatives, > 1, exact .5 steps, NaN, inf, denormals"""
    img = util.rgba_test_image(w, h, seed, lo=-0.3, hi=1.4)
    flat = img.reshape(-1)
    rng = np.random.default_rng(seed)
    k = rng.integers(0, flat.size, 400)
    flat[k[:50]] = np.nan
    flat[k[50:100]] = np.inf
    flat[k[100:150]] = -np.inf
    flat[k[150:200]] = 1e-41
    flat[k[200:300]] = (rng.integers(0, 256, 100) + 0.5) / np.float32(255.0)
    flat[k[300:400]] = (rng.integers(0, 65536, 100) + 0.5) / np.float32(65535.0)
    return img


# ---- finalscale ---------------------------------------------------------------------------------------------------------
def _plan(lib, fn, interpolator, n_in, in_x0, n_out, out_x0, scale):
    per = 160
    lengths, kernel, index = np.zeros(n_out, np.int32), np.zeros(per * n_out, np.float32), np.zeros(per * n_out, np.int32)
    f = getattr(lib, fn)
    f.restype = C.c_int
    f.argtypes = [C.c_int] * 5 + [C.c_float, VP, VP, VP, C.c_int]
    n = f(interpolator, n_in, in_x0, n_out, out_x0, scale, vp(lengths), vp(kernel), vp(index), per * n_out)
    return n, lengths, kernel[:max(n, 0)], index[:max(n, 0)]


def oracle_plan(*a):
    return _plan(util.oracle(), "orc_resampling_plan", *a)


@util.recorded(lambda *a, kind="strict": oracle_plan(*a))
def ref_plan(*a, kind="strict"):
    lib = util.ref(kind)
    return None if lib is None else _plan(lib, "ref_resampling_plan", *a)


def _finalscale(lib, fn, img, out_w, out_h, in_scale, out_scale, interpolator):
    h, w = img.shape[:2]
    src, out = util.aligned_empty(img.shape), util.aligned_empty((out_h, out_w, 4))
    src[...] = img
    out[...] = -7.0
    f = getattr(lib, fn)
    f.restype = C.c_int
    f.argtypes = [VP, VP, C.c_int, C.c_int, C.c_double, C.c_int, C.c_int, C.c_double, C.c_int]
    assert f(vp(src), vp(out), w, h, in_scale, out_w, out_h, out_scale, interpolator) == 0
    return np.array(out)


def oracle_finalscale(img, out_w, out_h, in_scale, out_scale, interpolator):
    return _finalscale(util.oracle(), "orc_finalscale", img, out_w, out_h, in_scale, out_scale, interpolator)


@util.recorded(lambda img, out_w, out_h, in_scale, out_scale, interpolator, kind="strict": oracle_finalscale(img, out_w, out_h, in_scale, out_scale, interpolator))
def ref_finalscale(img, out_w, out_h, in_scale, out_scale, interpolator, kind="strict"):
    lib = util.ref(kind)
    return None if lib is None else _finalscale(lib, "ref_finalscale", img, out_w, out_h, in_scale, out_scale, interpolator)


# ---- colour calibration (channelmixerrgb) -------------------------------------------------------------------------------
def oracle_channelmixerrgb(img, cp):
    h, w = img.shape[:2]
    out = np.full_like(img, -7.0)
    f = util.oracle().orc_channelmixerrgb
    f.restype = C.c_int
    assert f(vp(np.ascontiguousarray(img)), vp(out), w, h, C.byref(cp)) == 0
    return out


@util.recorded(lambda img, cp, kind="strict": oracle_channelmixerrgb(img, cp))
def ref_channelmixerrgb(img, cp, kind="strict"):
    lib = util.ref(kind)
    if lib is None:
        return None
    h, w = img.shape[:2]
    src, out = util.aligned_empty(img.shape), util.aligned_empty(img.shape)
    src[...] = img
    out[...] = -7.0
    f = lib.ref_channelmixerrgb
    f.restype = C.c_int
    assert f(vp(src), vp(out), w, h, C.byref(cp), C.byref(cp, ab.ChannelmixerPiece.work_in.offset), C.byref(cp, ab.ChannelmixerPiece.work_out.offset)) == 0
    return np.array(out)


# ---- initialscale (clip and zoom with ROI origins) and flip -----------------------------------------------------------------
def _clip_and_zoom(lib, fn, img, roi_in, roi_out, interpolator):
    """roi = (x, y, width, height, scale); img holds roi_in"""
    src, out = util.aligned_empty(img.shape), util.aligned_empty((roi_out[3], roi_out[2], 4))
    src[...] = img
    out[...] = -7.0
    f = getattr(lib, fn)
    f.restype = C.c_int
    f.argtypes = [VP, VP] + [C.c_int] * 4 + [C.c_double] + [C.c_int] * 4 + [C.c_double, C.c_int]
    assert f(vp(src), vp(out), *roi_in, *roi_out, interpolator) == 0
    return np.array(out)


def oracle_clip_and_zoom(img, roi_in, roi_out, interpolator):
    return _clip_and_zoom(util.oracle(), "orc_clip_and_zoom", img, roi_in, roi_out, interpolator)


@util.recorded(lambda img, roi_in, roi_out, interpolator, kind="strict": oracle_clip_and_zoom(img, roi_in, roi_out, interpolator))
def ref_clip_and_zoom(img, roi_in, roi_out, interpolator, kind="strict"):
    lib = util.ref(kind)
    return None if lib is None else _clip_and_zoom(lib, "ref_clip_and_zoom", img, roi_in, roi_out, interpolator)


def _flip(lib, fn, img, orientation, ch_arg):
    h, w = img.shape[:2]
    ch = img.shape[2] if img.ndim == 3 else 1
    src = util.aligned_empty(img.shape)
    src[...] = img
    out = util.aligned_empty((w, h) + img.shape[2:]) if orientation & 4 else util.aligned_empty(img.shape)
    out[...] = -7.0
    f = getattr(lib, fn)
    f.restype = C.c_int
    assert f(vp(src), vp(out), ch * 4 if ch_arg == "bpp" else ch, w, h, orientation) == 0
    return np.array(out)


def oracle_flip(img, orientation):
    return _flip(util.oracle(), "orc_flip", img, orientation, "bpp")


@util.recorded(lambda img, orientation, kind="strict": oracle_flip(img, orientation))
def ref_flip(img, orientation, kind="strict"):
    lib = util.ref(kind)
    return None if lib is None else _flip(lib, "ref_flip", img, orientation, "bpp")
