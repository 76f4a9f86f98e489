"""Helpers of the highlights "guided laplacians" tests (iop/highlights/laplacian.c)."""
import ctypes as C
import os
import numpy as np
import util

F4 = C.c_float * 4
XTRANS = [1, 1, 0, 1, 1, 2, 1, 1, 2, 1, 1, 0, 2, 0, 1, 0, 2, 1, 1, 1, 2, 1, 1, 0, 1, 1, 0, 1, 1, 2, 0, 2, 1, 2, 0, 1]   # a Fuji sensor's table, row by row
# name -> (width, height, filters, keywords): the frames of tests/golden/hl_laplacian.npz (inputs are regenerated from the name's length)
GOLDEN = {
    "bayer_noise": (240, 176, util.BAYER["RGGB"], dict(iterations=3, noise_level=0.2)),
    "bayer_roi": (200, 150, util.BAYER["GBRG"], dict(roi_scale=0.5, x=13, y=7, scales=7)),
    "rgba": (160, 120, 0, dict(iterations=2, noise_level=0.1, solid_color=0.2)),
    "xtrans_roi": (210, 150, 9, dict(xtrans=XTRANS, x=4, y=3, noise_level=0.1)),
}


def clips_of(clip=1.0, pmax=(1.0, 1.0, 1.0)):
    """process() :764-766"""
    f = np.float32
    m = min(pmax)
    return np.array([f(0.995) * f(clip) * f(pmax[0]), f(0.995) * f(clip) * f(pmax[1]), f(0.995) * f(clip) * f(pmax[2]),
                     f(clip) * f(m)], np.float32)


def clipped_mosaic(w, h, seed, filters=util.BAYER["RGGB"], blobs=6, level=1.0):
    """a natural mosaic with a few blown areas: soft blobs pushed past the clip level and cut there, as a sensor does"""
    rng = np.random.default_rng(seed)
    m = util.frame_natural(w, h, seed).astype(np.float32) * np.float32(0.6)
    yy, xx = np.mgrid[0:h, 0:w].astype(np.float32)
    for _ in range(blobs):
        cx, cy = rng.uniform(0, w), rng.uniform(0, h)
        r = rng.uniform(0.04, 0.16) * min(w, h)
        m += np.float32(rng.uniform(0.6, 1.6)) * np.exp(-((xx - cx) ** 2 + (yy - cy) ** 2) / np.float32(2 * r * r)).astype(np.float32)
    return np.minimum(m, np.float32(level)).astype(np.float32)


def clipped_rgba(w, h, seed, level=1.0):
    rng = np.random.default_rng(seed)
    img = util.rgba_scene(w, h, seed).astype(np.float32) * np.float32(0.5)
    yy, xx = np.mgrid[0:h, 0:w].astype(np.float32)
    for _ in range(5):
        cx, cy = rng.uniform(0, w), rng.uniform(0, h)
        r = rng.uniform(0.05, 0.15) * min(w, h)
        g = np.exp(-((xx - cx) ** 2 + (yy - cy) ** 2) / np.float32(2 * r * r)).astype(np.float32)
        img[..., :3] += (np.float32(1.2) * g)[..., None] * rng.uniform(0.7, 1.3, 3).astype(np.float32)
    img[..., :3] = np.minimum(img[..., :3], np.float32(level))
    return np.ascontiguousarray(img)


def _call(f, img, filters, clips, iterations, scales, noise_level, solid_color, iscale, roi_scale, norm, force, x, y, xtrans):
    h, w = img.shape[:2]
    out = np.full_like(img, -7.0)
    nv = F4(*(norm if norm is not None else (0, 0, 0, 0)))
    xt = (C.c_uint8 * 36)(*xtrans) if xtrans is not None else None
    f.restype = C.c_int
    util.oracle().orc_fp_fast_mode_all()   # FTZ|DAZ on every thread, as the reference's pipe threads have it (darktable.c:877)
    rc = f(util.fptr(img), util.fptr(out), x, y, w, h, C.c_uint32(filters), xt, F4(*clips), iterations, scales, C.c_float(noise_level),
           C.c_float(solid_color), C.c_float(iscale), C.c_float(roi_scale), nv, int(force))
    assert rc == 0
    return out, np.array(list(nv), np.float32)


@util.recorded(lambda img, filters, clips, *, iterations=2, scales=6, noise_level=0.0, solid_color=0.0, iscale=1.0, roi_scale=1.0, norm=None, x=0, y=0,
               xtrans=None, lib=None, threads=None: oracle(img, filters, clips, iterations=iterations, scales=scales, noise_level=noise_level,
                                                           solid_color=solid_color, iscale=iscale, roi_scale=roi_scale, norm=norm, x=x, y=y, xtrans=xtrans))
def ref(img, filters, clips, *, iterations=2, scales=6, noise_level=0.0, solid_color=0.0, iscale=1.0, roi_scale=1.0, norm=None, x=0, y=0,
        xtrans=None, lib=None, threads=None):
    """the reference's process_laplacian(); returns (output, the normalization vector the run used); threads: OpenMP threads"""
    lib = lib or util.ref("strict")
    if threads:
        C.CDLL("libgomp.so.1").omp_set_num_threads(threads)
    return _call(lib.ref_hl_laplacian, img, filters, clips, iterations, scales, noise_level, solid_color, iscale, roi_scale, norm,
                 norm is not None, x, y, xtrans)


def oracle(img, filters, clips, *, iterations=2, scales=6, noise_level=0.0, solid_color=0.0, iscale=1.0, roi_scale=1.0, norm=None, x=0, y=0,
           xtrans=None):
    """oracle/restate/highlights_laplacian_oracle.c; norm None: the serial float sum of one thread"""
    return _call(util.oracle().orc_hl_laplacian, img, filters, clips, iterations, scales, noise_level, solid_color, iscale, roi_scale, norm,
                 norm is not None, x, y, xtrans)


_EMUL = None


def emul(img, filters, clips, norm, *, iterations=2, scales=6, noise_level=0.0, solid_color=0.0, iscale=1.0, roi_scale=1.0, x=0, y=0, xtrans=None):
    """ansel_b200/csrc/highlights_laplacian.cu compiled with g++ (tests/emul/emul_hl_laplacian.cpp): the launch sequence with every kernel
    thread by thread; the normalization vector is an input"""
    global _EMUL
    if _EMUL is None:
        import subprocess
        here = os.path.join(os.path.dirname(os.path.abspath(__file__)), "emul")
        csrc = os.path.join(here, "..", "..", "ansel_b200", "csrc")
        so = os.path.join(here, "libemul_hl_laplacian.so")
        srcs = [os.path.join(here, "emul_hl_laplacian.cpp"), os.path.join(here, "cuda_on_cpu.h"), os.path.join(csrc, "highlights_laplacian.cu"),
                os.path.join(csrc, "bspline.cuh"), os.path.join(csrc, "flt32_math.cuh"), os.path.join(here, "..", "..", "include", "b200iop.h")]
        if not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in srcs):
            subprocess.run(["g++", "-O1", "-std=c++17", "-fno-fast-math", "-ffp-contract=off", "-I", here, "-shared", "-fPIC", "-o", so, srcs[0]], check=True)
        _EMUL = C.CDLL(so)
    import ansel_b200 as ab
    h, w = img.shape[:2]
    out = np.full_like(img, -7.0)
    f = _EMUL.emul_hl_laplacian
    f.restype = C.c_int
    shifted = ab.lib().b200_roi_filters(filters, x, y) if filters else 0
    xt = None
    if filters == 9:
        xt = (C.c_uint8 * 36)(*[xtrans[6 * ((r + y + 600) % 6) + (c + x + 600) % 6] for r in range(6) for c in range(6)])
    assert f(util.fptr(img), util.fptr(out), w, h, C.c_uint32(shifted), xt, F4(*clips), iterations, scales, C.c_float(noise_level), C.c_float(solid_color),
             C.c_float(iscale), C.c_float(roi_scale), F4(*norm)) == 0
    return out


def piece_of(ab, img, filters, *, clip=1.0, pmax=(1.0, 1.0, 1.0), iterations=2, scales=6, noise_level=0.0, solid_color=0.0, iscale=1.0, roi_scale=1.0,
             x=0, y=0, xtrans=None):
    h, w = img.shape[:2]
    d = ab.HighlightsData()
    d.mode, d.clip, d.iterations, d.scales, d.noise_level, d.solid_color = 3, clip, iterations, scales, noise_level, solid_color
    piece = ab.make_piece(w, h, filters=filters, channels=1 if filters else 4, data=d, devid=0, roi_x=x, roi_y=y, scale=roi_scale,
                          processed_maximum=tuple(pmax) + (1.0,))
    piece.roi_out.x, piece.roi_out.y, piece.iscale = x, y, iscale
    if xtrans is not None:
        for k, v in enumerate(xtrans):
            piece.xtrans[k // 6][k % 6] = int(v)
    return piece, d


def cuda(ab, img, filters, norm=None, through_module=False, **kw):
    """b200_highlights_laplacian_dev (norm: the vector to impose, None = the library's own) or the module's process_dev"""
    import torch
    piece, d = piece_of(ab, img, filters, **kw)
    d_in = torch.from_numpy(np.ascontiguousarray(img)).cuda()
    d_out = torch.full_like(d_in, -7.0)
    s = torch.cuda.current_stream().cuda_stream
    if through_module:
        ab.check(ab.lib().b200_highlights_process_dev(piece, d_in.data_ptr(), d_out.data_ptr(), s))
    else:
        nv = F4(*norm) if norm is not None else None
        ab.check(ab.lib().b200_highlights_laplacian_dev(piece, d_in.data_ptr(), d_out.data_ptr(), nv, s))
    torch.cuda.synchronize()
    return d_out.cpu().numpy()
