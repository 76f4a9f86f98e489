"""B200: several pipes at once, as the darkroom runs its preview and full pipes in two threads and a batch export keeps
several frames in flight (include/b200iop.h, "Threading").  Every output is compared bit for bit with the oracle.

Every expected output is computed before a worker thread starts; the workers only call the library (ctypes releases
the GIL) and copy, all released together by a barrier.  b200_last_error is per thread, so each worker checks its own
return codes.  Each case runs a fixed, small number of frames once."""
import ctypes as C
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np
import pytest

import util
import blend_util as bu
import hl_laplacian_util as hu
import lmmse_util as lu
import markesteijn_util as mu
from vng_util import XTRANS

pytestmark = pytest.mark.gpu
WORK = util.profile_pair(util.REC2020_TO_XYZ_D50)
EXPORT = util.profile_pair(util.SRGB_TO_XYZ_D50)
FILL = -7.0     # what output buffers start as: Markesteijn leaves lane 3 as found, AMaZE writes 0 there, LMMSE what the oracle does


def same_bits(a, b):
    return (a.view(np.uint32) == b.view(np.uint32)) | (np.isnan(a) & np.isnan(b))


def run_together(workers):
    """each callable in its own thread, released together; returns their results, re-raises the first failure"""
    barrier = threading.Barrier(len(workers))
    results, errors = [None] * len(workers), [None] * len(workers)

    def body(k):
        try:
            barrier.wait(timeout=120)
            results[k] = workers[k]()
        except BaseException as e:      # noqa: BLE001 -- handed to the main thread
            errors[k] = e
            barrier.abort()

    threads = [threading.Thread(target=body, args=(k,)) for k in range(len(workers))]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    for e in errors:
        if e is not None and not isinstance(e, threading.BrokenBarrierError):
            raise e
    for e in errors:
        if e is not None:
            raise e
    return results


def _lib():
    import ansel_b200 as ab
    ab.init()
    L = ab.lib()
    L.b200_blend_process_dev.restype = C.c_int
    L.b200_blend_process_dev.argtypes = [C.c_void_p, C.POINTER(bu.BlendParams), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.b200_kernel_timing_read.argtypes = [C.c_char_p, C.POINTER(C.c_double), C.POINTER(C.c_int)]
    return ab, L


def xtrans_piece(ab, w, h, x, y, passes):
    piece = ab.make_piece(w, h, filters=9, data=ab.demosaic_data(1025 if passes == 1 else 1026), devid=0, roi_x=x, roi_y=y)
    for i in range(6):
        for j in range(6):
            piece.xtrans[i][j] = int(XTRANS[i][j])
    return piece


# ---- Markesteijn: four threads, four geometries (the plan cache has two slots) ----------------------------------------
GEOMETRIES = [  # (w, h, x, y, passes, entry point): ROI origins 0, 1, 3, 4 columns and 0, 4, 2, 5 rows off the pattern
    mu.CASES["origin"] + (1, "dev"),
    mu.CASES["roi"] + (3, "dev"),
    mu.CASES["roi2"] + (1, "host"),
    (1203, 907, 4, 5, 3, "host"),
]


def test_markesteijn_four_threads_four_geometries(built):
    import torch
    ab, L = _lib()
    jobs = []
    for k, (w, h, x, y, passes, entry) in enumerate(GEOMETRIES):
        frames = [np.ascontiguousarray(util.frame_natural(w, h, 40 + 3 * k + i), np.float32) for i in range(3)]
        want = [mu.oracle(m, x, y, passes) for m in frames]
        jobs.append((w, h, x, y, passes, entry, frames, want))

    def worker(w, h, x, y, passes, entry, frames, want):
        piece = xtrans_piece(ab, w, h, x, y, passes)
        if entry == "host":
            outs = [np.full((h, w, 4), FILL, np.float32) for _ in frames]
            for m, o in zip(frames, outs):
                ab.check(L.b200_demosaic_process_host(C.byref(piece), m.ctypes.data, o.ctypes.data))
            return outs
        s = torch.cuda.Stream()
        with torch.cuda.stream(s):          # torch's current stream is per thread
            d_in = [torch.from_numpy(m).cuda() for m in frames]
            d_out = [torch.full((h, w, 4), FILL, device="cuda") for _ in frames]
            for i, o in zip(d_in, d_out):
                ab.check(L.b200_demosaic_process_dev(C.byref(piece), i.data_ptr(), o.data_ptr(), torch.cuda.current_stream().cuda_stream))
            s.synchronize()
            return [o.cpu().numpy() for o in d_out]

    results = run_together([lambda j=j: worker(*j) for j in jobs])
    for (w, h, x, y, passes, entry, _, want), outs in zip(jobs, results):
        for i, (got, wnt) in enumerate(zip(outs, want)):
            assert same_bits(got[..., :3], wnt[..., :3]).all(), (w, h, x, y, passes, entry, i)
            assert (got[..., 3] == FILL).all(), (w, h, entry, i)


def test_markesteijn_plan_evicted_while_its_frame_is_queued(built):
    """one thread, a pipe queue of depth 3: three X-Trans geometries cycle through two plan slots, so a plan is replaced while
    the frame that uses it may still wait on another slot's stream"""
    import torch
    import ansel_b200.dtsurface as ds
    ab, L = _lib()
    M = ds.modlib()
    geos = [(300, 210, 0, 0, 1), (264, 148, 3, 2, 3), (131, 127, 1, 4, 1)]
    pipe = ds.make_pipe(devid=0)
    keep, nodes = [], []
    for (w, h, x, y, passes) in geos:
        piece = ds.make_piece_iop("demosaic", w, h, ab.demosaic_data(1025 if passes == 1 else 1026), channels_in=1, channels_out=4, filters=9)
        piece.roi_in = ds.Roi(x, y, w, h, 1.0)
        for k in range(36):
            piece.dsc_in.xtrans[k] = int(XTRANS[k // 6][k % 6])
        node = (ds.PipeNode * 1)()
        node[0].process_cl = C.cast(M.dt_iop_demosaic__process_cl, C.c_void_p)
        node[0].module = piece.module
        node[0].piece = C.pointer(piece)
        keep.append(piece)
        nodes.append(node)
    order = [k % 3 for k in range(7)]
    frames = [np.ascontiguousarray(util.frame_natural(geos[g][0], geos[g][1], 60 + i), np.float32) for i, g in enumerate(order)]
    want = [mu.oracle(m, geos[g][2], geos[g][3], geos[g][4]) for m, g in zip(frames, order)]
    ins = [torch.from_numpy(m).pin_memory() for m in frames]
    outs = [torch.zeros((geos[g][1], geos[g][0], 4), dtype=torch.float32).pin_memory() for g in order]
    q = M.b200_pipe_queue_new(3)
    assert q
    try:
        tickets = [M.b200_pixelpipe_submit(q, C.byref(pipe), nodes[g], 1, i.data_ptr(), o.data_ptr()) for g, i, o in zip(order, ins, outs)]
        assert tickets == list(range(len(order))), L.b200_last_error()
        for t in tickets:
            assert M.b200_pixelpipe_wait(q, t) == 0
    finally:
        M.b200_pipe_queue_free(q)
    for i, (o, wnt) in enumerate(zip(outs, want)):     # lane 3 is whatever the slot's buffer held
        assert same_bits(o.numpy()[..., :3], wnt[..., :3]).all(), (i, geos[order[i]])


# ---- LMMSE: the first call of a process, from four threads at once ----------------------------------------------------
CHILD = r"""
import ctypes as C, faulthandler, os, sys, threading
import numpy as np
faulthandler.enable()
root, tmp = sys.argv[1], sys.argv[2]
sys.path.insert(0, root)
import ansel_b200 as ab
ab.init()
L = ab.lib()
jobs = [tuple(int(v) for v in open(os.path.join(tmp, f"job{k}.txt")).read().split()) for k in range(4)]
barrier = threading.Barrier(4)
failed = []

def work(k, mode, filters):
    try:
        m = np.load(os.path.join(tmp, f"in{k}.npy"))
        h, w = m.shape
        d = ab.demosaic_data(6)
        d.lmmse_refine = mode
        piece = ab.make_piece(w, h, filters=filters, data=d, devid=0, processed_maximum=(1.0, 0.9, 1.1, 1.0))
        out = np.full((h, w, 4), -7.0, np.float32)
        barrier.wait(timeout=120)
        ab.check(L.b200_demosaic_process_host(C.byref(piece), m.ctypes.data, out.ctypes.data))
        np.save(os.path.join(tmp, f"out{k}.npy"), out)
    except BaseException as e:
        failed.append(f"thread {k}: {e!r}")
        barrier.abort()

threads = [threading.Thread(target=work, args=(k,) + jobs[k]) for k in range(4)]
for t in threads:
    t.start()
for t in threads:
    t.join()
# Python's join() returns before a thread's C++ thread-local destructors have run, and the library frees each thread's
# device memory, streams and pinned buffers there.  A normal exit would tear the CUDA runtime down under them: leave
# without running exit handlers, the outputs are on disk.
sys.stderr.write("\n".join(failed))
sys.stderr.flush()
os._exit(1 if failed else 0)
"""


def test_lmmse_first_use_from_four_threads(built):
    """the gamma tables are made by the first LMMSE call of a process on a device: four threads make it together"""
    assert lu.PMAX == (1.0, 0.9, 1.1)
    jobs = [("rggb", 0), ("bggr_odd", 1), ("grbg_one_tile", 3), ("rggb_wide", 4)]
    with tempfile.TemporaryDirectory() as tmp:
        want = []
        for k, (name, mode) in enumerate(jobs):
            m, f = lu.case(name, seed=30 + k)
            np.save(os.path.join(tmp, f"in{k}.npy"), m)
            with open(os.path.join(tmp, f"job{k}.txt"), "w") as fh:
                fh.write(f"{mode} {f}")
            want.append(lu.oracle(m, f, mode, carry=0))
        r = subprocess.run([sys.executable, "-c", CHILD, util.ROOT, tmp], capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr[-4000:]
        for k, (name, mode) in enumerate(jobs):
            got = np.load(os.path.join(tmp, f"out{k}.npy"))
            assert same_bits(got, want[k]).all(), (name, mode)


# ---- four different chains at once -----------------------------------------------------------------------------------
def _oracle_nlm_module(img, data):
    f = util.oracle().orc_denoiseprofile_nlmeans
    f.restype = C.c_int
    out = np.zeros_like(img)
    h, w = img.shape[:2]
    assert f(util.fptr(np.ascontiguousarray(img)), util.fptr(out), w, h, C.byref(data), C.c_float(1.0), 1, (C.c_float * 4)(2.0, 1.0, 1.5, 0.0),
             (C.c_float * 4)(1.0, 1.0, 1.0, 1.0)) == 0
    return out


class Chain:
    """one thread's device-resident modules on its own stream; every stage's output is kept for the comparison"""

    def __init__(self, ab, L, w, h):
        import torch
        self.torch, self.ab, self.L, self.w, self.h = torch, ab, L, w, h
        self.stream = torch.cuda.Stream()
        self.stages = []

    def dev(self, a):
        return self.torch.from_numpy(np.ascontiguousarray(a)).cuda()

    def buf(self, fill=0.0):
        return self.torch.full((self.h, self.w, 4), fill, device="cuda")

    def keep(self, name, d):
        self.stages.append((name, d))
        return d

    def run(self, op, data, src, channels_in=4, filters=0, fill=0.0, **piece_kw):
        piece = self.ab.make_piece(self.w, self.h, filters=filters, channels=channels_in, devid=0, **piece_kw)
        piece.data, piece.data_size = C.addressof(data), C.sizeof(data)
        if op == "demosaic" and filters == 9:
            for i in range(6):
                for j in range(6):
                    piece.xtrans[i][j] = int(XTRANS[i][j])
        dst = self.buf(fill)
        self.ab.check(getattr(self.L, f"b200_{op}_process_dev")(C.byref(piece), src.data_ptr(), dst.data_ptr(), self.stream.cuda_stream))
        return self.keep(op, dst)

    def finish(self):
        self.stream.synchronize()
        return [(name, d.cpu().numpy()) for name, d in self.stages]


def test_four_different_chains_at_once(built):
    import torch
    ab, L = _lib()
    rggb = util.BAYER["RGGB"]
    enc = util.srgb_encode_lut()
    co_t = util.fit_unbounded_coeffs(enc)
    blob = np.load(os.path.join(util.GOLDEN_DIR, "filmic_data.npz"))["default_v8"]

    # 1. C3 in small: RCD -> denoiseprofile (NLM) -> colorin -> filmic rgb.  RCD leaves a few pixels undefined in the reference
    # (tests/test_chains_gpu.py): the oracle chain starts from the kernel's own demosaic, made here before the threads start.
    w1, h1 = 480, 320
    mosaic1 = util.frame_natural(w1, h1, 71)
    conv_in = ab.make_conversion(util.MATRIX_CAM_TO_REC2020)
    dn = ab.denoiseprofile_data(ab.DENOISE_NLMEANS, radius=1, nbhood=7)
    fpiece = ab.filmic_piece(blob, WORK, EXPORT)
    piece = ab.make_piece(w1, h1, filters=rggb, data=ab.demosaic_data(ab.DEMOSAIC_RCD), devid=0)
    d_mosaic, d_dem = torch.from_numpy(mosaic1).cuda(), torch.zeros((h1, w1, 4), device="cuda")
    ab.check(L.b200_demosaic_process_dev(C.byref(piece), d_mosaic.data_ptr(), d_dem.data_ptr(), torch.cuda.current_stream().cuda_stream))
    dem1 = d_dem.cpu().numpy()
    defined1 = (util.oracle_rcd_mask(mosaic1, rggb) & 1) == 0
    o_rcd = util.oracle_rcd(mosaic1, rggb)
    assert (same_bits(dem1[..., :3], o_rcd[..., :3]).all(axis=2) | ~defined1).all()
    o = _oracle_nlm_module(dem1, dn)
    want1 = {"denoiseprofile": o}
    o = want1["colorin"] = util.oracle_convert(o, util.MATRIX_CAM_TO_REC2020, fp=util.FP_CONTRACT)
    want1["filmicrgb"] = util.oracle_filmic_agx(o, blob, WORK, EXPORT)

    def c3():
        ch = Chain(ab, L, w1, h1)
        with torch.cuda.stream(ch.stream):
            g = ch.run("demosaic", ab.demosaic_data(ab.DEMOSAIC_RCD), ch.dev(mosaic1), channels_in=1, filters=rggb)
            g = ch.run("denoiseprofile", dn, g)
            g = ch.run("colorin", ab.colorin_data(conv_in), g)
            ch.run("filmicrgb", fpiece, g)
            return ch.finish()

    # 2. AMaZE -> colorout with a tone curve: the curve goes through the library's per-device cache (identity != 0)
    w2, h2 = 501, 333
    mosaic2 = util.frame_natural(w2, h2, 72)
    conv_out = ab.make_conversion(util.MATRIX_REC2020_TO_SRGB, lut_target=enc, coeffs_target=co_t, identity=0x5151)
    o = util.oracle_amaze(mosaic2, rggb)
    want2 = {"demosaic": o, "colorout": util.oracle_convert(o, util.MATRIX_REC2020_TO_SRGB, lut_t=enc, co_t=co_t, fp=util.FP_CONTRACT)}

    def amaze_colorout():
        ch = Chain(ab, L, w2, h2)
        with torch.cuda.stream(ch.stream):
            g = ch.run("demosaic", ab.demosaic_data(ab.DEMOSAIC_AMAZE), ch.dev(mosaic2), channels_in=1, filters=rggb, fill=FILL)
            ch.run("colorout", ab.colorout_data(conv_out), g)
            return ch.finish()

    # 3. LMMSE -> RGB to Lab -> blend in Lab (a parametric mask on L of the input and b of the output: from 0 to the opacity)
    mosaic3, f3 = lu.case("bggr_odd", seed=73)
    h3, w3 = mosaic3.shape
    o = lu.oracle(mosaic3, f3, 2, carry=0)
    want3 = {"demosaic": o}
    o = want3["glue"] = util.oracle_rgb_to_lab(o, WORK)
    layer = bu.frames_lab(w3, h3, 73)[1]
    bp = bu.params(cst=bu.CS_LAB, mode="softlight", mask_mode=bu.MASK_ENABLED | bu.MASK_PARAMETRIC, channels={0: (0.1, 0.3, 0.7, 0.9), 6: (0.4, 0.5, 0.6, 0.8)})
    rc, want3["blend"], want3["mask"] = bu.oracle(o, layer, bp)
    assert rc == 0
    pm = ab.profile_matrices(*WORK)
    glue = L.b200_colorspace_transform_dev
    glue.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(ab.ProfileMatrices), C.c_int, C.c_void_p]

    def lmmse_lab_blend():
        ch = Chain(ab, L, w3, h3)
        with torch.cuda.stream(ch.stream):
            d = ab.demosaic_data(6)
            d.lmmse_refine = 2
            g = ch.run("demosaic", d, ch.dev(mosaic3), channels_in=1, filters=f3, fill=FILL, processed_maximum=lu.PMAX + (1.0,))
            lab = ch.keep("glue", g.clone())        # in place, as the pipe does: lane 3 is kept
            ab.check(glue(lab.data_ptr(), lab.data_ptr(), w3, h3, ab.CS_RGB, ab.CS_LAB, C.byref(pm), 0, ch.stream.cuda_stream))
            out = ch.keep("blend", ch.dev(layer))
            mask = ch.keep("mask", torch.full((h3, w3), -3.0, device="cuda"))
            bpiece = ab.make_piece(w3, h3, channels=4, devid=0)
            ab.check(L.b200_blend_process_dev(C.byref(bpiece), C.byref(bp), lab.data_ptr(), out.data_ptr(), None, mask.data_ptr(),
                                              ch.stream.cuda_stream))
            return ch.finish()

    # 4. Markesteijn -> highlights' guided Laplacians on its RGBA output (some of it beyond the clip)
    w4, h4, x4, y4 = 420, 300, 2, 1
    mosaic4 = np.ascontiguousarray(util.frame_natural(w4, h4, 74) * np.float32(1.6))
    o = mu.oracle(mosaic4, x4, y4, 1)
    hl_kw = dict(iterations=2, noise_level=0.1, solid_color=0.1)
    hl_want, hl_norm = hu.oracle(o, 0, hu.clips_of(), **hl_kw)
    want4 = {"demosaic": o, "highlights": hl_want}
    hpiece, _hd = hu.piece_of(ab, o, 0, **hl_kw)
    norm = (C.c_float * 4)(*hl_norm)

    def markesteijn_highlights():
        ch = Chain(ab, L, w4, h4)
        with torch.cuda.stream(ch.stream):
            g = ch.run("demosaic", ab.demosaic_data(1025), ch.dev(mosaic4), channels_in=1, filters=9, fill=FILL, roi_x=x4, roi_y=y4)
            out = ch.keep("highlights", ch.buf(FILL))
            ab.check(L.b200_highlights_laplacian_dev(hpiece, g.data_ptr(), out.data_ptr(), norm, ch.stream.cuda_stream))
            return ch.finish()

    torch.cuda.synchronize()
    results = run_together([c3, amaze_colorout, lmmse_lab_blend, markesteijn_highlights])
    c3_out = dict(results[0])
    assert same_bits(c3_out["demosaic"], dem1).all(), "C3: RCD"
    for name, want in want1.items():
        assert same_bits(c3_out[name], want).all(), f"C3: {name}"
    for k, want in ((1, want2), (2, want3), (3, want4)):
        got = dict(results[k])
        for name, wnt in want.items():
            if name == "demosaic" and k == 3:
                assert same_bits(got[name][..., :3], wnt[..., :3]).all() and (got[name][..., 3] == FILL).all(), (k, name)
            else:
                assert same_bits(got[name], wnt).all(), (k, name)


# ---- kernel timing from two threads -------------------------------------------------------------------------------------
def test_kernel_timing_from_two_threads(built):
    """every launch gets its own pair of events, whichever thread times what at the same moment"""
    import torch
    ab, L = _lib()
    K = 3
    w, h = 640, 480
    rggb = util.BAYER["RGGB"]
    mosaic = util.frame_natural(w, h, 80)
    img = (util.rgba_scene(320, 240, 81, noise=0.02) * 60).astype(np.float32)
    assert L.b200_kernel_timing(1) == 0
    try:
        def worker():
            s = torch.cuda.Stream()
            with torch.cuda.stream(s):
                d_m, d_rgb = torch.from_numpy(mosaic).cuda(), torch.zeros((h, w, 4), device="cuda")
                d_img, d_nlm = torch.from_numpy(img).cuda(), torch.zeros_like(torch.from_numpy(img)).cuda()
                s.synchronize()
                piece = ab.make_piece(w, h, filters=rggb, data=ab.demosaic_data(ab.DEMOSAIC_RCD), devid=0)
                t0 = time.perf_counter()
                for _ in range(K):
                    ab.check(L.b200_demosaic_process_dev(C.byref(piece), d_m.data_ptr(), d_rgb.data_ptr(), s.cuda_stream))
                    ab.check(L.b200_nlmeans_denoise_dev(d_img.data_ptr(), d_nlm.data_ptr(), 320, 240, 0.0, 1.0, 1.0, 1.0, 0.1, 0.005, 1, 7, 0,
                                                        (C.c_float * 4)(1.0, 1.0, 1.0, 1.0), s.cuda_stream))
                s.synchronize()
                return (time.perf_counter() - t0) * 1e3, d_nlm.cpu().numpy()

        results = run_together([worker, worker])
        wall_ms = sum(r[0] for r in results)
        for name in ("rcd_tiles_kernel", "nlm_kernel"):
            total, count = C.c_double(), C.c_int()
            ab.check(L.b200_kernel_timing_read(name.encode(), C.byref(total), C.byref(count)))
            assert count.value == 2 * K, (name, count.value)
            assert 0.0 < total.value <= wall_ms, (name, total.value, wall_ms)
    finally:
        assert L.b200_kernel_timing(0) == 0
    want = util.oracle_nlmeans(img)
    for _, got in results:
        assert same_bits(got, want).all()
