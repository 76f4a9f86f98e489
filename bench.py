#!/usr/bin/env python
"""bench.py -- the develop-pipe benchmark contract (see DESIGN.md "Measurement").

  python bench.py --gpus N --steps K --warmup W              # this repo's B200 path
  python bench.py --impl reference --gpus N --steps K ...    # the reference's CPU path (oracle/_ref)

Workload (BASELINE.json configs[2], SURVEY.md 8d "C3", the pipe north_star sets its target on): one synthetic 45.44 MP RGGB
Bayer frame (8256x5504, D-natural, seed 20260922) per step through
    demosaic(RCD) -> denoiseprofile(non-local means, P = 1, K = 7) -> colorin(matrix) -> filmicrgb(v8 defaults).
A "step" is one frame through that chain.
  value : device-resident chain throughput, MP/s, frames already in HBM, CUDA-event timed.
  e2e   : the same chain through the C module adapters and the device-resident pixelpipe glue
          (ansel_b200/iop/), host (pinned) buffers in and out, H2D + D2H inside the timed region.
  config.c2 : the lighter chain of configs[1] (RCD -> colorin -> colorout), same frame, device-resident.
Multi-GPU (torchrun): frames are independent, each rank develops its own frame per step, no data-path collective (weak
scaling, SURVEY.md 8e "batch (C5) replicas"); `banded_one_frame` reports the second mode, ONE frame in row bands.
"""
from __future__ import annotations

import os
import sys


def _physical_cores() -> int:
    """cores this process may run on, one per (package, core) pair"""
    try:
        allowed = os.sched_getaffinity(0)
    except AttributeError:
        allowed = set(range(os.cpu_count() or 1))
    seen, cpu, phys = set(), None, None
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("processor"):
                cpu = int(line.split(":")[1])
            elif line.startswith("physical id"):
                phys = int(line.split(":")[1])
            elif line.startswith("core id") and cpu in allowed:
                seen.add((phys, int(line.split(":")[1])))
    except OSError:
        pass
    return len(seen) or max(1, len(allowed) // 2)


# The CPU arm is OpenMP: BASELINE.md section 3 asks for one thread per physical core, bound (OMP_PROC_BIND=close).  libgomp reads
# these when it is loaded, so they are set before anything imports it -- and a launcher's OMP_NUM_THREADS=1 (torchrun exports it to
# every rank) is not the machine's answer: it is overridden, a user's explicit B200_BENCH_OMP_THREADS is kept.
_CPU_THREADS = int(os.environ.get("B200_BENCH_OMP_THREADS", "0")) or _physical_cores()
os.environ["OMP_NUM_THREADS"] = str(_CPU_THREADS)
os.environ.setdefault("OMP_PROC_BIND", "close")
os.environ.setdefault("OMP_PLACES", "cores")

import argparse  # noqa: E402
import ctypes as C  # noqa: E402
import json  # noqa: E402
import threading  # noqa: E402
import time  # noqa: E402

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import warnings  # noqa: E402

warnings.filterwarnings("ignore")  # numpy notices the FTZ/DAZ mode the reference sets on its threads

import numpy as np  # noqa: E402

METRIC = "megapixels/sec full develop pipe @45MP"
UNIT = "MP/s"
WORKLOAD = ("C3: 45MP RGGB Bayer (8256x5504) -> demosaic(RCD) -> denoiseprofile(non-local means P=1 K=7) -> colorin(matrix) "
            "-> filmicrgb(v8 defaults)")
WORKLOAD_C2 = "C2: 45MP RGGB Bayer (8256x5504) -> demosaic(RCD) -> colorin(matrix) -> colorout(matrix+sRGB TRC)"
W45, H45 = 8256, 5504
SEED = 20260922
WB = (2.0, 1.0, 1.5, 0.0)           # white-balance coefficients the denoise profile sees (the tests' values)
ALGO_BYTES_PER_PX = {"demosaic": 20, "denoiseprofile": 32, "colorin": 32, "filmicrgb": 32, "colorout": 32}  # SURVEY.md 8(d)
# non-local means, arithmetic per pixel and patch as the reference's loops write it (nlmeans_core.c:384-483): column sums 12 (x 1.07
# for the halo columns and rows), running distortion 2, weight and accumulation 24 -> 38.8 flop; 225 patches at K = 7
NLM_FLOP_PER_PX_PATCH = 12 * 1.07 + 2 + 24
FP32_PEAK_TFLOPS = 148 * 4 * 32 * 2 * 1.965e9 / 1e12   # 148 SMs x 4 schedulers x one packed (2-wide) 32-lane FP32 instruction per clock


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=60)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--width", type=int, default=W45)
    ap.add_argument("--height", type=int, default=H45)
    ap.add_argument("--e2e-steps", type=int, default=12)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the C3 chain returned in its last step to DIR/c3_out.npy (float32 RGBA; the whole "
                         "frame when it fits 64 MB, else a fixed seeded sample of its pixels in ascending order)")
    ap.add_argument("--no-batch", action="store_true", help="skip the 64-frame batch export (BASELINE.json configs[4])")
    ap.add_argument("--c4", action="store_true", help="at N > 1: also the 100 MP C4 chain over the ranks (always run at N = 4, the configuration BASELINE.json names)")
    ap.add_argument("--no-other-modules", action="store_true", help="skip the untimed per-module table of the non-C2 modules")
    ap.add_argument("--pipe-ends-only", action="store_true",
                    help="internal: run the pipe-end module table in this process and print it as one JSON object (the main run calls this in a "
                         "child process so that code which has not been through a GPU round cannot take the headline down)")
    return ap.parse_args()


DUMP_BYTES = 64_000_000
DUMP_PIXELS = 1 << 21          # 32 MiB of RGBA float32


def dump_outputs(out_dir, frame):
    """write the (h, w, 4) device frame to out_dir/c3_out.npy: whole, or DUMP_PIXELS-odd pixels drawn with the bench seed"""
    os.makedirs(out_dir, exist_ok=True)
    px = frame.reshape(-1, 4)
    if px.numel() * 4 <= DUMP_BYTES:
        arr = frame.cpu().numpy()
    else:
        import torch
        idx = np.unique(np.random.default_rng(SEED).integers(0, px.shape[0], DUMP_PIXELS))
        arr = px[torch.from_numpy(idx).to(px.device)].cpu().numpy()
    np.save(os.path.join(out_dir, "c3_out.npy"), np.ascontiguousarray(arr, np.float32))


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------
# CPU arm: the reference's own sources compiled by oracle/Makefile (oracle/_ref), else the port
# ------------------------------------------------------------------------------------------
class CpuChain:
    """The C3 chain (or C2) on the host cores, module by module as pixelpipe_process_on_CPU calls them: rcd_demosaic ->
    [precondition_v2 -> nlmeans_denoise -> backtransform_v2] (process_nlmeans_cpu, denoiseprofile.c:1599-1648) ->
    dt_colorspaces_apply_matrix_conversion (colorin) -> filmic's AgX loop.  Runs on any frame height (bounded samples)."""

    def __init__(self, w, h, chain="c3"):
        import util
        import ansel_b200 as ab
        self.util, self.ab = util, ab
        self.w, self.h, self.chain = w, h, chain
        self.kind = "reference" if util.ref("fast") is not None else "port"
        self.lib = util.ref("fast") if self.kind == "reference" else util.oracle()
        self.enc = util.srgb_encode_lut()
        self.co_t = util.fit_unbounded_coeffs(self.enc)
        self.rgb = [util.aligned_empty((h, w, 4)) for _ in range(3)]
        self.work = util.profile_pair(util.REC2020_TO_XYZ_D50)
        self.export = util.profile_pair(util.SRGB_TO_XYZ_D50)
        self.fblob = np.ascontiguousarray(np.load(os.path.join(util.GOLDEN_DIR, "filmic_data.npz"))["default_v8"])
        self.dn = ab.denoiseprofile_data(ab.DENOISE_NLMEANS, radius=1, nbhood=7)
        plan = np.zeros(51, np.float32)
        f4 = lambda v: (C.c_float * 4)(*v)  # noqa: E731
        util.oracle().orc_dn_plan_export_nlm(C.byref(self.dn), C.c_float(1.0), w, h, f4(WB), f4((1.0, 1.0, 1.0, 1.0)), util.fptr(plan))
        self.vst = dict(wb=f4(plan[1:5]), p=f4(plan[5:9]), a=C.c_float(plan[9]), b=C.c_float(plan[10]), bias=C.c_float(plan[11]))
        self.f9 = [np.ascontiguousarray(m, np.float32).reshape(-1).copy() for m in (*self.work, *self.export)]

    def _conv(self, src, dst, matrix, lut_t=None, co_t=None):
        u = self.util
        m = np.ascontiguousarray(matrix, np.float32).reshape(-1)
        lt = u.fptr(lut_t) if lut_t is not None else None
        ct = u.fptr(np.ascontiguousarray(co_t, np.float32).reshape(-1)) if co_t is not None else None
        if self.kind == "reference":
            f = self.lib.ref_apply_matrix_conversion
            f.restype = C.c_int
            f(u.fptr(src), u.fptr(dst), C.c_size_t(self.w), C.c_size_t(self.h), u.fptr(m), None, C.c_int(0), None, None, lt, ct)
        else:
            f = self.lib.orc_apply_matrix_conversion
            f.restype = C.c_int
            f(u.fptr(src), u.fptr(dst), C.c_size_t(self.w), C.c_size_t(self.h), u.fptr(m), None, C.c_int(0), None, None, lt, ct,
              C.c_int(u.FP_CONTRACT))

    def _denoise(self, src, tmp, dst):
        u, v, w, h = self.util, self.vst, self.w, self.h
        if self.kind != "reference":
            f = self.lib.orc_denoiseprofile_nlmeans
            f.restype = C.c_int
            f(u.fptr(src), u.fptr(dst), w, h, C.byref(self.dn), C.c_float(1.0), 1, (C.c_float * 4)(*WB), (C.c_float * 4)(1.0, 1.0, 1.0, 1.0))
            return
        L = self.lib
        L.ref_dn_precondition_v2(u.fptr(src), u.fptr(tmp), w, h, v["a"], v["p"], v["b"], v["wb"])
        norm = np.float32(0.045) / np.float32(9.0)           # nlmeans_norm(), denoiseprofile.c:1456-1470, P = 1
        L.ref_nlmeans_denoise(u.fptr(tmp), u.fptr(dst), w, h, C.c_float(0.0), C.c_float(1.0), C.c_float(1.0), C.c_float(1.0),
                              C.c_float(self.dn.central_pixel_weight), C.c_float(norm), 1, 7, 0, (C.c_float * 4)(1.0, 1.0, 1.0, 1.0))
        L.ref_dn_backtransform_v2(u.fptr(dst), w, h, v["a"], v["p"], v["b"], v["bias"], v["wb"])

    def _filmic(self, src, dst):
        u = self.util
        f = self.lib.ref_filmic_agx if self.kind == "reference" else self.lib.orc_filmic_agx
        f(u.fptr(src), u.fptr(dst), C.c_size_t(self.w), C.c_size_t(self.h), self.fblob.ctypes.data_as(C.c_void_p), *[u.fptr(m) for m in self.f9])

    def step(self, mosaic):
        u = self.util
        pm = (C.c_float * 3)(1.0, 1.0, 1.0)
        f = getattr(self.lib, "ref_rcd_demosaic" if self.kind == "reference" else "orc_rcd_demosaic")
        f.restype = C.c_int
        a, b, c = self.rgb
        f(u.fptr(a), u.fptr(mosaic), self.w, self.h, C.c_uint32(u.BAYER["RGGB"]), pm, C.c_float(0.0))
        if self.chain == "c2":
            self._conv(a, b, u.MATRIX_CAM_TO_REC2020)
            self._conv(b, c, u.MATRIX_REC2020_TO_SRGB, self.enc, self.co_t)
            return c
        self._denoise(a, b, c)
        self._conv(c, a, u.MATRIX_CAM_TO_REC2020)
        self._filmic(a, b)
        return b


def cpu_sample_rows(w, h, budget_s, steps):
    """rows of the frame one CPU step develops so that `steps` steps fit `budget_s` seconds: a full-width strip (the chunk
    grids of the tiled modules keep their widths; the strip height keeps a multiple of 64 rows = the NLM chunk rows of this frame)"""
    probe_h = 256
    chain = CpuChain(w, probe_h)
    import util
    mosaic = util.frame_natural(w, probe_h, SEED)
    chain.step(mosaic)
    t0 = time.perf_counter()
    chain.step(mosaic)
    per_row = (time.perf_counter() - t0) / probe_h
    rows = int(budget_s / max(steps, 1) / per_row)
    if rows >= h:
        return h, per_row
    return max(256, rows // 64 * 64), per_row


def time_cpu(chain, mosaic, warm, steps):
    for _ in range(warm):
        chain.step(mosaic)
    ts = []
    for _ in range(steps):
        t0 = time.perf_counter()
        chain.step(mosaic)
        ts.append(time.perf_counter() - t0)
    return ts


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import util
    w, h = args.width, args.height
    warm, steps = max(args.warmup, 3), max(args.steps, 1)
    rows, per_row = cpu_sample_rows(w, h, 150.0, warm + steps)
    mosaic = util.frame_natural(w, h, SEED)[:rows].copy()
    chain = CpuChain(w, rows)
    ts = time_cpu(chain, mosaic, warm, steps)
    med = float(np.median(ts))
    mps = w * rows / med / 1e6
    sample = (f"{len(ts)} steps after {warm} warm-ups, each the top {rows} rows of the {w}x{h} frame through the chain "
              f"({'the whole frame' if rows == h else 'a bounded sample: the full frame would take %.1f s per step' % (per_row * h)}); median step")
    line = {
        "impl": "reference", "metric": METRIC, "value": mps, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * med, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "frame": f"{w}x{h}", "cpu_threads": _CPU_THREADS, "host_logical_cpus": os.cpu_count(),
                   "omp": {k: os.environ.get(k) for k in ("OMP_NUM_THREADS", "OMP_PROC_BIND", "OMP_PLACES")},
                   "what": "reference sources compiled in place (oracle/_ref, release flags)" if chain.kind == "reference"
                   else "oracle port (oracle/_ref not built)",
                   "sample_rows": rows, "step_ms": [round(1e3 * t, 1) for t in ts]},
        "cpu_baseline": {"value": mps, "unit": UNIT, "cores": _CPU_THREADS, "kind": chain.kind, "sample": sample},
        "e2e": {"value": mps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------
# clocks: sample SM clock and throttle reasons during the timed region
# ------------------------------------------------------------------------------------------
class ClockSampler:
    def __init__(self, index):
        self.samples, self.reasons, self.stop = [], set(), threading.Event()
        self.max_mhz = None
        try:
            import pynvml
            self.nv = pynvml
            pynvml.nvmlInit()
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None
        self.t = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        nv = self.nv
        names = {"nvmlClocksEventReasonHwSlowdown": "hw_slowdown", "nvmlClocksEventReasonHwThermalSlowdown": "hw_thermal_slowdown",
                 "nvmlClocksEventReasonSwThermalSlowdown": "sw_thermal_slowdown", "nvmlClocksEventReasonSwPowerCap": "sw_power_cap",
                 "nvmlClocksThrottleReasonHwSlowdown": "hw_slowdown", "nvmlClocksThrottleReasonHwThermalSlowdown": "hw_thermal_slowdown",
                 "nvmlClocksThrottleReasonSwThermalSlowdown": "sw_thermal_slowdown", "nvmlClocksThrottleReasonSwPowerCap": "sw_power_cap"}
        bits = {getattr(nv, k): v for k, v in names.items() if hasattr(nv, k)}
        while not self.stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for b, name in bits.items():
                    if r & b:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.01)

    def __enter__(self):
        if self.nv:
            self.t.start()
        return self

    def __exit__(self, *a):
        self.stop.set()
        if self.nv:
            self.t.join(timeout=1)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["unavailable"]}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


# ------------------------------------------------------------------------------------------
# B200 arm
# ------------------------------------------------------------------------------------------
def pipe_ends_extras(ab, ds, util, L, M, torch, w, h, local, dev, stream, conv_in, conv_out, d_cin, d_cout):
    """Per-module device times of rawprepare / temperature / highlights(clip) / their fused pass / exposure / gamma /
    finalscale at the bench frame size, and the sensor-to-display chain end to end: uint16 sensor data up (2 B/px), uint8
    display pixels down (4 B/px), rawprepare -> temperature -> highlights -> demosaic(RCD) -> colorin -> colorout -> gamma
    through the C module adapters with two frames in flight."""
    npx = w * h
    wb = (2.13, 1.0, 1.57, 1.02)
    pm = (wb[0], wb[1], wb[2], 0.0)
    filters = util.BAYER["RGGB"]
    sub, div = (512.0, 520.0, 508.0, 515.0), (15871.0, 15863.0, 15875.0, 15868.0)
    rng = np.random.default_rng(SEED)
    raw = np.clip(util.frame_natural(w, h, SEED) * 15871.0 * 0.45 + 512.0 + rng.normal(0, 3, (h, w)), 0, 16383).astype(np.uint16)
    raw[rng.integers(0, h, 4000), rng.integers(0, w, 4000)] = 16383           # blown samples: highlights takes the clip branch
    d_rp, d_tp, d_hl = ab.rawprepare_data(sub, div), ab.temperature_data(wb), ab.highlights_data(ab.HIGHLIGHTS_CLIP, 1.0)
    d_ex, d_fs, d_dem = ab.exposure_data(0.0, 0.5), ab.finalscale_data(ab.INTERPOLATION_MITCHELL), ab.demosaic_data(ab.DEMOSAIC_RCD)

    def piece(data, ch, datatype=ab.TYPE_FLOAT, pmax=(1.0, 1.0, 1.0, 1.0), out=None):
        p = ab.make_piece(w, h, filters=filters if ch == 1 else 0, channels=ch, data=data, processed_maximum=pmax, devid=local,
                          out_width=out[0] if out else None, out_height=out[1] if out else None)
        p.datatype = datatype
        return p

    p_rp, p_tp, p_hl = piece(d_rp, 1, ab.TYPE_UINT16), piece(d_tp, 1), piece(d_hl, 1, pmax=pm)
    p_ex, p_gm = piece(d_ex, 4), piece(None, 4)
    p_fs = piece(d_fs, 4, out=(w // 2, h // 2))
    p_fs.roi_out.scale = 0.5
    t_raw = torch.from_numpy(raw).to(dev)
    t_m = [torch.empty((h, w), dtype=torch.float32, device=dev) for _ in range(2)]
    t_rgba = torch.rand((h, w, 4), dtype=torch.float32, device=dev)
    t_out = torch.empty((h, w, 4), dtype=torch.float32, device=dev)
    t_u8 = torch.zeros((h, w, 4), dtype=torch.uint8, device=dev)

    def timed(call, reps=5):
        call()
        torch.cuda.synchronize()
        ts = []
        for _ in range(reps):
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a0.record()
            call()
            a1.record()
            torch.cuda.synchronize()
            ts.append(a0.elapsed_time(a1))
        return float(np.median(ts))

    res = {}

    def report(label, call, bytes_per_px, reps=5):
        """time one entry point; a failure is recorded under its label and does not stop the table"""
        try:
            ms = timed(call, reps)
            res[label] = {"ms": ms, "MP_per_s": npx / ms / 1e3, "algorithmic_GBps": bytes_per_px * npx / (ms * 1e-3) / 1e9,
                          "algorithmic_bytes_per_px": bytes_per_px}
        except Exception as e:
            res[label] = {"unavailable": f"{type(e).__name__}: {e}"[:200]}

    report("rawprepare_uint16", lambda: ab.check(L.b200_rawprepare_process_dev(p_rp, t_raw.data_ptr(), t_m[0].data_ptr(), stream)), 6)
    report("temperature", lambda: ab.check(L.b200_temperature_process_dev(p_tp, t_m[0].data_ptr(), t_m[1].data_ptr(), stream)), 8)
    report("highlights_clip", lambda: ab.check(L.b200_highlights_process_dev(p_hl, t_m[1].data_ptr(), t_m[0].data_ptr(), stream)), 8)
    report("rawfront_fused_uint16", lambda: ab.check(L.b200_rawfront_process_dev(p_rp, p_tp, p_hl, t_raw.data_ptr(), t_m[0].data_ptr(), stream)), 6)
    report("exposure", lambda: ab.check(L.b200_exposure_process_dev(p_ex, t_rgba.data_ptr(), t_out.data_ptr(), stream)), 32)
    report("gamma_uint8", lambda: ab.check(L.b200_gamma_process_dev(p_gm, t_rgba.data_ptr(), t_u8.data_ptr(), stream)), 20)
    report("export_uint16", lambda: ab.check(L.b200_export_convert_dev(t_rgba.data_ptr(), t_out.data_ptr(), w, h, ab.EXPORT_UINT16, stream)), 24)
    report("finalscale_half_mitchell", lambda: ab.check(L.b200_finalscale_process_dev(p_fs, t_rgba.data_ptr(), t_out.data_ptr(), stream)), 20)

    # the demosaicers, colour calibration, the bilateral grid and highlight inpainting added with them
    t_dem = torch.empty((h, w, 4), dtype=torch.float32, device=dev)
    for label, method in (("demosaic_ppg_median", ab.DEMOSAIC_PPG), ("demosaic_vng4", ab.DEMOSAIC_VNG4), ("demosaic_rcd_dual_vng4", ab.DEMOSAIC_RCD | 2048)):
        dd = ab.demosaic_data(method)
        dd.median_thrs, dd.dual_thrs = 0.02, 0.2
        p_d = piece(dd, 1)
        report(label, lambda: ab.check(L.b200_demosaic_process_dev(p_d, t_m[0].data_ptr(), t_dem.data_ptr(), stream)), 20, reps=3)
    # the half-size method (algorithmic bytes per INPUT pixel: 4 in + 16 / 4 out), its post-filter, and the X-Trans variant
    hw, hh = (w + 1) // 2, (h + 1) // 2
    for label, smoothing, xtrans in (("demosaic_downsample", 0, False), ("demosaic_downsample_postfilter1", 1, False), ("demosaic_downsample_xtrans", 0, True)):
        dd = ab.demosaic_data(7)
        dd.color_smoothing = smoothing
        p_d = piece(dd, 1, out=(hw, hh))
        if xtrans:
            p_d.filters = 9
            for i, rowv in enumerate(((1, 1, 0, 1, 1, 2), (1, 1, 2, 1, 1, 0), (2, 0, 1, 0, 2, 1), (1, 1, 2, 1, 1, 0), (1, 1, 0, 1, 1, 2), (0, 2, 1, 2, 0, 1))):
                for j, v in enumerate(rowv):
                    p_d.xtrans[i][j] = v
        report(label, lambda: ab.check(L.b200_demosaic_process_dev(p_d, t_m[0].data_ptr(), t_dem.data_ptr(), stream)), 8, reps=3)
    cp = ab.channelmixer_piece(util.profile_pair(util.REC2020_TO_XYZ_D50), illuminant=(0.93, 1.02, 0.71))
    p_cm = piece(None, 4)
    p_cm.data, p_cm.data_size = C.addressof(cp), C.sizeof(cp)
    report("channelmixerrgb_cat16_v3", lambda: ab.check(L.b200_channelmixerrgb_process_dev(p_cm, t_rgba.data_ptr(), t_out.data_ptr(), stream)), 32)
    t_lab = t_rgba * torch.tensor([100.0, 60.0, 60.0, 1.0], device=dev)
    p_bl = piece(ab.bilat_data(sigma_r=5.0, sigma_s=50.0, detail=0.5, mode=0), 4)
    report("bilat_bilateral_grid_sigma50", lambda: ab.check(L.b200_bilat_process_dev(p_bl, t_lab.data_ptr(), t_out.data_ptr(), stream)), 32, reps=3)
    p_hi = piece(ab.highlights_data(ab.HIGHLIGHTS_INPAINT, 1.0), 1, pmax=pm)
    report("highlights_inpaint", lambda: ab.check(L.b200_highlights_process_dev(p_hi, t_m[1].data_ptr(), t_m[0].data_ptr(), stream)), 8, reps=3)
    hd = ab.highlights_data(ab.HIGHLIGHTS_LAPLACIAN, 1.0)     # iop/highlights/common.h:466-468: 30 iterations, diameter parameter 8
    hd.iterations, hd.scales = 30, 8
    p_hg = piece(hd, 1, pmax=pm)
    report("highlights_guided_laplacians_30it", lambda: ab.check(L.b200_highlights_process_dev(p_hg, t_m[1].data_ptr(), t_m[0].data_ptr(), stream)), 8, reps=3)
    p_lm = piece(ab.demosaic_data(6), 1, pmax=pm)
    C.cast(p_lm.data, C.POINTER(ab.DemosaicData)).contents.lmmse_refine = 1
    report("demosaic_lmmse_median", lambda: ab.check(L.b200_demosaic_process_dev(p_lm, t_m[0].data_ptr(), t_dem.data_ptr(), stream)), 20, reps=3)
    # X-Trans: Markesteijn with one pass (the default demosaicer of X-Trans frames)
    p_mk = piece(ab.demosaic_data(1025), 1)
    p_mk.filters = 9
    for i, rowv in enumerate(((1, 1, 0, 1, 1, 2), (1, 1, 2, 1, 1, 0), (2, 0, 1, 0, 2, 1), (1, 1, 2, 1, 1, 0), (1, 1, 0, 1, 1, 2), (0, 2, 1, 2, 0, 1))):
        for j, v in enumerate(rowv):
            p_mk.xtrans[i][j] = v
    report("demosaic_markesteijn_1pass_xtrans", lambda: ab.check(L.b200_demosaic_process_dev(p_mk, t_m[0].data_ptr(), t_dem.data_ptr(), stream)), 20, reps=3)
    # blending of a module's output over its input: parametric mask on two channels + a drawn mask, one fused pass (52 B/px: in, out, form mask in; out)
    try:
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import blend_util as bu
        bp = bu.params(mode="normal", opacity=70.0, mask_mode=bu.MASK_ENABLED | bu.MASK_SHAPE | bu.MASK_PARAMETRIC, drawn=1,
                       channels={0: (0.05, 0.2, 0.8, 1.0), 5: (0.0, 0.0, 0.7, 0.9)})
        t_form = torch.rand((h, w), dtype=torch.float32, device=dev)
        p_b = piece(None, 4)
        L.b200_blend_process_dev.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        report("blend_rgb_scene_drawn_and_parametric",
               lambda: ab.check(L.b200_blend_process_dev(C.byref(p_b), C.byref(bp), t_rgba.data_ptr(), t_out.data_ptr(), t_form.data_ptr(), None, stream)), 52)
        # the same in Lab (what local contrast blends in): the overlay operator under a mask on lightness, chroma and hue of the input
        bl = bu.params(cst=bu.CS_LAB, mode="overlay", opacity=70.0, mask_mode=bu.MASK_ENABLED | bu.MASK_SHAPE | bu.MASK_PARAMETRIC, drawn=1,
                       channels={0: (0.05, 0.2, 0.8, 1.0), 8: (0.02, 0.1, 0.6, 0.8), 9: (0.1, 0.2, 0.7, 0.8)})
        report("blend_lab_overlay_drawn_and_parametric_lch",
               lambda: ab.check(L.b200_blend_process_dev(C.byref(p_b), C.byref(bl), t_lab.data_ptr(), t_out.data_ptr(), t_form.data_ptr(), None, stream)), 52)
        # and with the Jz / Cz / hz channels of the RGB space (the PQ curve twice per channel, atan2f, hypotf per pixel of input and output)
        bj = bu.params(mode="normal", opacity=70.0, mask_mode=bu.MASK_ENABLED | bu.MASK_PARAMETRIC,
                       channels={8: (0.002, 0.006, 0.015, 0.02), 14: (0.1, 0.2, 0.7, 0.85)})
        report("blend_rgb_scene_parametric_jzczhz",
               lambda: ab.check(L.b200_blend_process_dev(C.byref(p_b), C.byref(bj), t_rgba.data_ptr(), t_out.data_ptr(), None, None, stream)), 48)
    except Exception as e:
        res.setdefault("blend_rgb_scene_drawn_and_parametric", {"unavailable": f"{type(e).__name__}: {e}"[:200]})
    try:   # colour inpainting on an X-Trans mosaic (the Bayer one is `highlights_inpaint` above)
        p_hx = piece(ab.highlights_data(ab.HIGHLIGHTS_INPAINT, 1.0), 1, pmax=pm)
        p_hx.filters = 9
        for i, rowv in enumerate(((1, 1, 0, 1, 1, 2), (1, 1, 2, 1, 1, 0), (2, 0, 1, 0, 2, 1), (1, 1, 2, 1, 1, 0), (1, 1, 0, 1, 1, 2), (0, 2, 1, 2, 0, 1))):
            for j, v in enumerate(rowv):
                p_hx.xtrans[i][j] = v
        report("highlights_inpaint_xtrans", lambda: ab.check(L.b200_highlights_process_dev(p_hx, t_m[1].data_ptr(), t_m[0].data_ptr(), stream)), 8, reps=3)
    except Exception as e:
        res["highlights_inpaint_xtrans"] = {"unavailable": f"{type(e).__name__}: {e}"[:200]}

    # sensor-to-display chain, end to end
    try:
        order = [("rawprepare", d_rp, 1, 1, 2, 1, (1.0,) * 4), ("temperature", d_tp, 1, 1, 1, 1, (1.0,) * 4), ("highlights", d_hl, 1, 1, 1, 1, pm),
                 ("demosaic", d_dem, 1, 4, 1, 1, pm), ("colorin", d_cin, 4, 4, 1, 1, pm), ("colorout", d_cout, 4, 4, 1, 1, pm), ("gamma", None, 4, 4, 1, 3, pm)]
        pieces = [ds.make_piece_iop(op, w, h, data, channels_in=ci, channels_out=co, filters=filters, processed_maximum=pmx, wb=wb, type_in=ti, type_out=to)
                  for op, data, ci, co, ti, to, pmx in order]
        nodes = (ds.PipeNode * len(order))()
        for k, (op, *_rest) in enumerate(order):
            nodes[k].process_cl = C.cast(getattr(M, f"dt_iop_{op}__process_cl"), C.c_void_p)
            nodes[k].module = pieces[k].module
            nodes[k].piece = C.pointer(pieces[k])
        pipe = ds.make_pipe(devid=local, stream=None)
        DEPTH, steps = 2, 12
        queue = M.b200_pipe_queue_new(DEPTH)
        try:
            h_in = torch.from_numpy(raw).pin_memory()
            h_out = [torch.zeros((h, w, 4), dtype=torch.uint8).pin_memory() for _ in range(DEPTH)]

            def run(n):
                tickets = []
                for i in range(n):
                    t = M.b200_pixelpipe_submit(queue, C.byref(pipe), nodes, len(order), h_in.data_ptr(), h_out[i % DEPTH].data_ptr())
                    if t < 0:
                        raise RuntimeError("chain failed: " + L.b200_last_error().decode())
                    tickets.append(t)
                    if i >= DEPTH - 1 and M.b200_pixelpipe_wait(queue, tickets[i - DEPTH + 1]) != 0:
                        raise RuntimeError("wait failed: " + L.b200_last_error().decode())
                if M.b200_pixelpipe_wait(queue, tickets[-1]) != 0:
                    raise RuntimeError("wait failed: " + L.b200_last_error().decode())

            run(3)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            run(steps)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
        finally:
            M.b200_pipe_queue_free(queue)
        res["sensor_to_display_e2e"] = {"value": npx * steps / dt / 1e6, "unit": UNIT, "steps": steps, "h2d_bytes_per_step": 2 * npx, "d2h_bytes_per_step": 4 * npx,
                                        "chain": "rawprepare(uint16) -> temperature -> highlights(clip) -> demosaic(RCD) -> colorin -> colorout -> gamma(uint8)",
                                        "path": "dt_iop_<op>__process_cl adapters via b200_pixelpipe_submit/_wait (the raw front fused into one launch by the pipe glue), 2 frames in flight, pinned host buffers",
                                        "mean_display_value": float(h_out[0][..., :3].float().mean())}
    except Exception as e:
        res["sensor_to_display_e2e"] = {"unavailable": f"{type(e).__name__}: {e}"[:300]}
    return res


def pipe_ends_in_child(w, h, local):
    """pipe_ends_extras() in a child process with a time limit: its kernels were written after round 1's GPU budget was spent, so a
    crash or a hang there must not cost the benchmark line.  Reported, never fatal."""
    import subprocess
    cmd = [sys.executable, os.path.abspath(__file__), "--pipe-ends-only", "--width", str(w), "--height", str(h)]
    env = dict(os.environ, LOCAL_RANK=str(local), WORLD_SIZE="1", RANK="0")
    try:
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=240, env=env)
    except subprocess.TimeoutExpired:
        return {"unavailable": "child process exceeded 240 s"}
    for line in reversed(r.stdout.strip().splitlines()):
        if line.startswith("{"):
            try:
                return json.loads(line)
            except Exception:
                break
    return {"unavailable": f"child exit {r.returncode}: {(r.stderr or r.stdout).strip()[-300:]}"}


def run_pipe_ends_only(args):
    import torch
    import ansel_b200 as ab
    import ansel_b200.dtsurface as ds
    import util
    local = int(os.environ.get("LOCAL_RANK", "0"))
    try:
        if not torch.cuda.is_available():
            raise RuntimeError("no CUDA device")
        torch.cuda.set_device(local)
        ab.init()
        L, M = ab.lib(), ds.modlib()
        enc = util.srgb_encode_lut()
        co_t = np.zeros((3, 3), np.float32)
        L.b200_fit_unbounded_coeffs((C.c_void_p * 3)(*[enc[k].ctypes.data for k in range(3)]), co_t.ctypes.data)
        conv_in = ab.make_conversion(util.MATRIX_CAM_TO_REC2020, identity=0x2001)
        conv_out = ab.make_conversion(util.MATRIX_REC2020_TO_SRGB, lut_target=enc, coeffs_target=co_t, identity=0x2002)
        res = pipe_ends_extras(ab, ds, util, L, M, torch, args.width, args.height, local, torch.device("cuda", local), torch.cuda.current_stream().cuda_stream,
                               conv_in, conv_out, ab.colorin_data(conv_in), ab.colorout_data(conv_out))
    except Exception as e:
        res = {"unavailable": f"{type(e).__name__}: {e}"[:300]}
    print(json.dumps(res))


def bind_near_gpu(local):
    """N > 1: run this rank (and allocate its pinned host buffers: first touch) on the CPUs of the GPU's NUMA node.  Returns a note."""
    try:
        import pynvml
        pynvml.nvmlInit()
        bus = pynvml.nvmlDeviceGetPciInfo(pynvml.nvmlDeviceGetHandleByIndex(local)).busId
        bus = (bus.decode() if isinstance(bus, bytes) else bus).lower()
        if len(bus.split(":")[0]) == 8:
            bus = bus[4:]
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read())
        if node < 0:
            return "no NUMA node reported for the GPU"
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return f"NUMA node {node}: no allowed CPU"
        os.sched_setaffinity(0, cpus)
        return f"NUMA node {node}, {len(cpus)} CPUs"
    except Exception as e:  # affinity is an optimisation, never a requirement
        return f"unbound ({type(e).__name__})"


class DeviceChain:
    """a chain of modules on device-resident buffers through the C ABI (b200_<op>_process_dev), per-module CUDA events on request"""

    def __init__(self, ab, torch, ops, w, h, dev, stream):
        self.ab, self.torch, self.ops, self.stream = ab, torch, ops, stream
        self.L = ab.lib()
        self.bufs = [torch.empty((h, w, 4), dtype=torch.float32, device=dev) for _ in range(2)]
        self.fns = [getattr(self.L, f"b200_{op}_process_dev") for op, _ in ops]

    def step(self, src, record=False):
        torch, ab = self.torch, self.ab
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(len(self.ops) + 1)] if record else None
        cur = src
        for k, ((op, piece), fn) in enumerate(zip(self.ops, self.fns)):
            if record:
                evs[k].record()
            dst = self.bufs[k & 1]
            ab.check(fn(piece, cur.data_ptr(), dst.data_ptr(), self.stream))
            cur = dst
        if record:
            evs[-1].record()
        self.out = cur
        return evs


def run_b200(args):
    import torch
    import torch.distributed as dist
    import ansel_b200 as ab
    import ansel_b200.dtsurface as ds
    import util

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the B200 path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    numa = bind_near_gpu(local) if world > 1 else "single rank: all host CPUs (the CPU baseline runs on them)"
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    ab.init()
    L = ab.lib()
    L.b200_kernel_timing_read.argtypes = [C.c_char_p, C.POINTER(C.c_double), C.POINTER(C.c_int)]
    w, h = args.width, args.height
    npx = w * h

    mosaic = util.frame_natural(w, h, SEED + rank)
    filters = util.BAYER["RGGB"]
    enc = util.srgb_encode_lut()
    co_t = np.zeros((3, 3), np.float32)
    lut_ptrs = (C.c_void_p * 3)(*[enc[k].ctypes.data for k in range(3)])
    L.b200_fit_unbounded_coeffs(lut_ptrs, co_t.ctypes.data)
    conv_in = ab.make_conversion(util.MATRIX_CAM_TO_REC2020, identity=0x1001)
    conv_out = ab.make_conversion(util.MATRIX_REC2020_TO_SRGB, lut_target=enc, coeffs_target=co_t, identity=0x1002)
    work, export = util.profile_pair(util.REC2020_TO_XYZ_D50), util.profile_pair(util.SRGB_TO_XYZ_D50)
    fblob = np.ascontiguousarray(np.load(os.path.join(util.GOLDEN_DIR, "filmic_data.npz"))["default_v8"], np.uint8)
    d_dem, d_cin, d_cout = ab.demosaic_data(ab.DEMOSAIC_RCD), ab.colorin_data(conv_in), ab.colorout_data(conv_out)
    d_dn = ab.denoiseprofile_data(ab.DENOISE_NLMEANS, radius=1, nbhood=7)
    d_fp = ab.filmic_piece(fblob, work, export)

    def piece_of(data, ch):
        p = ab.make_piece(w, h, filters=filters if ch == 1 else 0, channels=ch, devid=local)
        p.data, p.data_size = C.addressof(data), C.sizeof(data)
        return p

    dev = torch.device("cuda", local)
    stream = torch.cuda.current_stream().cuda_stream
    t_mosaic = torch.from_numpy(mosaic).to(dev)
    c3 = DeviceChain(ab, torch, [("demosaic", piece_of(d_dem, 1)), ("denoiseprofile", piece_of(d_dn, 4)), ("colorin", piece_of(d_cin, 4)),
                                 ("filmicrgb", piece_of(d_fp, 4))], w, h, dev, stream)
    c2 = DeviceChain(ab, torch, [("demosaic", piece_of(d_dem, 1)), ("colorin", piece_of(d_cin, 4)), ("colorout", piece_of(d_cout, 4))], w, h, dev, stream)
    c2.bufs = c3.bufs                       # the two chains never run at the same time
    # kernels per step: rcd_ring + rcd_tiles | vst_forward + nlm_group + vst_backward | convert | filmic_agx
    LAUNCHES_C3 = 2 + 3 + 1 + 1

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed_steps(chain, steps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        all_evs = [chain.step(t_mosaic, record=True) for _ in range(steps)]
        e1.record()
        barrier()
        t_ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t_ms, op=dist.ReduceOp.MAX)
        mod = {op: float(np.mean([evs[k].elapsed_time(evs[k + 1]) for evs in all_evs])) for k, (op, _) in enumerate(chain.ops)}
        return float(t_ms.item()), mod

    for _ in range(max(args.warmup, 3)):
        c3.step(t_mosaic)
    barrier()

    # ---- timed region: exactly K steps, device-resident, the two headline kernels bracketed by events on their stream ----
    L.b200_kernel_timing(1)
    with ClockSampler(local) as clk:
        ms_max, mod_ms = timed_steps(c3, args.steps)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, c3.out)
    ksum, kcnt = C.c_double(), C.c_int()
    kernel_ms = {}
    for name in ("nlm_kernel", "rcd_tiles_kernel"):
        ab.check(L.b200_kernel_timing_read(name.encode(), C.byref(ksum), C.byref(kcnt)))
        kernel_ms[name] = (ksum.value / kcnt.value) if kcnt.value else None
    L.b200_kernel_timing(0)
    value = world * npx * args.steps / (ms_max * 1e-3) / 1e6
    gpu_launches = LAUNCHES_C3 * args.steps

    # ---- the lighter chain of configs[1], same frame, for continuity with round 1 --------------------------
    for _ in range(3):
        c2.step(t_mosaic)
    c2_ms, c2_mod = timed_steps(c2, args.steps)
    c2_line = {"workload": WORKLOAD_C2, "value": world * npx * args.steps / (c2_ms * 1e-3) / 1e6, "unit": UNIT, "ms_per_step": c2_ms / args.steps,
               "per_module_ms": c2_mod}

    # ---- e2e: host buffers through the C module adapters + device-resident pipe glue -----------
    M = ds.modlib()
    pipe = ds.make_pipe(devid=local, stream=None, work_profile=ds.profile_info(*work), output_profile=ds.profile_info(*export))
    fdata = (C.c_uint8 * fblob.size).from_buffer_copy(fblob.tobytes())
    chain_ops = [("demosaic", d_dem, 1), ("denoiseprofile", d_dn, 4), ("colorin", d_cin, 4), ("filmicrgb", fdata, 4)]
    pieces = [ds.make_piece_iop(op, w, h, data, channels_in=ch, channels_out=4, filters=filters if ch == 1 else 0, wb=WB) for op, data, ch in chain_ops]
    nodes = (ds.PipeNode * len(chain_ops))()
    for k, (op, _d, _c) in enumerate(chain_ops):
        nodes[k].process_cl = C.cast(getattr(M, f"dt_iop_{op}__process_cl"), C.c_void_p)
        nodes[k].module = pieces[k].module
        nodes[k].piece = C.pointer(pieces[k])
    # two frames in flight (b200_pixelpipe_submit/_wait): the read-back of frame n overlaps upload + compute of
    # frame n+1.  Every step still uploads its own input and reads its own result back inside the timed region.
    DEPTH = 2
    queue = M.b200_pipe_queue_new(DEPTH)
    h_in = torch.from_numpy(mosaic).pin_memory()
    h_out = [torch.empty((h, w, 4), dtype=torch.float32).pin_memory() for _ in range(DEPTH)]

    def e2e_run(n):
        tickets = []
        for i in range(n):
            t = M.b200_pixelpipe_submit(queue, C.byref(pipe), nodes, len(chain_ops), h_in.data_ptr(), h_out[i % DEPTH].data_ptr())
            if t < 0:
                raise RuntimeError("e2e chain failed: " + L.b200_last_error().decode())
            tickets.append(t)
            if i >= DEPTH - 1:                      # the consumer takes frame i-DEPTH+1 before its buffer is reused
                if M.b200_pixelpipe_wait(queue, tickets[i - DEPTH + 1]) != 0:
                    raise RuntimeError("e2e wait failed: " + L.b200_last_error().decode())
        for t in tickets[-(DEPTH - 1):] if DEPTH > 1 else []:
            if M.b200_pixelpipe_wait(queue, t) != 0:
                raise RuntimeError("e2e wait failed: " + L.b200_last_error().decode())

    e2e_run(3)
    barrier()
    t0 = time.perf_counter()
    e2e_run(args.e2e_steps)
    barrier()
    e2e_s = time.perf_counter() - t0
    # the adapters must give what the ABI chain gives
    e2e_same = bool(torch.equal(h_out[(args.e2e_steps - 1) % DEPTH].to(dev).view(torch.int32), c3_out_bits(c3, t_mosaic, torch)))
    # the synchronous single-frame call, for reference (one frame at a time: upload, chain, read back)
    bufs = M.b200_pipe_buffers_new()
    for _ in range(2):
        M.b200_pixelpipe_process_on_gpu(C.byref(pipe), nodes, len(chain_ops), bufs, h_in.data_ptr(), h_out[0].data_ptr())
    t1 = time.perf_counter()
    for _ in range(4):
        if M.b200_pixelpipe_process_on_gpu(C.byref(pipe), nodes, len(chain_ops), bufs, h_in.data_ptr(), h_out[0].data_ptr()) != 0:
            raise RuntimeError("e2e chain failed: " + L.b200_last_error().decode())
    e2e_sync_ms = (time.perf_counter() - t1) / 4 * 1e3
    M.b200_pipe_buffers_free(bufs)
    t_e = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t_e, op=dist.ReduceOp.MAX)
    e2e_value = world * npx * args.e2e_steps / float(t_e.item()) / 1e6
    M.b200_pipe_queue_free(queue)
    del h_out

    # ---- C5: the batch export, frames dealt to the ranks ---------------------------------------------------
    batch = None
    if not args.no_batch:
        try:
            batch = batch_export(ab, ds, util, L, M, torch, dist, world, rank, local, w, h, barrier,
                                 dict(dem=d_dem, dn=d_dn, cin=d_cin, cout=d_cout, fdata=fdata, work_info=ds.profile_info(*work), export_info=ds.profile_info(*export)))
        except Exception as e:
            batch = {"unavailable": f"{type(e).__name__}: {e}"[:300]}

    # ---- the other modules of SURVEY.md 8a at the same frame size (outside the timed region; N=1 only) ----
    other = None
    t_rgb = c3.bufs
    if world == 1 and not args.no_other_modules:
        other = {}
        cases = [("denoiseprofile_wavelets", "denoiseprofile", ab.denoiseprofile_data(ab.DENOISE_WAVELETS), 2),
                 ("diffuse_sharpen_demosaic_1it_5scales", "diffuse", ab.diffuse_data(**ab.DIFFUSE_PRESETS["sharpen_demosaic_aa"]), 2),
                 ("bilat_local_laplacian", "bilat", ab.bilat_data(), 2)]
        t_rgb[0].copy_(torch.rand((h, w, 4), device=dev))
        for label, op, data, reps in cases:
            pc = piece_of(data, 4)
            fn = getattr(L, f"b200_{op}_process_dev")
            ab.check(fn(pc, t_rgb[0].data_ptr(), t_rgb[1].data_ptr(), stream))
            torch.cuda.synchronize()
            ts = []
            for _ in range(reps):
                a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a0.record()
                ab.check(fn(pc, t_rgb[0].data_ptr(), t_rgb[1].data_ptr(), stream))
                a1.record()
                torch.cuda.synchronize()
                ts.append(a0.elapsed_time(a1))
            m = float(np.median(ts))
            other[label] = {"ms": m, "MP_per_s": npx / m / 1e3, "algorithmic_GBps": 32 * npx / (m * 1e-3) / 1e9}
        # the second demosaicer of the north star on the bench frame (20 B/px at the module boundary)
        d_amz = ab.demosaic_data(ab.DEMOSAIC_AMAZE)   # the piece points at it: keep it alive
        p_amz = piece_of(d_amz, 1)
        ts = []
        for k in range(4):
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a0.record()
            ab.check(L.b200_demosaic_process_dev(p_amz, t_mosaic.data_ptr(), t_rgb[1].data_ptr(), stream))
            a1.record()
            torch.cuda.synchronize()
            if k:
                ts.append(a0.elapsed_time(a1))
        m = float(np.median(ts))
        other["demosaic_amaze"] = {"ms": m, "MP_per_s": npx / m / 1e3, "algorithmic_GBps": 20 * npx / (m * 1e-3) / 1e9}

        # the modules either side of the path (SURVEY.md 8f) and the sensor-to-display chain; never part of the headline
        other["pipe_ends"] = pipe_ends_in_child(w, h, local)

    # ---- second mode at N>1 (SURVEY.md 8e / C5): ONE frame cut into row bands + one all-gather ---------
    banded = None
    if world > 1:
        del c2_mod
        torch.cuda.empty_cache()
        banded = banded_modes(args, ab, util, torch, dist, world, rank, dev, stream, w, h, npx, barrier,
                              dict(dem=d_dem, dn=d_dn, cin=d_cin, cout=d_cout, fp=d_fp), c3, c2)

    # ---- roofline of the dominant kernel (non-local means) and of RCD ------------------------------------
    peak, peak_src = peaks()
    nlm_ms = kernel_ms["nlm_kernel"]
    traffic = {}
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath):
        try:
            traffic = json.load(open(tpath))
        except Exception:
            traffic = {}
    per_module = {k: {"ms": v, "algorithmic_GBps": ALGO_BYTES_PER_PX[k] * npx / (v * 1e-3) / 1e9,
                      "frac_of_hbm_peak": ALGO_BYTES_PER_PX[k] * npx / (v * 1e-3) / 1e9 / peak} for k, v in mod_ms.items()}
    chain_bytes = sum(ALGO_BYTES_PER_PX[k] for k in mod_ms)
    roof = None
    if nlm_ms:
        achieved = ALGO_BYTES_PER_PX["denoiseprofile"] * npx / (nlm_ms * 1e-3) / 1e9
        flops = NLM_FLOP_PER_PX_PATCH * 225 * npx / (nlm_ms * 1e-3) / 1e12
        roof = {"bound": "hbm", "kernel": "nlm_pipe_kernel (non-local means, 225 patches; the vst kernels either side are < 2% of the module)",
                "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic.get("nlm_pipe_kernel_dram_bytes_per_launch"),
                "peak_source": peak_src, "algorithmic_bytes_per_launch": ALGO_BYTES_PER_PX["denoiseprofile"] * npx, "avg_launch_ms": nlm_ms,
                "launches_timed": args.steps, "share_of_step": nlm_ms / (ms_max / args.steps),
                "fp32": {"achieved_tflops": flops, "peak_tflops": FP32_PEAK_TFLOPS, "frac": flops / FP32_PEAK_TFLOPS,
                         "flop_per_pixel": NLM_FLOP_PER_PX_PATCH * 225,
                         "note": "the kernel is arithmetic-bound by construction (8.7 kflop per pixel against 32 B): the FP32 fraction is the meaningful one; "
                                 "peak = one packed FP32 instruction per scheduler and clock at 1965 MHz, unfused (bit parity forbids FMA contraction)"},
                "chain": {"algorithmic_bytes_per_px": chain_bytes, "achieved_GBps": chain_bytes * npx / (ms_max / args.steps * 1e-3) / 1e9,
                          "frac": chain_bytes * npx / (ms_max / args.steps * 1e-3) / 1e9 / peak},
                "rcd_tiles_kernel": None if not kernel_ms["rcd_tiles_kernel"] else {
                    "avg_launch_ms": kernel_ms["rcd_tiles_kernel"], "achieved": ALGO_BYTES_PER_PX["demosaic"] * npx / (kernel_ms["rcd_tiles_kernel"] * 1e-3) / 1e9,
                    "frac": ALGO_BYTES_PER_PX["demosaic"] * npx / (kernel_ms["rcd_tiles_kernel"] * 1e-3) / 1e9 / peak,
                    "traffic": traffic.get("rcd_tiles_kernel_dram_bytes_per_launch")}}

    # ---- CPU baseline, rank 0 at N=1 only, bounded sample ---------------------------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        rows, per_row = cpu_sample_rows(w, h, 20.0, 4)
        chain = CpuChain(w, rows)
        ts = time_cpu(chain, mosaic[:rows].copy(), 1, 3)
        cpu = {"value": w * rows / float(np.median(ts)) / 1e6, "unit": UNIT, "cores": _CPU_THREADS, "kind": chain.kind,
               "sample": f"3 steps after 1 warm-up (median), each the top {rows} rows of the {w}x{h} frame through the same chain, "
                         f"{'reference sources, release flags, ' if chain.kind == 'reference' else 'oracle port, '}OpenMP, {_CPU_THREADS} threads "
                         f"(one per physical core), OMP_PROC_BIND={os.environ.get('OMP_PROC_BIND')}"}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms_max / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "frame": f"{w}x{h}", "frames_per_step": world,
                       "parallelism": f"{world} independent frame replicas, no data-path collective",
                       "l2": "inputs larger than L2: 182 MB mosaic + 2 x 727 MB RGBA ping-pong per step vs 126 MB L2",
                       "fp": "C-standard float semantics (no contraction) = the strict build of the reference's sources; colorin: the release build's contraction",
                       "per_module": per_module, "host_binding": numa, "c2": c2_line},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": 4 * npx, "d2h_bytes_per_step": 16 * npx,
                    "steps": args.e2e_steps,
                    "path": "dt_iop_<op>__process_cl adapters via b200_pixelpipe_submit/_wait, 2 frames in flight, pinned host buffers",
                    "single_frame_sync_ms": e2e_sync_ms, "bit_identical_to_the_abi_chain": e2e_same},
            "gpu_launches": gpu_launches,
            "clocks": clk.summary(),
            "roofline": roof,
        }
        if cpu is not None:
            line["cpu_baseline"] = cpu
        if other is not None:
            line["config"]["other_modules_45mp"] = other
        if banded is not None:
            line["banded_one_frame"] = banded
        if batch is not None:
            line["batch_export_c5"] = batch
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def batch_export(ab, ds, util, L, M, torch, dist, world, rank, local, w, h, barrier, datas, n_frames=64):
    """BASELINE.json configs[4] ("C5"): a batch of 64 x 45 MP frames through the full export pipe -- uint16 sensor data up, uint8 display
    pixels down: rawprepare -> temperature -> highlights(clip) -> demosaic(RCD) -> denoiseprofile(NLM) -> colorin -> filmicrgb ->
    colorout -> gamma -- the frames dealt to the ranks (64 / N each), every frame through the C module adapters and the device-resident
    pipe glue with two frames in flight.  Frames are independent: no collective moves pixels."""
    npx = w * h
    wb = (2.13, 1.0, 1.57, 1.02)
    pm = (wb[0], wb[1], wb[2], 0.0)
    filters = util.BAYER["RGGB"]
    sub, div = (512.0, 520.0, 508.0, 515.0), (15871.0, 15863.0, 15875.0, 15868.0)
    rng = np.random.default_rng(SEED + rank)
    raw = np.clip(util.frame_natural(w, h, SEED + rank) * 15871.0 * 0.45 + 512.0 + rng.normal(0, 3, (h, w)), 0, 16383).astype(np.uint16)
    raw[rng.integers(0, h, 4000), rng.integers(0, w, 4000)] = 16383
    d_rp, d_tp, d_hl = ab.rawprepare_data(sub, div), ab.temperature_data(wb), ab.highlights_data(ab.HIGHLIGHTS_CLIP, 1.0)
    order = [("rawprepare", d_rp, 1, 1, 2, 1, (1.0,) * 4), ("temperature", d_tp, 1, 1, 1, 1, (1.0,) * 4), ("highlights", d_hl, 1, 1, 1, 1, pm),
             ("demosaic", datas["dem"], 1, 4, 1, 1, pm), ("denoiseprofile", datas["dn"], 4, 4, 1, 1, pm), ("colorin", datas["cin"], 4, 4, 1, 1, pm),
             ("filmicrgb", datas["fdata"], 4, 4, 1, 1, pm), ("colorout", datas["cout"], 4, 4, 1, 1, pm), ("gamma", None, 4, 4, 1, 3, pm)]
    pieces = [ds.make_piece_iop(op, w, h, data, channels_in=ci, channels_out=co, filters=filters, processed_maximum=pmx, wb=wb, type_in=ti, type_out=to)
              for op, data, ci, co, ti, to, pmx in order]
    nodes = (ds.PipeNode * len(order))()
    for k, (op, *_rest) in enumerate(order):
        nodes[k].process_cl = C.cast(getattr(M, f"dt_iop_{op}__process_cl"), C.c_void_p)
        nodes[k].module = pieces[k].module
        nodes[k].piece = C.pointer(pieces[k])
    pipe = ds.make_pipe(devid=local, stream=None, work_profile=datas["work_info"], output_profile=datas["export_info"])
    DEPTH = 2
    mine = n_frames // world + (1 if rank < n_frames % world else 0)
    queue = M.b200_pipe_queue_new(DEPTH)
    try:
        h_in = torch.from_numpy(raw).pin_memory()
        h_out = [torch.zeros((h, w, 4), dtype=torch.uint8).pin_memory() for _ in range(DEPTH)]

        def run(n):
            tickets = []
            for i in range(n):
                t = M.b200_pixelpipe_submit(queue, C.byref(pipe), nodes, len(order), h_in.data_ptr(), h_out[i % DEPTH].data_ptr())
                if t < 0:
                    raise RuntimeError("chain failed: " + L.b200_last_error().decode())
                tickets.append(t)
                if i >= DEPTH - 1 and M.b200_pixelpipe_wait(queue, tickets[i - DEPTH + 1]) != 0:
                    raise RuntimeError("wait failed: " + L.b200_last_error().decode())
            if tickets and M.b200_pixelpipe_wait(queue, tickets[-1]) != 0:
                raise RuntimeError("wait failed: " + L.b200_last_error().decode())

        run(2)
        barrier()
        t0 = time.perf_counter()
        run(mine)
        barrier()
        dt = time.perf_counter() - t0
        mean = float(h_out[0][..., :3].float().mean())
    finally:
        M.b200_pipe_queue_free(queue)
    t_e = torch.tensor([dt], dtype=torch.float64, device=torch.device("cuda", local))
    if world > 1:
        dist.all_reduce(t_e, op=dist.ReduceOp.MAX)
    dt = float(t_e.item())
    return {"workload": "C5: 64 x 45MP frames, full export pipe: rawprepare(uint16) -> temperature -> highlights(clip) -> demosaic(RCD) -> "
                        "denoiseprofile(NLM P=1 K=7) -> colorin -> filmicrgb -> colorout -> gamma(uint8)",
            "value": npx * n_frames / dt / 1e6, "unit": UNIT, "frames": n_frames, "frames_per_rank": mine, "seconds": dt,
            "h2d_bytes_per_frame": 2 * npx, "d2h_bytes_per_frame": 4 * npx,
            "path": "dt_iop_<op>__process_cl adapters via b200_pixelpipe_submit/_wait (raw front fused by the pipe glue), 2 frames in flight per rank, pinned host buffers",
            "collective": "none: frames are independent (SURVEY.md 8e); one frame over several GPUs is `banded_one_frame`",
            "mean_display_value": mean}


def c4_mode(args, ab, util, torch, dist, world, rank, dev, stream, barrier, d):
    """C4: 100 MP Bayer (11648x8736) -> demosaic(RCD) -> denoiseprofile(NLM) -> colorin -> diffuse(sharpen) -> filmicrgb -> [RGB->Lab]
    bilat(local Laplacian) [Lab->RGB] -> colorout, ONE frame over the ranks (ansel_b200/bands.py SegmentedChain): two banded segments
    around the local Laplacian, which runs on the whole frame on every rank after an all-gather (its pyramid reaches across the
    frame; the reference refuses to tile it: bilat.c:310-311)."""
    from ansel_b200 import bands
    w, h = 11648, 8736
    npx = w * h
    frame0 = util.frame_natural(w, h, SEED)
    work = util.profile_pair(util.REC2020_TO_XYZ_D50)
    pm = ab.profile_matrices(*work)
    dd = ab.diffuse_data(**ab.DIFFUSE_PRESETS["sharpen_demosaic_aa"])
    nodes = [bands.Node("demosaic", d["dem"], channels_in=1), bands.Node("denoiseprofile", d["dn"]), bands.Node("colorin", d["cin"]),
             bands.Node("diffuse", dd), bands.Node("filmicrgb", d["fp"]), bands.Node("colorspace", (ab.CS_RGB, ab.CS_LAB, pm)),
             bands.Node("bilat", ab.bilat_data()), bands.Node("colorspace", (ab.CS_LAB, ab.CS_RGB, pm)), bands.Node("colorout", d["cout"])]
    ch = bands.SegmentedChain(nodes, w, h, rank, world, device=dev)
    t_band = torch.from_numpy(np.ascontiguousarray(ch.band_rows(frame0))).to(dev)
    steps = 3
    ch(t_band, stream=stream)
    barrier()
    b0, b1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    b0.record()
    for _ in range(steps):
        frame = ch(t_band, stream=stream)
    b1.record()
    barrier()
    t_b = torch.tensor([b0.elapsed_time(b1) / steps], dtype=torch.float64, device=dev)
    dist.all_reduce(t_b, op=dist.ReduceOp.MAX)
    res = {"workload": "C4: 100MP RGGB Bayer (11648x8736) -> demosaic(RCD) -> denoiseprofile(NLM P=1 K=7) -> colorin -> diffuse(sharpen demosaicing) -> "
                       "filmicrgb -> [RGB->Lab] bilat(local Laplacian) [Lab->RGB] -> colorout",
           "value": npx / (float(t_b.item()) * 1e-3) / 1e6, "unit": UNIT, "ms_per_frame": float(t_b.item()), "n_gpus": world, "scaling": "strong",
           "plan": [list(p) for p in ch.plan], "collectives_per_frame": ch.collectives,
           "collective": "ncclAllGather of the finished RGBA bands, once in front of the whole-frame local Laplacian and once at the end"}
    # rank 0: the same chain untiled on one GPU, for the speed-up and the distance
    stat = torch.zeros(3, dtype=torch.float64, device=dev)
    if rank == 0:
        one = bands.SegmentedChain(nodes, w, h, 0, 1, device=dev)
        t_full = torch.from_numpy(frame0).to(dev)
        one(t_full, stream=stream)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        ref = one(t_full, stream=stream)
        e1.record()
        torch.cuda.synchronize()
        stat[0] = e0.elapsed_time(e1)
        stat[1] = float((frame.view(torch.int32) != ref.view(torch.int32)).sum().item())
        stat[2] = float((frame - ref).abs().nan_to_num(0.0).max().item())
        del one, ref, t_full
    dist.broadcast(stat, 0)
    res.update({"one_gpu_ms_per_frame": float(stat[0].item()), "speedup_over_one_gpu": float(stat[0].item()) / float(t_b.item()),
                "vs_untiled": {"floats_differing": int(stat[1].item()), "max_abs": float(stat[2].item()),
                               "why": "the banded segments are the reference's own tiles (RCD tile grid, NLM chunk grid and the diffuse wavelet borders follow the tile "
                                      "origin); the local Laplacian itself is computed on the whole frame"}})
    return res


def c3_out_bits(chain, t_mosaic, torch):
    chain.step(t_mosaic)
    torch.cuda.synchronize()
    return chain.out.view(torch.int32)


def banded_modes(args, ab, util, torch, dist, world, rank, dev, stream, w, h, npx, barrier, d, c3, c2):
    """ONE frame over the ranks in row bands (ansel_b200/bands.py): the C3 chain (tiling.c-style cuts: halo = the modules' overlaps,
    one all-gather of the finished bands) and the C2 chain (RCD block-grid cuts, bit-identical to the untiled frame; NCCL and the
    gather fused into colorout's stores)."""
    from ansel_b200 import bands
    out = {}
    frame0 = util.frame_natural(w, h, SEED)          # the same frame on every rank
    t_full = torch.from_numpy(frame0).to(dev)

    def timed(chain, t_band, steps):
        for _ in range(3):
            chain(t_band, stream=stream)
        barrier()
        b0, b1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        b0.record()
        for _ in range(steps):
            res = chain(t_band, stream=stream)
        b1.record()
        barrier()
        t_b = torch.tensor([b0.elapsed_time(b1)], dtype=torch.float64, device=dev)
        dist.all_reduce(t_b, op=dist.ReduceOp.MAX)
        return float(t_b.item()) / steps, res

    # C3 in bands
    try:
        nodes3 = [bands.Node("demosaic", d["dem"], channels_in=1), bands.Node("denoiseprofile", d["dn"]), bands.Node("colorin", d["cin"]),
                  bands.Node("filmicrgb", d["fp"])]
        ch = bands.BandedChain(nodes3, w, h, rank, world, device=dev)
        t_band = torch.from_numpy(np.ascontiguousarray(ch.band_rows(frame0))).to(dev)
        ms, frame = timed(ch, t_band, args.steps)
        c3.step(t_full)
        torch.cuda.synchronize()
        diff = (frame - c3.out).abs()
        ndiff = torch.tensor([float((frame.view(torch.int32) != c3.out.view(torch.int32)).sum().item()), float(diff.max().item())], dtype=torch.float64, device=dev)
        dist.all_reduce(ndiff, op=dist.ReduceOp.MAX)
        one_ms = torch.tensor([0.0], dtype=torch.float64, device=dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        c3.step(t_full)
        e1.record()
        torch.cuda.synchronize()
        one_ms[0] = e0.elapsed_time(e1)
        dist.all_reduce(one_ms, op=dist.ReduceOp.MAX)
        out["c3"] = {"workload": WORKLOAD, "value": npx / (ms * 1e-3) / 1e6, "unit": UNIT, "ms_per_frame": ms, "one_gpu_ms_per_frame": float(one_ms.item()),
                     "speedup_over_one_gpu": float(one_ms.item()) / ms, "scaling": "strong",
                     "cuts": f"tiling.c-style full-width tiles, halo {ch.halo} rows = the sum of the modules' tiling_callback overlaps",
                     "collective": ch.collective, "gathered_bytes_per_frame": 16 * npx,
                     "vs_untiled": {"floats_differing": int(ndiff[0].item()), "max_abs": float(ndiff[1].item()),
                                    "why": "the reference's own tiles differ from its untiled frame the same way: RCD's tile grid and the non-local-means "
                                           "chunk grid start at the tile origin (tests/test_bands_gpu.py checks each band against the oracle on the same cuts)"}}
    except Exception as e:
        out["c3"] = {"unavailable": f"{type(e).__name__}: {e}"[:300]}

    # C4: the 100 MP full pipe over the ranks, whole-frame local Laplacian inside (BASELINE.json configs[3] names 4 GPUs)
    if world == 4 or args.c4:
        try:
            out["c4"] = c4_mode(args, ab, util, torch, dist, world, rank, dev, stream, barrier, d)
        except Exception as e:
            out["c4"] = {"unavailable": f"{type(e).__name__}: {e}"[:300]}
        torch.cuda.empty_cache()

    # C2 in bands: NCCL exchange, then the gather fused into colorout
    try:
        nodes2 = [bands.Node("demosaic", d["dem"], channels_in=1), bands.Node("colorin", d["cin"]), bands.Node("colorout", d["cout"])]
        ch = bands.BandedChain(nodes2, w, h, rank, world, device=dev)
        t_band = torch.from_numpy(np.ascontiguousarray(ch.band_rows(frame0))).to(dev)
        ms, frame = timed(ch, t_band, args.steps)
        c2.step(t_full)
        torch.cuda.synchronize()
        same = torch.tensor([int(torch.equal(frame.view(torch.int32), c2.out.view(torch.int32)))], dtype=torch.int32, device=dev)
        dist.all_reduce(same, op=dist.ReduceOp.MIN)
        out["c2"] = {"workload": WORKLOAD_C2, "value": npx / (ms * 1e-3) / 1e6, "unit": UNIT, "ms_per_frame": ms, "collective": ch.collective,
                     "cuts": "RCD 94-row block grid, 9-row halo", "bit_identical_to_untiled": bool(same.item()), "gathered_bytes_per_frame": 16 * npx}
        ref_frame = frame.clone()
        for key, dst in (("fused_p2p", None), ("fused_p2p_gather_to_rank0", 0)):
            try:
                chp = bands.BandedChain(nodes2, w, h, rank, world, device=dev, p2p=True, p2p_dst=dst)
                msp, fr = timed(chp, t_band, args.steps)
                ok = torch.ones(1, dtype=torch.int32, device=dev)
                if fr is not None:
                    ok[0] = int(torch.equal(fr.view(torch.int32), ref_frame.view(torch.int32)))
                dist.all_reduce(ok, op=dist.ReduceOp.MIN)
                chp.close()
                out["c2"][key] = {"value": npx / (msp * 1e-3) / 1e6, "ms_per_frame": msp, "bit_identical_to_collective": bool(ok.item()),
                                  "how": "colorout stores each pixel into the destination frames itself (CUDA IPC peer mappings), then one barrier"}
            except Exception as e:  # no peer access on this box: keep the NCCL number
                out["c2"][key] = {"unavailable": str(e)[:200]}
    except Exception as e:
        out["c2"] = {"unavailable": f"{type(e).__name__}: {e}"[:300]}
    return out


if __name__ == "__main__":
    a = parse()
    if a.pipe_ends_only:
        run_pipe_ends_only(a)
    elif a.impl == "reference":
        run_reference(a)
    else:
        run_b200(a)
