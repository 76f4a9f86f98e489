"""Shared helpers for the parity tests: oracle/_ref loaders, ULP distance, synthetic frames.

The oracle (oracle/liboracle.so) and the compiled reference (oracle/_ref/*.so) are CHECKERS; only
tests/, __graft_entry__.smoke() and bench.py's CPU legs may load them.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")
GOLDEN_DIR = os.path.join(ROOT, "tests", "golden")
FP = C.POINTER(C.c_float)

BAYER = {"RGGB": 0x94949494, "BGGR": 0x16161616, "GRBG": 0x61616161, "GBRG": 0x49494949}
SEEDS = (20260922, 1, 2)

# synthetic frame sizes of SURVEY.md 8
SIZE_24MP = (6000, 4000)
SIZE_45MP = (8256, 5504)
SIZE_100MP = (11648, 8736)


def build_oracle() -> None:
    subprocess.run(["make", "-s", "-C", ORACLE_DIR, "oracle"], check=True)
    if os.path.isdir("/root/reference/src"):
        subprocess.run(["make", "-s", "-C", ORACLE_DIR, "ref"], check=True)


_cache = {}


def oracle() -> C.CDLL:
    if "oracle" not in _cache:
        path = os.path.join(ORACLE_DIR, "liboracle.so")
        if not os.path.exists(path):
            build_oracle()
        _cache["oracle"] = C.CDLL(path)
    return _cache["oracle"]


def ref(kind: str = "strict"):
    """oracle/_ref/libref_{strict,fast}.so or None when it was never built (the reference sources are absent)."""
    key = "ref_" + kind
    if key not in _cache:
        path = os.path.join(ORACLE_DIR, "_ref", f"libref_{kind}.so")
        _cache[key] = C.CDLL(path) if os.path.exists(path) else None
    return _cache[key]


# ---- the reference's outputs, recorded ----------------------------------------------------------------------------------
# oracle/_ref can only be built where the reference sources are.  Every helper that calls into it is wrapped by
# `recorded`: with the library present it runs the reference; without it, it returns what the reference returned for the
# same arguments, read from tests/golden/reference/ (written by tests/golden/make_golden_reference.py).  The arguments are
# fingerprinted by content, so a test whose inputs change no longer finds a recording and fails instead of comparing
# against a stale output.  `candidate` (optional) computes the same outputs with the oracle: the recording then keeps only
# the elements where the reference differs from it plus a SHA-256 of the reference's bytes, and the replay checks that
# digest, so what it returns is bit for bit what the reference returned.
RECORD_DIR = os.path.join(GOLDEN_DIR, "reference")
RECORDING = os.environ.get("B200_RECORD_REFERENCE") == "1"
_records, _recorded_now = {}, {}


def _fingerprint(h, v) -> None:
    if isinstance(v, np.ndarray):
        h.update(f"a{v.dtype.str}{v.shape}".encode())
        h.update(np.ascontiguousarray(v).tobytes())
    elif isinstance(v, (C.Structure, C.Union)):
        h.update(type(v).__name__.encode())
        if isinstance(getattr(v, "_keepalive", None), (C.Structure, C.Union, C.Array)):   # the data a piece points at (ansel_b200.make_piece)
            _fingerprint(h, v._keepalive)
        for field in v._fields_:
            name, typ = field[0], field[1]
            while issubclass(typ, C.Array):
                typ = typ._type_
            if issubclass(typ, (C._Pointer, C.c_void_p, C.c_char_p, C._CFuncPtr)):
                h.update(b"*")          # an address is not content; what a piece points at is fingerprinted by the caller's arrays
            else:
                _fingerprint(h, getattr(v, name))
    elif isinstance(v, C.Array):
        h.update(b"[")
        for x in v:
            _fingerprint(h, x)
    elif isinstance(v, (list, tuple)):
        h.update(b"(%d" % len(v))
        for x in v:
            _fingerprint(h, x)
    elif isinstance(v, dict):
        h.update(b"{")
        for k in sorted(v):
            h.update(repr(k).encode())
            _fingerprint(h, v[k])
    elif isinstance(v, C._SimpleCData):
        h.update(type(v).__name__.encode() + repr(v.value).encode())
    elif isinstance(v, np.generic):
        h.update(v.dtype.str.encode() + v.tobytes())
    elif v is None or isinstance(v, (bool, int, float, str, bytes)):
        h.update(repr(v).encode())
    else:
        raise TypeError(f"recorded: cannot fingerprint an argument of type {type(v).__name__}")


def _flatten(obj, leaves):
    if isinstance(obj, tuple):
        return ["t"] + [_flatten(x, leaves) for x in obj]
    if obj is None:
        return None
    leaves.append(np.asarray(obj))
    return len(leaves) - 1


def _unflatten(spec, leaves):
    if isinstance(spec, list):
        return tuple(_unflatten(x, leaves) for x in spec[1:])
    if spec is None:
        return None
    a = leaves[spec]
    return a if a.ndim else a[()]


def _raw(a: np.ndarray) -> np.ndarray:
    return np.ascontiguousarray(a).reshape(-1).view(f"u{a.dtype.itemsize}") if a.dtype.itemsize in (1, 2, 4, 8) else None


def _store(name: str, key: str, out, cand) -> None:
    import hashlib
    import json
    leaves, cleaves = [], []
    spec = _flatten(out, leaves)
    if cand is not None:
        _flatten(cand, cleaves)
    entry = {key: np.array(json.dumps([spec, len(leaves)]))}
    for i, a in enumerate(leaves):
        c = cleaves[i] if i < len(cleaves) else None
        if a.ndim and c is not None and c.shape == a.shape and c.dtype == a.dtype and _raw(a) is not None:
            ra, rc = _raw(a), _raw(c)
            idx = np.flatnonzero(ra != rc)
            entry[f"{key}.{i}.sha"] = np.array(hashlib.sha256(ra.tobytes()).hexdigest())
            entry[f"{key}.{i}.shape"] = np.array(a.shape, np.int64)
            entry[f"{key}.{i}.idx"] = idx.astype(np.int32 if ra.size < 2 ** 31 else np.int64)
            entry[f"{key}.{i}.val"] = ra[idx]
        else:
            entry[f"{key}.{i}"] = a
    _recorded_now.setdefault(name, {}).update(entry)


def _load(name: str, key: str, cand_fn, args, kwargs):
    import hashlib
    import json
    if name not in _records:
        _records[name] = {}
        for path in _record_files(name):
            _records[name].update(np.load(path))
    rec = _records[name]
    if key not in rec:
        raise AssertionError(f"{name}: the reference is not built here and these arguments were never recorded "
                             "(tests/golden/make_golden_reference.py records them where the reference sources are)")
    spec, n = json.loads(str(rec[key]))
    cleaves = None
    leaves = []
    for i in range(n):
        if f"{key}.{i}" in rec:
            leaves.append(rec[f"{key}.{i}"])
            continue
        if cleaves is None:
            cleaves = []
            _flatten(cand_fn(*args, **kwargs), cleaves)
        c = np.array(cleaves[i])
        assert tuple(c.shape) == tuple(rec[f"{key}.{i}.shape"]), f"{name}: the oracle's output no longer has the recorded shape"
        rc = _raw(c)
        rc[rec[f"{key}.{i}.idx"]] = rec[f"{key}.{i}.val"]
        assert hashlib.sha256(rc.tobytes()).hexdigest() == str(rec[f"{key}.{i}.sha"]), (
            f"{name}: the oracle plus the recorded differences no longer rebuilds the reference's output "
            "(the oracle changed where it used to equal the reference)")
        leaves.append(c)
    return _unflatten(spec, leaves)


def recorded(candidate=None):
    """wrap a helper that calls oracle/_ref (see the comment above); `candidate` takes the helper's arguments"""
    import functools
    import hashlib
    import inspect

    def wrap(fn):
        sig = inspect.signature(fn)
        name = f"{fn.__module__}.{fn.__name__}"

        @functools.wraps(fn)
        def call(*args, **kwargs):
            bound = sig.bind(*args, **kwargs)
            bound.apply_defaults()
            h = hashlib.sha256(name.encode())
            _fingerprint(h, dict(bound.arguments))
            key = h.hexdigest()[:24]
            if ref(bound.arguments.get("kind", "strict")) is None:
                return _load(name, key, candidate, args, kwargs)
            out = fn(*args, **kwargs)
            if RECORDING:
                _store(name, key, out, candidate(*args, **kwargs) if candidate else None)
            return out
        return call
    return wrap


def _save_recordings() -> None:
    """merge what this process recorded into tests/golden/reference/<helper>[.<shard>].npz, each file under 1 MB"""
    import io
    os.makedirs(RECORD_DIR, exist_ok=True)
    for name, entry in _recorded_now.items():
        old = {}
        for path in _record_files(name):
            old.update(np.load(path))
            os.remove(path)
        old.update(entry)
        n = 1
        while True:
            shards = [{k: v for k, v in old.items() if int(k[:6], 16) % n == i} for i in range(n)]
            blobs = []
            for shard in shards:
                buf = io.BytesIO()
                np.savez_compressed(buf, **shard)
                blobs.append(buf.getvalue())
            if max(len(b) for b in blobs) < 900_000:
                break
            n *= 2
        for i, blob in enumerate(blobs):
            with open(os.path.join(RECORD_DIR, f"{name}.npz" if n == 1 else f"{name}.{i}.npz"), "wb") as f:
                f.write(blob)


def _record_files(name: str):
    import glob
    return sorted(glob.glob(os.path.join(RECORD_DIR, glob.escape(name) + ".npz")) + glob.glob(os.path.join(RECORD_DIR, glob.escape(name) + ".[0-9]*.npz")))


@recorded()
def ref_size_t(fn: str, *args: int, kind: str = "strict") -> int:
    """a size or offset the reference's compiler gives (the ref_sizeof_* / ref_offsetof_* exports of oracle/_ref)"""
    f = getattr(ref(kind), fn)
    f.restype = C.c_size_t
    return int(f(*args))


def fptr(a: np.ndarray):
    assert a.dtype == np.float32 and a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(FP)


def ulp_distance(a: np.ndarray, b: np.ndarray) -> np.ndarray:
    """Distance in units of float32 representable values (sign-magnitude ordered)."""
    ai = a.view(np.int32).astype(np.int64)
    bi = b.view(np.int32).astype(np.int64)
    ai = np.where(ai < 0, -(ai & 0x7FFFFFFF), ai)
    bi = np.where(bi < 0, -(bi & 0x7FFFFFFF), bi)
    return np.abs(ai - bi)


# ---- RCD through the checkers ------------------------------------------------------------
def oracle_rcd(mosaic: np.ndarray, filters: int, pm=(1.0, 1.0, 1.0), fill: float = 0.0) -> np.ndarray:
    h, w = mosaic.shape
    out = np.zeros((h, w, 4), np.float32)
    f = oracle().orc_rcd_demosaic
    f.restype = C.c_int
    rc = f(fptr(out), fptr(mosaic), w, h, C.c_uint32(filters), (C.c_float * 3)(*pm), C.c_float(fill))
    assert rc in (0, 1)
    return out


def oracle_rcd_mask(mosaic: np.ndarray, filters: int, pm=(1.0, 1.0, 1.0)) -> np.ndarray:
    """bit 0: colour depends on memory the reference never initialised; bit 1: alpha never written."""
    h, w = mosaic.shape
    mask = np.zeros((h, w), np.uint8)
    f = oracle().orc_rcd_undefined_mask
    f.restype = C.c_int
    rc = f(mask.ctypes.data_as(C.POINTER(C.c_uint8)), fptr(mosaic), w, h, C.c_uint32(filters), (C.c_float * 3)(*pm))
    assert rc in (0, 1)
    return mask


@recorded(lambda mosaic, filters, pm=(1.0, 1.0, 1.0), kind="strict", poison=0.0: oracle_rcd(mosaic, filters, pm))
def ref_rcd(mosaic: np.ndarray, filters: int, pm=(1.0, 1.0, 1.0), kind: str = "strict", poison: float = 0.0):
    lib = ref(kind)
    if lib is None:
        return None
    h, w = mosaic.shape
    out = np.zeros((h, w, 4), np.float32)
    f = lib.ref_rcd_demosaic
    f.restype = C.c_int
    rc = f(fptr(out), fptr(mosaic), w, h, C.c_uint32(filters), (C.c_float * 3)(*pm), C.c_float(poison))
    assert rc in (0, 1)
    return out


# ---- synthetic Bayer frames (SURVEY.md 8d) ----------------------------------------------
def frame_uniform(w: int, h: int, seed: int) -> np.ndarray:
    """D-uniform: i.i.d. U[0,1) mosaic."""
    return np.random.Generator(np.random.PCG64(seed)).random((h, w), dtype=np.float32)


def _scene(w: int, h: int, rng) -> np.ndarray:
    xn = (np.arange(w, dtype=np.float32) / max(w, 1))[None, :]
    yn = (np.arange(h, dtype=np.float32) / max(h, 1))[:, None]
    s = (0.35 + 0.25 * xn + 0.1 * yn).astype(np.float32)
    for _ in range(6):
        fx, fy = rng.uniform(0.5, 6.0, 2)
        ph = rng.uniform(0, 2 * np.pi)
        ax = (2 * np.pi * fx * xn + ph).astype(np.float32)
        ay = (2 * np.pi * fy * yn).astype(np.float32)
        s += np.float32(0.06) * (np.cos(ax) * np.cos(ay) - np.sin(ax) * np.sin(ay))
    for _ in range(3):
        cx, cy, rad = rng.uniform(0.2, 0.8), rng.uniform(0.2, 0.8), rng.uniform(0.05, 0.2)
        d = np.sqrt((xn - np.float32(cx)) ** 2 + (yn - np.float32(cy)) ** 2)
        t = np.clip((d - np.float32(rad)) * np.float32(120.0), -60.0, 60.0)
        s += np.float32(0.25) / (np.float32(1.0) + np.exp(t))
    return s.astype(np.float32)


def cfa_colours(w: int, h: int, filters: int) -> np.ndarray:
    """FC() of every site (develop/imageop_math.h:190-193) as an (h, w) uint8 array."""
    rows = np.arange(h, dtype=np.uint32)[:, None]
    cols = np.arange(w, dtype=np.uint32)[None, :]
    sh = (((rows << 1) & 14) + (cols & 1)) << 1
    return ((np.uint32(filters) >> sh) & 3).astype(np.uint8)


def frame_natural(w: int, h: int, seed: int, filters: int = BAYER["RGGB"], iso: float = 100.0) -> np.ndarray:
    """D-natural: smooth scene through the CFA with Poisson-Gaussian noise, exact 0s and 1s sprinkled in."""
    rng = np.random.Generator(np.random.PCG64(seed))
    s = _scene(w, h, rng)
    gains = np.array([0.5, 1.0, 0.65, 1.0], np.float32)
    m = s * gains[cfa_colours(w, h, filters)]
    a = np.float32(1e-4 * (iso / 100.0))
    m += rng.standard_normal((h, w), dtype=np.float32) * np.sqrt(np.maximum(a * m, 0))
    np.clip(m, 0.0, 1.0, out=m)
    r = rng.random((h, w), dtype=np.float32)
    m[r < 0.005] = 0.0
    m[r > 0.995] = 1.0
    return np.ascontiguousarray(m, dtype=np.float32)


def frame_edge(w: int, h: int, kind: str) -> np.ndarray:
    """D-edge cases."""
    if kind == "zeros":
        return np.zeros((h, w), np.float32)
    if kind == "ones":
        return np.ones((h, w), np.float32)
    if kind == "impulses":
        m = np.full((h, w), 0.25, np.float32)
        m[::17, ::13] = 1.0
        m[5::23, 7::19] = 0.0
        return m
    if kind == "negative":
        m = frame_uniform(w, h, 7)
        m[::3, ::5] = -0.01
        return m
    if kind == "tiny":
        m = frame_uniform(w, h, 8) * 1e-3
        m[::2, ::3] = 1e-30
        m[1::4, 1::5] = 1e-41  # subnormal: flushed by FTZ/DAZ on both sides
        return m.astype(np.float32)
    raise ValueError(kind)


# ---- colour conversion fixtures and checkers (SURVEY.md 8d "fixed metadata") -----------------
LUT_SAMPLES = 0x10000
FP_STRICT, FP_CONTRACT = 0, 1

# camera RGB -> linear Rec2020 (a fixed, plausible composite; rows sum to ~1) and
# linear Rec2020 -> linear sRGB (ITU-R BT.2087)
MATRIX_CAM_TO_REC2020 = np.array([[0.7398, 0.1873, 0.0729],
                                  [0.0825, 0.9672, -0.0497],
                                  [0.0209, -0.1264, 1.1055]], np.float32)
MATRIX_REC2020_TO_SRGB = np.array([[1.6605, -0.5876, -0.0728],
                                   [-0.1246, 1.1329, -0.0083],
                                   [-0.0182, -0.1006, 1.1187]], np.float32)
MATRIX_CLIP_IN = np.array([[0.6274, 0.3293, 0.0433],
                           [0.0691, 0.9195, 0.0114],
                           [0.0164, 0.0880, 0.8956]], np.float32)


def srgb_encode_lut() -> np.ndarray:
    """sRGB OETF sampled at 65536 points in double, rounded to float (3 identical channels)."""
    x = np.arange(LUT_SAMPLES, dtype=np.float64) / (LUT_SAMPLES - 1)
    y = np.where(x <= 0.0031308, 12.92 * x, 1.055 * np.power(x, 1 / 2.4) - 0.055)
    return np.ascontiguousarray(np.tile(y.astype(np.float32), (3, 1)))


def srgb_decode_lut() -> np.ndarray:
    x = np.arange(LUT_SAMPLES, dtype=np.float64) / (LUT_SAMPLES - 1)
    y = np.where(x <= 0.04045, x / 12.92, np.power((x + 0.055) / 1.055, 2.4))
    return np.ascontiguousarray(np.tile(y.astype(np.float32), (3, 1)))


def _lut_at(lut: np.ndarray, v: float) -> np.float32:
    ft = np.float32(min(max(np.float32(v) * np.float32(LUT_SAMPLES - 1), 0), LUT_SAMPLES - 1))
    t = int(ft) if ft < LUT_SAMPLES - 2 else LUT_SAMPLES - 2
    f = np.float32(ft - np.float32(t))
    return np.float32(lut[t] * (np.float32(1) - f) + lut[t + 1] * f)


def fit_unbounded_coeffs(lut3: np.ndarray) -> np.ndarray:
    """dt_ioppr_init_unbounded_coeffs (colorprofiles/iop_profile.c:303-329) + dt_iop_estimate_exp
    (develop/imageop_math.h:135-165), in float32."""
    out = np.zeros((3, 3), np.float32)
    xs = [np.float32(v) for v in (0.7, 0.8, 0.9, 1.0)]
    for k in range(3):
        lut = lut3[k]
        if lut[0] < 0:
            out[k, 0] = -1.0
            continue
        ys = [_lut_at(lut, x) for x in xs]
        x0, y0 = xs[-1], ys[-1]
        g, cnt = np.float32(0), 0
        for x, y in zip(xs[:-1], ys[:-1]):
            if y / y0 > 0 and x / x0 > 0:
                g = np.float32(g + np.float32(np.log(np.float32(y / y0))) / np.float32(np.log(np.float32(x / x0))))
                cnt += 1
        g = np.float32(g * np.float32(1.0 / cnt)) if cnt else np.float32(1)
        out[k] = (np.float32(1) / x0, y0, g)
    return out


def aligned_empty(shape, dtype=np.float32, align: int = 64) -> np.ndarray:
    n = int(np.prod(shape)) * np.dtype(dtype).itemsize
    raw = np.empty(n + align, np.uint8)
    off = (-raw.ctypes.data) % align
    return raw[off:off + n].view(dtype).reshape(shape)


def _fp_or_null(a):
    return fptr(a) if a is not None else None


def _conv_args(rgba, matrix, clip, lut_s, co_s, lut_t, co_t):
    h, w = rgba.shape[:2]
    src = aligned_empty(rgba.shape)
    src[...] = rgba
    dst = aligned_empty(rgba.shape)
    dst[...] = 0
    keep = [np.ascontiguousarray(a, np.float32) if a is not None else None for a in (matrix, clip, lut_s, co_s, lut_t, co_t)]
    args = [fptr(src), fptr(dst), C.c_size_t(w), C.c_size_t(h), _fp_or_null(keep[0].reshape(-1)),
            _fp_or_null(keep[1].reshape(-1) if keep[1] is not None else None), C.c_int(1 if clip is not None else 0),
            _fp_or_null(keep[2]), _fp_or_null(keep[3].reshape(-1) if keep[3] is not None else None),
            _fp_or_null(keep[4]), _fp_or_null(keep[5].reshape(-1) if keep[5] is not None else None)]
    return src, dst, keep, args


def oracle_convert(rgba, matrix, clip=None, lut_s=None, co_s=None, lut_t=None, co_t=None, fp=FP_CONTRACT):
    src, dst, keep, args = _conv_args(rgba, matrix, clip, lut_s, co_s, lut_t, co_t)
    f = oracle().orc_apply_matrix_conversion
    f.restype = C.c_int
    assert f(*args, C.c_int(fp)) == 0
    return np.array(dst)


@recorded(lambda rgba, matrix, clip=None, lut_s=None, co_s=None, lut_t=None, co_t=None, kind="fast":
          oracle_convert(rgba, matrix, clip, lut_s, co_s, lut_t, co_t, fp=FP_CONTRACT if kind == "fast" else FP_STRICT))
def ref_convert(rgba, matrix, clip=None, lut_s=None, co_s=None, lut_t=None, co_t=None, kind="fast"):
    lib = ref(kind)
    if lib is None:
        return None
    src, dst, keep, args = _conv_args(rgba, matrix, clip, lut_s, co_s, lut_t, co_t)
    f = lib.ref_apply_matrix_conversion
    f.restype = C.c_int
    assert f(*args) == 0
    return np.array(dst)


def rgba_test_image(w: int, h: int, seed: int, lo: float = -0.05, hi: float = 1.6) -> np.ndarray:
    """RGBA floats covering negatives, [0,1], and values past white (the eval_exp branch)."""
    rng = np.random.Generator(np.random.PCG64(seed))
    a = rng.uniform(lo, hi, (h, w, 4)).astype(np.float32)
    a[..., 3] = rng.uniform(0, 1, (h, w)).astype(np.float32)
    a[0, 0, :3] = (0.0, 1.0, 1.0)
    a[0, 1, :3] = (-0.0, 0.5, 2.0)
    return a


# ---- profiled denoise (wavelets) through the checkers ------------------------------------------
def oracle_eaw_decompose(img: np.ndarray, scale: int, inv_sigma2: float):
    h, w = img.shape[:2]
    coarse, detail = np.zeros_like(img), np.zeros_like(img)
    sums = (C.c_double * 4)()
    oracle().orc_eaw_dn_decompose(fptr(coarse), fptr(img), fptr(detail), sums, scale, C.c_float(inv_sigma2), w, h)
    return coarse, detail, np.array(list(sums))


@recorded(lambda img, scale, inv_sigma2, kind="strict": oracle_eaw_decompose(img, scale, inv_sigma2))
def ref_eaw_decompose(img: np.ndarray, scale: int, inv_sigma2: float, kind: str = "strict"):
    lib = ref(kind)
    if lib is None:
        return None
    h, w = img.shape[:2]
    coarse, detail = np.zeros_like(img), np.zeros_like(img)
    sums = (C.c_float * 4)()
    lib.eaw_dn_decompose(fptr(coarse), fptr(img), fptr(detail), sums, scale, C.c_float(inv_sigma2), w, h)
    return coarse, detail, np.array(list(sums))


def oracle_eaw_synthesize(base: np.ndarray, detail: np.ndarray, thr, boost=(1, 1, 1, 1)):
    h, w = base.shape[:2]
    out = np.zeros_like(base)
    oracle().orc_eaw_synthesize(fptr(out), fptr(base), fptr(detail), (C.c_float * 4)(*thr), (C.c_float * 4)(*boost), w, h)
    return out


@recorded(lambda base, detail, thr, boost=(1, 1, 1, 1), kind="strict": oracle_eaw_synthesize(base, detail, thr, boost))
def ref_eaw_synthesize(base, detail, thr, boost=(1, 1, 1, 1), kind="strict"):
    lib = ref(kind)
    if lib is None:
        return None
    h, w = base.shape[:2]
    out = np.zeros_like(base)
    lib.eaw_synthesize(fptr(out), fptr(base), fptr(detail), (C.c_float * 4)(*thr), (C.c_float * 4)(*boost), w, h)
    return out


def oracle_denoise_wavelets(rgba: np.ndarray, data, roi_scale=1.0, buf=None, wb=(2.0, 1.0, 1.5, 0.0), pm=(1.0, 1.0, 1.0, 1.0)):
    """data: ansel_b200.DenoiseProfileData (the public ABI struct)."""
    h, w = rgba.shape[:2]
    out = np.zeros_like(rgba)
    bw, bh = buf if buf else (w, h)
    f = oracle().orc_denoiseprofile_wavelets
    f.restype = C.c_int
    rc = f(fptr(np.ascontiguousarray(rgba)), fptr(out), w, h, C.byref(data), C.c_float(roi_scale), bw, bh,
           (C.c_float * 4)(*wb), (C.c_float * 4)(*pm))
    assert rc == 0
    return out


def rgba_scene(w: int, h: int, seed: int, noise: float = 0.02) -> np.ndarray:
    """A demosaiced-looking RGBA frame: smooth scene + noise, alpha 0 (what demosaic hands to denoise)."""
    rng = np.random.Generator(np.random.PCG64(seed))
    s = _scene(w, h, rng)
    img = np.empty((h, w, 4), np.float32)
    for c, g in enumerate((0.5, 1.0, 0.65)):
        img[..., c] = s * np.float32(g) + rng.standard_normal((h, w), dtype=np.float32) * np.float32(noise)
    np.clip(img[..., :3], 0.0, None, out=img[..., :3])
    img[..., 3] = 0.0
    return img


# ---- filmic rgb ------------------------------------------------------------------------------------
# RGB -> XYZ(D50) of linear Rec2020 (the default work profile) and of sRGB (the default output profile)
REC2020_TO_XYZ_D50 = np.array([[0.6734241, 0.1656411, 0.1251286],
                               [0.2790177, 0.6753402, 0.0456377],
                               [-0.0019300, 0.0299784, 0.7973330]])
SRGB_TO_XYZ_D50 = np.array([[0.4360747, 0.3850649, 0.1430804],
                            [0.2225045, 0.7168786, 0.0606169],
                            [0.0139322, 0.0971045, 0.7141733]])


def profile_pair(m_in64: np.ndarray):
    """(matrix_in, matrix_out) as float32 3x3, matrix_out the float64 inverse rounded once."""
    return np.ascontiguousarray(m_in64, np.float32), np.ascontiguousarray(np.linalg.inv(m_in64), np.float32)


def filmic_default_params(**over) -> dict:
    """$DEFAULT values of dt_iop_filmicrgb_params_t (src/iop/filmicrgb.c:244-274), field order preserved."""
    p = dict(grey_point_source=18.45, black_point_source=-8.0, white_point_source=4.0, reconstruct_threshold=16.0,
             reconstruct_feather=3.0, reconstruct_bloom_vs_details=100.0, reconstruct_grey_vs_color=100.0,
             reconstruct_structure_vs_texture=100.0, security_factor=0.0, grey_point_target=18.45,
             black_point_target=0.01517634, white_point_target=100.0, output_power=4.0, latitude=10.0, contrast=1.18,
             saturation=0.0, balance=0.0, noise_level=0.05, preserve_color=1, version=7, auto_hardness=1, custom_grey=0,
             high_quality_reconstruction=1, noise_distribution=2, shadows=3, highlights=3, compensate_icc_black=0,
             spline_version=2)
    p.update(over)
    return p


def filmic_params_blob(p: dict) -> np.ndarray:
    floats = ["grey_point_source", "black_point_source", "white_point_source", "reconstruct_threshold", "reconstruct_feather",
              "reconstruct_bloom_vs_details", "reconstruct_grey_vs_color", "reconstruct_structure_vs_texture", "security_factor",
              "grey_point_target", "black_point_target", "white_point_target", "output_power", "latitude", "contrast",
              "saturation", "balance", "noise_level"]
    ints = ["preserve_color", "version", "auto_hardness", "custom_grey", "high_quality_reconstruction", "noise_distribution",
            "shadows", "highlights", "compensate_icc_black", "spline_version"]
    blob = np.zeros(112, np.uint8)
    blob[:72].view(np.float32)[:] = [p[k] for k in floats]
    blob[72:112].view(np.int32)[:] = [p[k] for k in ints]
    return blob


@recorded()
def ref_filmic_commit(params: dict, kind: str = "strict"):
    """dt_iop_filmicrgb_data_t (832 bytes) from the reference's own commit_params()."""
    lib = ref(kind)
    if lib is None:
        return None
    lib.ref_filmic_sizeof_params.restype = C.c_size_t
    lib.ref_filmic_sizeof_data.restype = C.c_size_t
    assert lib.ref_filmic_sizeof_params() == 112 and lib.ref_filmic_sizeof_data() == 832
    blob = filmic_params_blob(params)
    data = np.zeros(832, np.uint8)
    lib.ref_filmic_commit(blob.ctypes.data_as(C.c_void_p), data.ctypes.data_as(C.c_void_p))
    return data


def _f9(a):
    return fptr(np.ascontiguousarray(a, np.float32).reshape(-1).copy()) if a is not None else None


@recorded(lambda rgba, data_blob, work, export=None, kind="strict": oracle_filmic_agx(rgba, data_blob, work, export))
def ref_filmic_agx(rgba, data_blob, work, export=None, kind="strict"):
    lib = ref(kind)
    h, w = rgba.shape[:2]
    src, dst = aligned_empty(rgba.shape), aligned_empty(rgba.shape)
    src[...] = rgba
    dst[...] = 0
    keep = [_f9(work[0]), _f9(work[1]), _f9(export[0]) if export else None, _f9(export[1]) if export else None]
    lib.ref_filmic_agx(fptr(src), fptr(dst), C.c_size_t(w), C.c_size_t(h), data_blob.ctypes.data_as(C.c_void_p), *keep)
    return np.array(dst)


def oracle_filmic_agx(rgba, data_blob, work, export=None):
    h, w = rgba.shape[:2]
    src = np.ascontiguousarray(rgba)
    dst = np.zeros_like(src)
    keep = [_f9(work[0]), _f9(work[1]), _f9(export[0]) if export else None, _f9(export[1]) if export else None]
    data = aligned_empty((832,), np.uint8)
    data[:] = data_blob
    f = oracle().orc_filmic_agx
    f.restype = C.c_int
    rc = f(fptr(src), fptr(dst), C.c_size_t(w), C.c_size_t(h), data.ctypes.data_as(C.c_void_p), *keep)
    assert rc == 0, rc
    return dst


@recorded(lambda rgba, data_blob, work, export=None, kind="strict": oracle_filmic_legacy(rgba, data_blob, work, export))
def ref_filmic_legacy(rgba, data_blob, work, export=None, kind="strict"):
    """the v1..v5 colour sciences through the reference's own functions; lanes a branch does not write keep the input's"""
    lib = ref(kind)
    h, w = rgba.shape[:2]
    src, dst = aligned_empty(rgba.shape), aligned_empty(rgba.shape)
    src[...] = rgba
    dst[...] = rgba
    keep = [_f9(work[0]), _f9(work[1]), _f9(export[0]) if export else None, _f9(export[1]) if export else None]
    lib.ref_filmic_legacy.restype = C.c_int
    assert lib.ref_filmic_legacy(fptr(src), fptr(dst), C.c_size_t(w), C.c_size_t(h), data_blob.ctypes.data_as(C.c_void_p), *keep) == 0
    return np.array(dst)


def oracle_filmic_legacy(rgba, data_blob, work, export=None):
    h, w = rgba.shape[:2]
    src = np.ascontiguousarray(rgba)
    dst = src.copy()
    keep = [_f9(work[0]), _f9(work[1]), _f9(export[0]) if export else None, _f9(export[1]) if export else None]
    data = aligned_empty((832,), np.uint8)
    data[:] = data_blob
    f = oracle().orc_filmic_legacy
    f.restype = C.c_int
    rc = f(fptr(src), fptr(dst), C.c_size_t(w), C.c_size_t(h), data.ctypes.data_as(C.c_void_p), *keep)
    assert rc == 0, rc
    return dst


def _filmic_reconstruct(lib, fn, rgba, data_blob, iscale, roi_scale, buf):
    h, w = rgba.shape[:2]
    src, dst, mask = aligned_empty(rgba.shape), aligned_empty(rgba.shape), aligned_empty((h, w))
    src[...] = rgba
    dst[...] = 0
    f = getattr(lib, fn)
    f.restype = C.c_int
    oracle().orc_fp_fast_mode_all()   # values next to FLT_MIN occur here (lane 3): every thread flushes, like the pipe's
    bw, bh = buf if buf else (w, h)
    rc = f(fptr(src), fptr(dst), fptr(mask), C.c_size_t(w), C.c_size_t(h), data_blob.ctypes.data_as(C.c_void_p), C.c_float(iscale), C.c_double(roi_scale),
           int(bw), int(bh))
    return rc, np.array(dst), np.array(mask)


@recorded(lambda rgba, data_blob, iscale=1.0, roi_scale=1.0, buf=None, kind="strict": oracle_filmic_reconstruct(rgba, data_blob, iscale, roi_scale, buf))
def ref_filmic_reconstruct(rgba, data_blob, iscale=1.0, roi_scale=1.0, buf=None, kind="strict"):
    """process() :2729-2838 on the cut functions: (recovered?, frame the tone mapping reads, clipping mask)"""
    lib = ref(kind)
    return None if lib is None else _filmic_reconstruct(lib, "ref_filmic_reconstruct", rgba, data_blob, iscale, roi_scale, buf)


def oracle_filmic_reconstruct(rgba, data_blob, iscale=1.0, roi_scale=1.0, buf=None):
    return _filmic_reconstruct(oracle(), "orc_filmic_reconstruct", rgba, data_blob, iscale, roi_scale, buf)


def filmic_prepare(lib, fn, version, work, export=None):
    out = np.zeros(72, np.float32)
    keep = [_f9(work[0]), _f9(work[1]), _f9(export[0]) if export else None, _f9(export[1]) if export else None]
    getattr(lib, fn)(version, *keep, fptr(out))
    return out


@recorded(lambda version, work, export=None, kind="strict": filmic_prepare(oracle(), "orc_filmic_prepare", version, work, export))
def ref_filmic_prepare(version, work, export=None, kind="strict"):
    return filmic_prepare(ref(kind), "ref_filmic_prepare", version, work, export)


def hdr_rgba(w: int, h: int, seed: int) -> np.ndarray:
    """Scene-referred RGBA for tone mapping: log-uniform over ~16 EV, some negatives, NaN, huge values."""
    rng = np.random.Generator(np.random.PCG64(seed))
    ev = rng.uniform(-11, 5, (h, w, 1)).astype(np.float32)
    base = np.float32(0.1845) * np.exp2(ev)
    img = (base * rng.uniform(0.3, 1.7, (h, w, 4)).astype(np.float32)).astype(np.float32)
    neg = rng.random((h, w)) < 0.02
    img[neg, rng.integers(0, 3)] *= -0.05
    img[..., 3] = rng.uniform(0, 1, (h, w)).astype(np.float32)
    img[0, 0, :3] = (np.nan, 0.5, 0.5)
    img[0, 1, :3] = (1e9, -1e9, 0.0)
    img[0, 2, :3] = 0.0
    img[0, 3, :3] = 0.1845
    return img


# ---- non-local means ----------------------------------------------------------------------------------
def _nlm_call(lib, fn, img, scattering, scale, luma, chroma, center_weight, sharpness, P, K, decimate, norm):
    h, w = img.shape[:2]
    src = aligned_empty(img.shape)
    src[...] = img
    out = aligned_empty(img.shape)
    out[...] = 0
    f = getattr(lib, fn)
    f(fptr(src), fptr(out), w, h, C.c_float(scattering), C.c_float(scale), C.c_float(luma), C.c_float(chroma),
      C.c_float(center_weight), C.c_float(sharpness), P, K, decimate, (C.c_float * 4)(*norm))
    return np.array(out)


def oracle_nlmeans(img, *, scattering=0.0, scale=1.0, luma=1.0, chroma=1.0, center_weight=0.1, sharpness=0.005, P=1, K=7,
                   decimate=0, norm=(1.0, 1.0, 1.0, 1.0)):
    return _nlm_call(oracle(), "orc_nlmeans_denoise", img, scattering, scale, luma, chroma, center_weight, sharpness, P, K, decimate, norm)


@recorded(lambda img, kind="strict", **kw: oracle_nlmeans(img, **kw))
def ref_nlmeans(img, kind="strict", **kw):
    lib = ref(kind)
    if lib is None:
        return None
    d = dict(scattering=0.0, scale=1.0, luma=1.0, chroma=1.0, center_weight=0.1, sharpness=0.005, P=1, K=7, decimate=0,
             norm=(1.0, 1.0, 1.0, 1.0))
    d.update(kw)
    return _nlm_call(lib, "ref_nlmeans_denoise", img, d["scattering"], d["scale"], d["luma"], d["chroma"], d["center_weight"],
                     d["sharpness"], d["P"], d["K"], d["decimate"], d["norm"])


# ---- local Laplacian (local contrast) ---------------------------------------------------------------
def lab_scene(w: int, h: int, seed: int) -> np.ndarray:
    """Lab-like RGBA: L in [0, 100] with structure, a/b small, alpha arbitrary."""
    rng = np.random.Generator(np.random.PCG64(seed))
    s = _scene(w, h, rng)
    img = np.empty((h, w, 4), np.float32)
    img[..., 0] = np.clip(s * 70 + rng.standard_normal((h, w), dtype=np.float32) * 1.5, 0, 100)
    img[..., 1] = rng.uniform(-20, 20, (h, w)).astype(np.float32)
    img[..., 2] = rng.uniform(-20, 20, (h, w)).astype(np.float32)
    img[..., 3] = rng.uniform(0, 1, (h, w)).astype(np.float32)
    return img


def _ll_call(lib, fn, img, sigma, shadows, highlights, clarity):
    h, w = img.shape[:2]
    src = aligned_empty(img.shape)
    src[...] = img
    out = aligned_empty(img.shape)
    out[...] = 0
    f = getattr(lib, fn)
    f.restype = C.c_int
    assert f(fptr(src), fptr(out), w, h, C.c_float(sigma), C.c_float(shadows), C.c_float(highlights), C.c_float(clarity)) == 0
    return np.array(out)


def oracle_local_laplacian(img, sigma=0.5, shadows=0.5, highlights=0.5, clarity=0.25):
    """defaults = dt_iop_bilat_params_t $DEFAULTs (midtone, sigma_s, sigma_r, detail), iop/bilat.c:78-86,354"""
    return _ll_call(oracle(), "orc_local_laplacian", img, sigma, shadows, highlights, clarity)


@recorded(lambda img, sigma=0.5, shadows=0.5, highlights=0.5, clarity=0.25, kind="strict": oracle_local_laplacian(img, sigma, shadows, highlights, clarity))
def ref_local_laplacian(img, sigma=0.5, shadows=0.5, highlights=0.5, clarity=0.25, kind="strict"):
    lib = ref(kind)
    return None if lib is None else _ll_call(lib, "ref_local_laplacian", img, sigma, shadows, highlights, clarity)


# ---- diffuse or sharpen -------------------------------------------------------------------------------
def _diffuse_call(lib, fn, img, data, iscale, roi_scale):
    h, w = img.shape[:2]
    src = aligned_empty(img.shape)
    src[...] = img
    out = aligned_empty(img.shape)
    out[...] = 0
    f = getattr(lib, fn)
    f.restype = C.c_int
    assert f(fptr(src), fptr(out), w, h, C.byref(data), C.c_float(iscale), C.c_float(roi_scale)) == 0
    return np.array(out)


def oracle_diffuse(img, data, iscale=1.0, roi_scale=1.0):
    """data: ansel_b200.DiffuseData (== dt_iop_diffuse_params_t)"""
    return _diffuse_call(oracle(), "orc_diffuse", img, data, iscale, roi_scale)


@recorded(lambda img, data, iscale=1.0, roi_scale=1.0, kind="strict": oracle_diffuse(img, data, iscale, roi_scale))
def ref_diffuse(img, data, iscale=1.0, roi_scale=1.0, kind="strict"):
    lib = ref(kind)
    if lib is None:
        return None
    lib.ref_diffuse_sizeof_params.restype = C.c_size_t
    assert lib.ref_diffuse_sizeof_params() == C.sizeof(data)
    return _diffuse_call(lib, "ref_diffuse_process", img, data, iscale, roi_scale)


# ---- RGB <-> Lab glue, denoise (non-local means) iop --------------------------------------------------
def _glue(lib, fn, img, m, nargs):
    h, w = img.shape[:2]
    src = aligned_empty(img.shape)
    src[...] = img
    out = aligned_empty(img.shape)
    out[...] = img            # lane 3 of RGB->Lab is not written by the reference: compare it as "kept"
    f = getattr(lib, fn)
    f.restype = C.c_int
    mats = [(C.c_float * 9)(*np.asarray(x, np.float32).reshape(-1)) for x in m]
    assert f(fptr(src), fptr(out), w, h, *mats[:nargs]) == 0
    return np.array(out)


def oracle_rgb_to_lab(img, work):
    return _glue(oracle(), "orc_rgb_to_lab", img, (work[0],), 1)


def oracle_lab_to_rgb(img, work):
    return _glue(oracle(), "orc_lab_to_rgb", img, (work[1],), 1)


@recorded(lambda img, work, kind="strict": oracle_rgb_to_lab(img, work))
def ref_rgb_to_lab(img, work, kind="strict"):
    lib = ref(kind)
    return None if lib is None else _glue(lib, "ref_rgb_to_lab", img, work, 2)


@recorded(lambda img, work, kind="strict": oracle_lab_to_rgb(img, work))
def ref_lab_to_rgb(img, work, kind="strict"):
    lib = ref(kind)
    return None if lib is None else _glue(lib, "ref_lab_to_rgb", img, work, 2)


def _glue_trc(lib, fn, img, mats, luts, coeffs):
    """luts / coeffs: one (3 x 65536, 3 x 3) pair per argument the entry takes, in order"""
    h, w = img.shape[:2]
    src = aligned_empty(img.shape)
    src[...] = img
    out = aligned_empty(img.shape)
    out[...] = img            # in place is how the pipe calls it: unwritten lanes keep the pixel
    f = getattr(lib, fn)
    f.restype = C.c_int
    m = [(C.c_float * 9)(*np.asarray(x, np.float32).reshape(-1)) for x in mats]
    keep = [np.ascontiguousarray(x, np.float32) for x in luts]
    co = [(C.c_float * 9)(*np.asarray(x, np.float32).reshape(-1)) for x in coeffs]
    assert f(fptr(src), fptr(out), w, h, *m, *[fptr(x) for x in keep], *co) == 0
    return np.array(out)


def oracle_rgb_to_lab_trc(img, work, lut_in, co_in):
    return _glue_trc(oracle(), "orc_rgb_to_lab_trc", img, (work[0],), (lut_in,), (co_in,))


def oracle_lab_to_rgb_trc(img, work, lut_out, co_out):
    return _glue_trc(oracle(), "orc_lab_to_rgb_trc", img, (work[1],), (lut_out,), (co_out,))


@recorded(lambda img, work, lut_in, co_in, lut_out, co_out, kind="strict": oracle_rgb_to_lab_trc(img, work, lut_in, co_in))
def ref_rgb_to_lab_trc(img, work, lut_in, co_in, lut_out, co_out, kind="strict"):
    lib = ref(kind)
    return None if lib is None else _glue_trc(lib, "ref_rgb_to_lab_trc", img, work, (lut_in, lut_out), (co_in, co_out))


@recorded(lambda img, work, lut_in, co_in, lut_out, co_out, kind="strict":
          oracle_lab_to_rgb(img, work) if (lut_in[:, 0] < 0).all() else oracle_lab_to_rgb_trc(img, work, lut_out, co_out))
def ref_lab_to_rgb_trc(img, work, lut_in, co_in, lut_out, co_out, kind="strict"):
    lib = ref(kind)
    return None if lib is None else _glue_trc(lib, "ref_lab_to_rgb_trc", img, work, (lut_in, lut_out), (co_in, co_out))


def oracle_nlmeans_iop(img, data, roi_scale=1.0, decimate=0, mask_display=0):
    h, w = img.shape[:2]
    src = aligned_empty(img.shape)
    src[...] = img
    out = aligned_empty(img.shape)
    out[...] = 0
    f = oracle().orc_nlmeans_iop
    f.restype = C.c_int
    assert f(fptr(src), fptr(out), w, h, C.byref(data), C.c_double(roi_scale), decimate, mask_display) == 0
    return np.array(out)


@recorded(lambda img, data, roi_scale=1.0, pipe_type=1, has_preview=0, mask_display=0, kind="strict":
          oracle_nlmeans_iop(img, data, roi_scale, 1 if (pipe_type == 4 or has_preview) else 0, mask_display))
def ref_nlmeans_iop(img, data, roi_scale=1.0, pipe_type=1, has_preview=0, mask_display=0, kind="strict"):
    lib = ref(kind)
    if lib is None:
        return None
    h, w = img.shape[:2]
    src = aligned_empty(img.shape)
    src[...] = img
    out = aligned_empty(img.shape)
    out[...] = 0
    f = lib.ref_nlmeans_iop
    f.restype = C.c_int
    assert f(fptr(src), fptr(out), w, h, (C.c_float * 4)(data.radius, data.strength, data.luma, data.chroma), C.c_double(roi_scale),
             pipe_type, has_preview, mask_display) == 0
    return np.array(out)


# ---- demosaic: green equilibration and colour smoothing ---------------------------------------------------
def _geq(lib, fn, mosaic, filters, x, y, thr=None):
    h, w = mosaic.shape
    src = aligned_empty(mosaic.shape)
    src[...] = mosaic
    out = aligned_empty(mosaic.shape)
    f = getattr(lib, fn)
    f.restype = None
    args = [fptr(out), fptr(src), w, h, C.c_uint32(filters), x, y]
    if thr is not None:
        args.append(C.c_float(thr))
    f(*args)
    return np.array(out)


def oracle_green_eq(mosaic, filters, mode, x=0, y=0, iso=100.0):
    """mode: dt_iop_demosaic_greeneq_t 1 local, 2 full, 3 both (iop/demosaic.c:1137-1170)"""
    thr = np.float32(0.0001) * np.float32(iso)
    m = mosaic
    if mode in (2, 3):
        m = _geq(oracle(), "orc_green_eq_favg", m, filters, x, y)
    if mode in (1, 3):
        m = _geq(oracle(), "orc_green_eq_lavg", m, filters, x, y, thr)
    return m


@recorded(lambda mosaic, filters, mode, x=0, y=0, iso=100.0, kind="strict": oracle_green_eq(mosaic, filters, mode, x, y, iso))
def ref_green_eq(mosaic, filters, mode, x=0, y=0, iso=100.0, kind="strict"):
    lib = ref(kind)
    if lib is None:
        return None
    thr = np.float32(0.0001) * np.float32(iso)
    m = mosaic
    if mode in (2, 3):
        m = _geq(lib, "ref_green_eq_favg", m, filters, x, y)
    if mode in (1, 3):
        m = _geq(lib, "ref_green_eq_lavg", m, filters, x, y, thr)
    return m


def _smooth(lib, fn, rgba, passes):
    h, w = rgba.shape[:2]
    buf = aligned_empty(rgba.shape)
    buf[...] = rgba
    f = getattr(lib, fn)
    f.restype = None
    f(fptr(buf), w, h, passes)
    return np.array(buf)


def oracle_color_smoothing(rgba, passes):
    return _smooth(oracle(), "orc_color_smoothing", rgba, passes)


@recorded(lambda rgba, passes, kind="strict": oracle_color_smoothing(rgba, passes))
def ref_color_smoothing(rgba, passes, kind="strict"):
    lib = ref(kind)
    return None if lib is None else _smooth(lib, "ref_color_smoothing", rgba, passes)


# ---- AMaZE demosaic ---------------------------------------------------------------------------------------
def oracle_amaze(mosaic, filters, pm=(1.0, 1.0, 1.0), scratch_mode=1):
    """scratch_mode 0: one scratch carried from tile to tile (= the reference with one thread); 1: zeroed per tile (what
    the CUDA kernel computes); 2: NaN-filled per tile.  Lane 3 is not written (comes back 0)."""
    h, w = mosaic.shape
    src = np.ascontiguousarray(mosaic)
    out = np.zeros((h, w, 4), np.float32)
    f = oracle().orc_amaze_demosaic
    f.restype = C.c_int
    assert f(fptr(out), fptr(src), w, h, C.c_uint32(filters), (C.c_float * 3)(*pm), scratch_mode) == 0
    return out


@recorded(lambda mosaic, filters, pm=(1.0, 1.0, 1.0), kind="strict", threads=1: oracle_amaze(mosaic, filters, pm, 0))
def ref_amaze(mosaic, filters, pm=(1.0, 1.0, 1.0), kind="strict", threads=1):
    lib = ref(kind)
    if lib is None:
        return None
    C.CDLL("libgomp.so.1").omp_set_num_threads(threads)
    oracle().orc_fp_fast_mode()      # FTZ|DAZ on this thread, as the reference's pipe threads have it (darktable.c:877)
    h, w = mosaic.shape
    src = aligned_empty(mosaic.shape)
    src[...] = mosaic
    out = aligned_empty((h, w, 4))
    out[...] = 0
    lib.ref_amaze_demosaic.restype = C.c_int
    lib.ref_amaze_demosaic(fptr(out), fptr(src), w, h, C.c_uint32(filters), (C.c_float * 3)(*pm))
    C.CDLL("libgomp.so.1").omp_set_num_threads(os.cpu_count() or 1)
    return np.array(out)


if RECORDING:
    import atexit
    atexit.register(_save_recordings)
