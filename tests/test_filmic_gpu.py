"""GPU parity: filmic rgb (AgX family) against the oracle, bit for bit on all four lanes.  The oracle is
itself bit-identical to the reference's pixel functions cut verbatim from filmicrgb.c; piece->data comes
from the reference's own commit_params() when oracle/_ref is present, else from the committed blobs."""
import os

import numpy as np
import pytest

import util

pytestmark = pytest.mark.gpu

WORK = util.profile_pair(util.REC2020_TO_XYZ_D50)
EXPORT = util.profile_pair(util.SRGB_TO_XYZ_D50)
CASES = {"default_v8": {}, "no_bleach": dict(version=5), "high_bleach_hue": dict(version=8, saturation=60.0),
         "poly_curves": dict(shadows=0, highlights=1), "rational_curves": dict(shadows=2, highlights=2, contrast=1.5),
         "wide_dr_gamma22": dict(white_point_source=6.0, black_point_source=-10.0, output_power=2.2)}


def same_bits(a, b):
    return (a.view(np.uint32) == b.view(np.uint32)) | (np.isnan(a) & np.isnan(b))


def data_blob(name):
    """dt_iop_filmicrgb_data_t for a case: the golden copy, checked against the reference's commit_params()."""
    g = np.load(os.path.join(util.GOLDEN_DIR, "filmic_data.npz"))
    live = util.ref_filmic_commit(util.filmic_default_params(**CASES[name]))
    assert (live == g[name]).all(), "committed filmic_data.npz is stale"
    return g[name]


def cuda_filmic(img, blob, export=EXPORT, host=False, mask_display=0, iscale=1.0, roi_scale=1.0, buf=None):
    import torch
    import ansel_b200 as ab
    import ctypes as C
    ab.init()
    h, w = img.shape[:2]
    fp = ab.filmic_piece(blob, WORK, export)
    piece = ab.make_piece(w, h, filters=0, channels=4, devid=0, scale=roi_scale)
    piece.data = C.addressof(fp)
    piece.data_size = C.sizeof(fp)
    piece.mask_display = mask_display
    piece.iscale = iscale
    if buf:
        piece.buf_in_width, piece.buf_in_height = buf
    if host:
        out = np.zeros_like(img)
        ab.check(ab.lib().b200_filmicrgb_process_host(piece, img.ctypes.data, out.ctypes.data))
        return out
    d_in = torch.from_numpy(np.ascontiguousarray(img)).cuda()
    d_out = torch.zeros_like(d_in)
    ab.check(ab.lib().b200_filmicrgb_process_dev(piece, d_in.data_ptr(), d_out.data_ptr(), torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    return d_out.cpu().numpy()


@pytest.mark.parametrize("export", [True, False])
@pytest.mark.parametrize("name", list(CASES))
def test_filmic_agx_bit_exact(built, name, export):
    img = util.hdr_rgba(900, 611, 2)
    blob = data_blob(name)
    e = EXPORT if export else None
    got = cuda_filmic(img, blob, e)
    want = util.oracle_filmic_agx(img, blob, WORK, e)
    bad = ~same_bits(got, want)
    assert not bad.any(), f"{int(bad.sum())} floats differ, first {np.argwhere(bad)[:4].tolist()}"
    assert np.isfinite(got[..., :3]).all() and got[..., :3].min() >= 0.0


def test_filmic_host_entry_and_alpha(built):
    import ansel_b200 as ab
    import ctypes as C
    img = util.hdr_rgba(320, 200, 3)
    blob = data_blob("default_v8")
    a, b = cuda_filmic(img, blob), cuda_filmic(img, blob, host=True)
    assert same_bits(a, b).all()
    c = cuda_filmic(img, blob, mask_display=1)
    assert (c[..., 3] == img[..., 3]).all() and same_bits(c[..., :3], a[..., :3]).all()


def test_filmic_45mp_matches_oracle(built):
    w, h = util.SIZE_45MP
    img = util.hdr_rgba(w, h, util.SEEDS[0])
    blob = data_blob("default_v8")
    got = cuda_filmic(img, blob)
    want = util.oracle_filmic_agx(img, blob, WORK, EXPORT)
    assert same_bits(got, want).all()


# ---- the colour sciences before AgX ("v3 (2019)" .. "v7 (2023)") ---------------------------------------------------
def legacy_cases():
    g = np.load(os.path.join(util.GOLDEN_DIR, "filmic_legacy.npz"))
    return g, sorted(k[5:] for k in g.files if k.startswith("data_"))


@pytest.mark.parametrize("export", [True, False])
def test_filmic_legacy_bit_exact(built, export):
    """every committed data block (versions 0..4, several norms) on a fresh scene-referred frame, all four lanes"""
    g, tags = legacy_cases()
    img = util.hdr_rgba(700, 467, 12)
    for tag in tags:
        blob = g["data_" + tag]
        got = cuda_filmic(img, blob, EXPORT if export else None)
        want = util.oracle_filmic_legacy(img, blob, WORK, EXPORT if export else None)
        assert same_bits(got, want).all(), tag


def test_filmic_legacy_golden_and_host(built):
    g, tags = legacy_cases()
    for tag in tags:
        got = cuda_filmic(g["img"], g["data_" + tag], EXPORT, host=True)
        lanes = 3 if tag in ("v0_n0", "v1_n0") else 4          # split v1..v3 leave lane 3 as found; here: the input's alpha
        assert same_bits(got[..., :lanes], g["out_" + tag][..., :lanes]).all(), tag


def legacy_live_blobs():
    return {(version, pc): util.ref_filmic_commit(util.filmic_default_params(version=version, preserve_color=pc, saturation=-15.0, shadows=0, highlights=2))
            for version in range(5) for pc in range(6)}


def test_filmic_legacy_all_norms_live(built):
    """every version x norm x parameter set from the reference's own commit_params()"""
    img = util.hdr_rgba(320, 200, 3)
    for (version, pc), blob in legacy_live_blobs().items():
        assert same_bits(cuda_filmic(img, blob, EXPORT), util.oracle_filmic_legacy(img, blob, WORK, EXPORT)).all(), (version, pc)
