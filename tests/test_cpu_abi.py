"""CPU tests: the C ABI library loads and exports every symbol include/b200iop.h declares; integer
CFA phase arithmetic is bit-exact; the product fails loudly without a GPU; the product never
touches oracle/."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

import util

ROOT = util.ROOT


def declared_symbols():
    hdr = open(os.path.join(ROOT, "include", "b200iop.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    return sorted(set(re.findall(r"\b(b200_[a-z0-9_]+)\s*\(", hdr)))


def test_library_exports_every_declared_symbol(built):
    import ansel_b200 as ab
    L = ab.lib()
    names = declared_symbols()
    assert len(names) >= 20
    for n in names:
        assert hasattr(L, n), f"{n} declared in include/b200iop.h but not exported"
    assert L.b200_abi_version() == 1


def test_module_adapters_export_reference_symbol_names(built):
    import ansel_b200.dtsurface as ds
    M = ds.modlib()
    for op in ds.ADAPTED_OPS:
        for fn in ("process", "process_cl", "tiling_callback"):
            assert hasattr(M, f"dt_iop_{op}__{fn}")


def test_no_cuda_device_fails_loudly(built):
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    import ansel_b200 as ab
    L = ab.lib()
    assert L.b200_init(0) == ab.B200_ERR_NODEVICE
    m = util.frame_uniform(64, 64, 1)
    out = np.zeros((64, 64, 4), np.float32)
    piece = ab.make_piece(64, 64, data=ab.demosaic_data())
    assert L.b200_demosaic_process_host(piece, m.ctypes.data, out.ctypes.data) != 0
    assert b"no CUDA device" in L.b200_last_error() or b"CUDA" in L.b200_last_error()
    assert (out == 0).all()
    # every other module: same refusal, nothing computed on the CPU
    rgba = np.zeros((64, 64, 4), np.float32)
    conv = ab.make_conversion(util.MATRIX_CAM_TO_REC2020)
    blob = np.load(os.path.join(util.GOLDEN_DIR, "filmic_data.npz"))["default_v8"]
    fp = ab.filmic_piece(blob, util.profile_pair(util.REC2020_TO_XYZ_D50))
    datas = dict(colorin=ab.colorin_data(conv), colorout=ab.colorout_data(conv), denoiseprofile=ab.denoiseprofile_data(),
                 nlmeans=ab.nlmeans_data(), filmicrgb=fp, diffuse=ab.diffuse_data(), bilat=ab.bilat_data())
    for op, data in datas.items():
        pc = ab.make_piece(64, 64, filters=0, channels=4)
        pc.data, pc.data_size = C.addressof(data), C.sizeof(data)
        out[...] = -3.0
        assert getattr(L, f"b200_{op}_process_host")(pc, rgba.ctypes.data, out.ctypes.data) != 0, op
        assert (out == -3.0).all(), op


def test_pipe_end_modules_fail_loudly_without_a_device(built):
    """rawprepare, temperature, highlights, exposure, gamma, the export conversion: refusal, nothing computed on the CPU"""
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    import ansel_b200 as ab
    L = ab.lib()
    raw = np.full((64, 64), 1000, np.uint16)
    mosaic, rgba = np.zeros((64, 64), np.float32), np.zeros((64, 64, 4), np.float32)
    cases = dict(rawprepare=(ab.rawprepare_data((512,) * 4, (15000,) * 4), raw, 1), temperature=(ab.temperature_data((2, 1, 1.5, 1)), mosaic, 1),
                 highlights=(ab.highlights_data(), mosaic, 1), exposure=(ab.exposure_data(0.0, 0.5), rgba, 4), gamma=(None, rgba, 4))
    for op, (data, src, ch) in cases.items():
        pc = ab.make_piece(64, 64, filters=0x94949494 if ch == 1 else 0, channels=ch, data=data)
        pc.datatype = ab.TYPE_UINT16 if op == "rawprepare" else ab.TYPE_FLOAT
        out = np.full((64, 64, 4), -3.0, np.float32)
        assert getattr(L, f"b200_{op}_process_host")(pc, src.ctypes.data, out.ctypes.data) != 0, op
        assert b"CUDA" in L.b200_last_error() or b"device" in L.b200_last_error(), op
        assert (out == -3.0).all(), op
    pc = ab.make_piece(64, 64, filters=0, channels=4, data=ab.finalscale_data(), out_width=32, out_height=32)
    pc.roi_out.scale = 0.5
    out = np.full((32, 32, 4), -3.0, np.float32)
    assert L.b200_finalscale_process_host(pc, rgba.ctypes.data, out.ctypes.data) != 0 and (out == -3.0).all()
    for op, data in (("flip", ab.FlipData(5)), ("initialscale", ab.finalscale_data())):
        pc = ab.make_piece(64, 64, filters=0, channels=4, data=data)
        out = np.full((64, 64, 4), -3.0, np.float32)
        assert getattr(L, f"b200_{op}_process_host")(pc, rgba.ctypes.data, out.ctypes.data) != 0 and (out == -3.0).all(), op
    cp = ab.channelmixer_piece(util.profile_pair(util.REC2020_TO_XYZ_D50))
    pc = ab.make_piece(64, 64, filters=0, channels=4)
    pc.data, pc.data_size = C.addressof(cp), C.sizeof(cp)
    out = np.full((64, 64, 4), -3.0, np.float32)
    assert L.b200_channelmixerrgb_process_host(pc, rgba.ctypes.data, out.ctypes.data) != 0 and (out == -3.0).all()
    out = np.full((64, 64, 4), 7, np.uint16)
    assert L.b200_export_convert_host(rgba.ctypes.data, out.ctypes.data, 64, 64, ab.EXPORT_UINT16) != 0
    assert (out == 7).all()


def test_pipe_end_tiling_callbacks(built):
    """default_tiling_callback (develop/tiling.c:1423-1463) for rawprepare (TILING_FULL_ROI), temperature, exposure, gamma;
    highlights' own (iop/highlights.c:575-644)"""
    import ansel_b200 as ab
    L = ab.lib()
    t = ab.Tiling()
    piece = ab.make_piece(6000, 4000, data=ab.rawprepare_data((512,) * 4, (15000,) * 4), out_width=5990, out_height=3990)
    L.b200_rawprepare_tiling(piece, t)
    want = np.float32(1.0) + (np.float32(5990) * np.float32(3990)) / (np.float32(6000) * np.float32(4000))
    assert (t.overlap, t.xalign, t.yalign) == (4, 2, 2) and np.float32(t.factor) == want
    piece = ab.make_piece(6000, 4000, filters=9, data=ab.temperature_data((2, 1, 1.5, 1)))
    L.b200_temperature_tiling(piece, t)
    assert (t.overlap, t.xalign, t.yalign, t.factor) == (0, 3, 3, 2.0)
    for op, data in (("exposure", ab.exposure_data()), ("gamma", None), ("channelmixerrgb", None)):
        piece = ab.make_piece(6000, 4000, filters=0, channels=4, data=data)
        getattr(L, f"b200_{op}_tiling")(piece, t)
        assert (t.overlap, t.xalign, t.yalign, t.factor) == (0, 1, 1, 2.0), op
    piece = ab.make_piece(6000, 4000, filters=0, channels=4, data=ab.finalscale_data(), out_width=3000, out_height=2000)
    L.b200_finalscale_tiling(piece, t)
    assert (t.overlap, t.xalign, t.yalign, t.factor) == (4, 1, 1, 1.25)      # IOP_FLAGS_TILING_FULL_ROI
    piece = ab.make_piece(6000, 4000, data=ab.highlights_data(ab.HIGHLIGHTS_LCH))
    L.b200_highlights_tiling(piece, t)
    assert (t.overlap, t.xalign, t.yalign, t.factor) == (1, 2, 2, 2.0)
    d = ab.highlights_data(ab.HIGHLIGHTS_HARMONIC)
    piece = ab.make_piece(6000, 4000, data=d)
    L.b200_highlights_tiling(piece, t)
    # scales = 8: final_radius = 256 / 4 = 64 -> 6 scales -> radius 64 -> overlap 64 * 1.5 / 4
    assert (t.overlap, t.xalign, t.yalign) == (24, 2, 2) and abs(t.factor - 16.0) < 1e-6 and abs(t.factor_cl - 20.0) < 1e-6


def test_piece_datatype_fills_padding(built):
    """b200_piece_t gained `datatype` where the compiler had padding: size and the offsets of its neighbours are unchanged"""
    import ansel_b200 as ab
    import ansel_b200.dtsurface as ds
    assert C.sizeof(ab.Piece) == 184 and ab.Piece.devid.offset == 160 and ab.Piece.datatype.offset == 164 and ab.Piece.data.offset == 168
    assert ds.modlib().b200_dt_surface_probe(10) == C.sizeof(ab.Piece)


def _shift_dcraw(filters, x, y):
    """ColorFilterArray::shiftDcrawFilter (rawspeed ColorFilterArray.cpp:143-170) in Python ints."""
    if abs(x) & 1:
        for n in range(8):
            i, j = n * 4, n * 4 + 2
            t = ((filters >> i) ^ (filters >> j)) & 3
            filters ^= (t << i) | (t << j)
    if y == 0:
        return filters
    y *= 4
    y = y % 32 if y >= 0 else 32 - ((-y) % 32)
    if y != 0 and y != 32:
        filters = ((filters >> y) | (filters << (32 - y))) & 0xFFFFFFFF
    return filters


def test_roi_filters_and_fc_bit_exact(built):
    import ansel_b200 as ab
    L = ab.lib()
    rng = np.random.default_rng(3)
    words = list(util.BAYER.values()) + [int(v) for v in rng.integers(1, 2 ** 32, 50)]
    for f in words:
        for x in (-5, -2, -1, 0, 1, 2, 3, 7, 1001):
            for y in (-9, -8, -1, 0, 1, 2, 7, 8, 9, 4003):
                assert L.b200_roi_filters(f, x, y) == _shift_dcraw(f, x, y), (hex(f), x, y)
        for r in range(16):
            for c in range(4):
                assert L.b200_fc(r, c, f) == (f >> ((((r << 1) & 14) + (c & 1)) << 1)) & 3
    assert L.b200_roi_filters(0, 1, 1) == 0 and L.b200_roi_filters(9, 1, 1) == 9
    f = util.BAYER["RGGB"]
    assert [L.b200_fc(0, 0, f), L.b200_fc(0, 1, f), L.b200_fc(1, 0, f), L.b200_fc(1, 1, f)] == [0, 1, 1, 2]
    # shifting the word is the same as reading the pattern at the shifted origin
    for x in range(4):
        for y in range(4):
            g = L.b200_roi_filters(f, x, y)
            for r in range(4):
                for c in range(4):
                    assert L.b200_fc(r, c, g) == L.b200_fc(r + y, c + x, f)


def test_tiling_callbacks_match_reference_contract(built):
    import ansel_b200 as ab
    L = ab.lib()
    t = ab.Tiling()
    piece = ab.make_piece(6000, 4000, data=ab.demosaic_data(ab.DEMOSAIC_RCD))
    L.b200_demosaic_tiling(piece, t)
    assert (t.overlap, t.xalign, t.yalign) == (10, 2, 2) and abs(t.factor - 3.0) < 1e-6  # demosaic.c:1972-1982
    conv = ab.make_conversion(util.MATRIX_CAM_TO_REC2020)
    piece = ab.make_piece(6000, 4000, filters=0, channels=4, data=ab.colorin_data(conv))
    L.b200_colorin_tiling(piece, t)
    assert (t.overlap, t.xalign, t.yalign, t.factor) == (0, 1, 1, 2.0)  # tiling.c:1423-1440
    piece = ab.make_piece(6000, 4000, filters=0, channels=4, data=ab.diffuse_data(radius=8))
    L.b200_diffuse_tiling(piece, t)
    assert (t.overlap, t.xalign, t.yalign) == (32, 1, 1) and abs(t.factor - (6.0625 + 5)) < 1e-6  # diffuse.c:585-610: 5 scales
    piece = ab.make_piece(6000, 4000, filters=0, channels=4, data=ab.nlmeans_data(radius=2.0))
    L.b200_nlmeans_tiling(piece, t)
    assert (t.overlap, t.xalign, t.yalign) == (2 + 7, 1, 1) and abs(t.factor - 4.0) < 1e-6    # nlmeans.c:400-414
    piece = ab.make_piece(6000, 4000, filters=0, channels=4, data=ab.denoiseprofile_data(ab.DENOISE_NLMEANS, radius=1, nbhood=7))
    L.b200_denoiseprofile_tiling(piece, t)
    assert t.overlap == 1 + 7                                                                  # denoiseprofile.c:803-811


def test_abi_struct_layout_matches_reference_headers(built):
    """include/b200iop.h mirrors; oracle/_ref exports the reference compiler's view of the same structs."""
    import ansel_b200 as ab
    assert C.sizeof(ab.Roi) == 24 and C.sizeof(ab.Tiling) == 32 and C.sizeof(ab.DemosaicData) == 128
    assert util.ref_size_t("ref_sizeof_roi") == C.sizeof(ab.Roi)
    import ansel_b200.dtsurface as ds
    ds.modlib()
    assert util.ref_size_t("ref_sizeof_dsc") == C.sizeof(ds.BufferDsc)
    for name, field in (("ref_offsetof_dsc_filters", ds.BufferDsc.filters), ("ref_offsetof_dsc_processed_maximum", ds.BufferDsc.processed_maximum),
                        ("ref_offsetof_dsc_temperature_coeffs", ds.BufferDsc.temperature_coeffs)):
        assert util.ref_size_t(name) == field.offset, name


def test_product_never_references_the_oracle():
    """Only tests/, __graft_entry__.smoke() and bench.py's CPU legs may touch oracle/."""
    bad = []
    for base, _, files in os.walk(os.path.join(ROOT, "ansel_b200")):
        for fn in files:
            if fn.endswith((".py", ".c", ".h", ".cu", ".cuh")):
                txt = open(os.path.join(base, fn), errors="replace").read()
                code = re.sub(r"//[^\n]*|/\*.*?\*/", "", txt, flags=re.S)  # comments may cite the oracle; code may not
                if re.search(r"#include[^\n]*oracle|liboracle|libref_|dlopen[^\n]*oracle|CDLL[^\n]*oracle|\borc_[a-z_]+\s*\(", code):
                    bad.append(os.path.join(base, fn))
    assert not bad, bad
    out = subprocess.run(["ldd", os.path.join(ROOT, "ansel_b200", "libb200iop.so")], capture_output=True, text=True).stdout
    assert "oracle" not in out


def test_band_grid_follows_the_demosaic_method(built):
    """RCD bands cut on its 94-row block grid (bit-identical to the untiled frame); AMaZE bands are tiling.c tiles"""
    import ansel_b200 as ab
    L = ab.lib()
    g, h, a = C.c_int(), C.c_int(), C.c_int()
    L.b200_demosaic_band_grid(None, C.byref(g), C.byref(h), C.byref(a))
    assert (g.value, h.value, a.value) == (94, 9, 2)
    for method, want in ((ab.DEMOSAIC_RCD, (94, 9, 2)), (ab.DEMOSAIC_AMAZE, (1, 5, 2))):
        d = ab.demosaic_data(method=method)
        piece = ab.make_piece(640, 480, filters=0x94949494, channels=1, data=d)
        L.b200_demosaic_band_grid(C.byref(piece), C.byref(g), C.byref(h), C.byref(a))
        assert (g.value, h.value, a.value) == want


def test_filmic_tiling_through_the_adapter_with_reconstruction_live(built):
    """tiling_callback(), filmicrgb.c:2668-2704: the reference's own piece->data (sizeof(dt_iop_filmicrgb_data_t), not the
    flattened piece the library entry points take) must report 9 buffers and 2^scales overlap while hl_deprecated == 0"""
    import ansel_b200 as ab
    import ansel_b200.dtsurface as ds
    g = np.load(os.path.join(util.GOLDEN_DIR, "filmic_reconstruct.npz"))
    blob = np.ascontiguousarray(g["data_default_poisson"], np.uint8)
    fdata = (C.c_uint8 * blob.size).from_buffer_copy(blob.tobytes())
    assert blob.size == 832
    piece = ds.make_piece_iop("filmicrgb", 6000, 4000, fdata, channels_in=4, channels_out=4)
    work, export = util.profile_pair(util.REC2020_TO_XYZ_D50), util.profile_pair(util.SRGB_TO_XYZ_D50)
    pipe = ds.make_pipe(devid=-1, work_profile=ds.profile_info(*work), output_profile=ds.profile_info(*export))
    t = ab.Tiling()
    ds.modlib().dt_iop_filmicrgb__tiling_callback(piece.module, C.byref(pipe), C.byref(piece), C.byref(t))
    f = util.oracle().orc_filmic_reconstruct_scales
    f.restype = C.c_int
    assert t.factor == 9.0 and t.overlap == 1 << f(C.c_float(1.0), C.c_double(1.0), 6000, 4000)
    # ... and a pointwise module again once the reconstruction is deprecated (every new edit)
    blob2 = np.ascontiguousarray(np.load(os.path.join(util.GOLDEN_DIR, "filmic_data.npz"))["default_v8"], np.uint8)
    fdata2 = (C.c_uint8 * blob2.size).from_buffer_copy(blob2.tobytes())
    piece2 = ds.make_piece_iop("filmicrgb", 6000, 4000, fdata2, channels_in=4, channels_out=4)
    ds.modlib().dt_iop_filmicrgb__tiling_callback(piece2.module, C.byref(pipe), C.byref(piece2), C.byref(t))
    assert (t.factor, t.overlap) == (2.0, 0)


def test_packed_fp32_is_never_contracted_in_the_nlm_group_kernel(built):
    """ptxas turns a packed multiply feeding a packed add into FFMA2 even under --fmad=false (nlm_group.cuh): the only FFMA2
    allowed in the group kernels are the two of Markstein's division per owned pixel pair (the accumulation loop exists twice:
    chunks in the interior of the frame, and patches that cover a chunk at its edge), and only in the variants using it"""
    so = os.path.join(ROOT, "ansel_b200", "libb200iop.so")
    r = subprocess.run(["cuobjdump", "-sass", so], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-300:]
    seen = 0
    for body in re.split(r"\n\s*Function : ", r.stdout)[1:]:
        name = body.split("\n", 1)[0]
        m = re.search(r"nlm_group_kernelILi(\d)ELi(\d+)ELb([01])ELb([01])ELb([01])ELi(\d)E", name)
        if not m:
            continue
        seen += 1
        divc, kp = m.group(5) == "1", int(m.group(6))
        assert len(re.findall(r"\bFFMA2\b", body)) == (4 * kp if divc else 0), name
        assert len(re.findall(r"\bFMUL2\b", body)) > 0 and len(re.findall(r"\bFADD2\b", body)) > 0, name
    assert seen >= 12


def test_packed_fp32_is_never_contracted_in_the_nlm_pipe_kernel(built):
    """the same for the pipelined kernel: the accumulation of a patch is inlined four times (two patches of a pair, in the loop of interior
    chunks and in the loop of edge chunks) -- six times where the half-height slots are compiled in (radius 1, shape 0) -- with Markstein's two
    FFMA2 per owned pixel pair each, 9 pairs per thread"""
    so = os.path.join(ROOT, "ansel_b200", "libb200iop.so")
    r = subprocess.run(["cuobjdump", "-sass", so], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-300:]
    seen = 0
    for body in re.split(r"\n\s*Function : ", r.stdout)[1:]:
        name = body.split("\n", 1)[0]
        m = re.search(r"nlm_pipe_kernelILi(\d)ELb([01])ELb([01])ELb([01])ELi(\d)E", name)
        if not m:
            continue
        seen += 1
        divc, kp = m.group(4) == "1", 9
        inlined = 6 if (m.group(1) == "1" and m.group(5) == "0") else 4
        assert len(re.findall(r"\bFFMA2\b", body)) == (2 * inlined * kp if divc else 0), name
        assert len(re.findall(r"\bFMUL2\b", body)) > 0 and len(re.findall(r"\bFADD2\b", body)) > 0, name
    assert seen >= 12


def test_markesteijn_divides_by_three(built):
    """nvcc rewrites `x / 3.f` into `x * 0.33333334f` under -ftz=true even with -prec-div=true (1-ulp differences in a tenth of the pixels on
    the device, none in the CPU emulation): the kernel's division by 3 goes through div.rn.ftz.f32, which the rewrite does not see"""
    so = os.path.join(ROOT, "ansel_b200", "libb200iop.so")
    r = subprocess.run(["cuobjdump", "-sass", "-fun", "markesteijn_tiles_kernel", so], capture_output=True, text=True)
    body = r.stdout
    if "markesteijn_tiles_kernel" not in body:      # cuobjdump wants the mangled name on some versions: take the whole listing
        r = subprocess.run(["cuobjdump", "-sass", so], capture_output=True, text=True)
        body = [b for b in re.split(r"\n\s*Function : ", r.stdout) if b.startswith("_Z") and "markesteijn_tiles_kernel" in b.split("\n", 1)[0]][0]
    assert not re.search(r"FMUL(\.FTZ)? R\d+, R\d+, 0\.33333", body)
    assert len(re.findall(r"MUFU\.RCP", body)) >= 4
