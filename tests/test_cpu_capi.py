"""CPU suite, part 2: the C-ABI library loads and exports exactly what include/dxtex_b200.h declares, host-side
logic (pitches, mip counts, argument validation, HRESULTs) matches the reference, and compute entry points fail
loudly when no CUDA device is present (no CPU fallback)."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from directxtex_b200 import capi, formats as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_symbols():
    txt = open(os.path.join(ROOT, "include", "dxtex_b200.h")).read()
    return sorted(set(re.findall(r"\b(dxb200_[a-z_0-9]+)\s*\(", txt)))


def test_library_exports_every_declared_symbol():
    syms = header_symbols()
    assert len(syms) >= 18
    for s in syms:
        assert hasattr(capi.lib, s), s
    assert sorted(capi.SYMBOLS) == syms


def test_version_and_device_count():
    assert b"sm_100a" in capi.lib.dxb200_version()
    assert capi.lib.dxb200_device_count() >= 0


def test_compute_pitch_matches_reference(oracle):
    for fmt in sorted(set(F.BYTES_PER_PIXEL) | set(F.BLOCK_BYTES)):
        for (w, h) in [(1, 1), (5, 7), (256, 256), (4096, 4096), (17, 3)]:
            r, s = C.c_size_t(), C.c_size_t()
            hr = capi.lib.dxb200_compute_pitch(fmt, w, h, r, s)
            hr_ref, rr, sr = oracle.compute_pitch(fmt, w, h)
            assert hr == 0 and hr_ref == 0
            assert (r.value, s.value) == (rr, sr) == F.compute_pitch(fmt, w, h), (fmt, w, h)
    r, s = C.c_size_t(), C.c_size_t()
    assert F.hr_u32(capi.lib.dxb200_compute_pitch(3, 4, 4, r, s)) == F.HRESULT_E_NOT_SUPPORTED     # R32G32B32A32_UINT: not implemented


def test_calculate_mip_levels():
    for (w, h, want) in [(4096, 4096, 13), (2048, 2048, 12), (1024, 1024, 11), (1, 1, 1), (5, 3, 3), (256, 16, 9)]:
        n = C.c_size_t(0)
        assert capi.lib.dxb200_calculate_mip_levels(w, h, n) == 0 and n.value == want == F.count_mips(w, h)
    n = C.c_size_t(14)
    assert F.hr_u32(capi.lib.dxb200_calculate_mip_levels(4096, 4096, n)) == F.E_INVALIDARG


def test_mip_chain_layout_matches_reference(oracle):
    for fmt in (28, 2, 10, 61):
        for (w, h) in [(64, 64), (32, 8), (17, 13), (1, 7)]:
            hr, nl, tot, levels = oracle.mipchain_layout(fmt, w, h, 0)
            assert hr == 0
            layout, total = F.mip_chain_layout(fmt, w, h, 0)
            assert total == tot and len(layout) == nl
            for i, (o, lw, lh, row, sl) in enumerate(layout):
                assert [o, lw, lh, row] == levels[i]


def _img(arr, w, h, fmt):
    return capi.make_image(arr.ctypes.data, w, h, fmt)


def test_argument_validation_hresults():
    """same error codes as CompressEx / ConvertEx argument checks (DirectXTexCompress.cpp:671-676, DirectXTexConvert.cpp:5113-5125)"""
    a = np.zeros((8, 8, 4), np.uint8)
    out = np.zeros(64, np.uint8)
    L = capi.lib
    s = capi.images([_img(a, 8, 8, 28)])
    d = capi.images([capi.Image(8, 8, 71, 16, 32, out.ctypes.data)])
    assert F.hr_u32(L.dxb200_compress(None, 1, 71, 0, 0.5, 1.0, d)) == F.E_INVALIDARG
    assert F.hr_u32(L.dxb200_compress(s, 0, 71, 0, 0.5, 1.0, d)) == F.E_INVALIDARG
    assert F.hr_u32(L.dxb200_compress(s, 1, 28, 0, 0.5, 1.0, d)) == F.E_INVALIDARG            # destination not a BC format
    sbc = capi.images([capi.Image(8, 8, 71, 16, 32, a.ctypes.data)])
    assert F.hr_u32(L.dxb200_compress(sbc, 1, 77, 0, 0.5, 1.0, d)) == F.E_INVALIDARG          # source already compressed
    snull = capi.images([capi.Image(8, 8, 28, 32, 256, None)])
    assert F.hr_u32(L.dxb200_compress(snull, 1, 71, 0, 0.5, 1.0, d)) == F.E_POINTER
    suint = capi.images([capi.Image(8, 8, 30, 32, 256, a.ctypes.data)])                        # R8G8B8A8_UINT
    assert F.hr_u32(L.dxb200_compress(suint, 1, 71, 0, 0.5, 1.0, d)) == F.HRESULT_E_NOT_SUPPORTED
    dbad = capi.images([capi.Image(4, 8, 71, 8, 16, out.ctypes.data)])
    assert F.hr_u32(L.dxb200_compress(s, 1, 71, 0, 0.5, 1.0, dbad)) == F.E_FAIL               # size mismatch (:800-804)
    dc = capi.images([capi.Image(8, 8, 28, 32, 256, out.ctypes.data)])
    assert F.hr_u32(L.dxb200_convert(s, 1, 28, 0, 0.5, dc)) == F.E_INVALIDARG                  # same format
    assert F.hr_u32(L.dxb200_convert(s, 1, 71, 0, 0.5, d)) == F.E_INVALIDARG                   # BC destination
    o2 = np.zeros(8 * 8 * 16, np.uint8)
    d2 = capi.images([capi.Image(8, 8, 2, 128, 1024, o2.ctypes.data)])
    assert F.hr_u32(L.dxb200_convert(s, 1, 2, 0x40000, 0.5, d2)) == F.HRESULT_E_NOT_SUPPORTED                # unknown dither mode bit
    chain = capi.images([_img(a, 8, 8, 28), capi.Image(4, 4, 28, 16, 64, out.ctypes.data)])
    assert F.hr_u32(L.dxb200_generate_mipmaps(chain, 1, 1, 0)) == F.E_INVALIDARG
    assert F.hr_u32(L.dxb200_generate_mipmaps(chain, 1, 5, 0)) == F.E_INVALIDARG               # more levels than the size allows
    odd = capi.images([_img(a, 6, 8, 28), capi.Image(3, 4, 28, 12, 48, out.ctypes.data)])
    assert F.hr_u32(L.dxb200_generate_mipmaps(odd, 1, 2, F.TEX_FILTER_BOX)) == F.E_FAIL        # box needs powers of two (:1005-1006)
    # Resize argument checking (DirectXTexResize.cpp:318-319, 875-879)
    r53 = capi.images([capi.Image(5, 3, 28, 20, 60, out.ctypes.data)])
    assert F.hr_u32(L.dxb200_resize(s, 1, F.TEX_FILTER_BOX, r53)) == F.E_FAIL                  # box is 2:1 only
    assert F.hr_u32(L.dxb200_resize(s, 0, 0, r53)) == F.E_INVALIDARG
    bc = capi.images([capi.Image(8, 8, 71, 16, 32, out.ctypes.data)])
    assert F.hr_u32(L.dxb200_resize(bc, 1, 0, bc)) == F.HRESULT_E_NOT_SUPPORTED                # compressed source
    wrongfmt = capi.images([capi.Image(4, 4, 2, 64, 256, out.ctypes.data)])
    assert F.hr_u32(L.dxb200_resize(s, 1, 0, wrongfmt)) == F.E_INVALIDARG                      # Resize never converts


def test_compute_entry_points_fail_loudly_without_gpu():
    if capi.lib.dxb200_device_count() > 0:
        pytest.skip("a CUDA device is present")
    a = np.zeros((8, 8, 4), np.uint8)
    with pytest.raises(capi.DxTexError) as e:
        capi.compress(a, 8, 8, 28, 71)
    assert e.value.hr == F.E_FAIL                    # no silent CPU path
    with pytest.raises(capi.DxTexError):
        capi.convert(a, 8, 8, 28, 2)
    with pytest.raises(capi.DxTexError):
        capi.generate_mipmaps(a, 8, 8, 28)
    with pytest.raises(capi.DxTexError):
        capi.resize(a, 8, 8, 28, 5, 3)
    with pytest.raises(capi.DxTexError):
        capi.premultiply_alpha(a, 8, 8, 28)


def test_options_round_trip_and_reject_unknown_ids():
    """dxb200_set_option / dxb200_get_option (no device needed): the BC7 feed option keeps what is set, maps out-of-range values to the
    automatic mode (4), and unknown option ids answer E_INVALIDARG / -1; the TMA launch counter starts at zero on a box without a GPU."""
    L = capi.lib
    before = L.dxb200_get_option(capi.OPT_BC7_FEED)
    assert before in (0, 1, 2, 3, 4)
    try:
        for v in (0, 1, 2, 3, 4):
            assert L.dxb200_set_option(capi.OPT_BC7_FEED, v) == 0 and L.dxb200_get_option(capi.OPT_BC7_FEED) == v
        assert L.dxb200_set_option(capi.OPT_BC7_FEED, 99) == 0 and L.dxb200_get_option(capi.OPT_BC7_FEED) == 4
        assert L.dxb200_set_option(capi.OPT_BC7_FEED, -5) == 0 and L.dxb200_get_option(capi.OPT_BC7_FEED) == 4
    finally:
        L.dxb200_set_option(capi.OPT_BC7_FEED, before)
    assert F.hr_u32(L.dxb200_set_option(12345, 1)) == 0x80070057
    assert L.dxb200_get_option(12345) == -1
    assert capi.tma_launch_count() >= 0
