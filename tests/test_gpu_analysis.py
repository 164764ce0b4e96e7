"""GPU suite: dxb200_compute_mse / dxb200_is_alpha_all_opaque (k_compute_mse, k_mse_finish, k_alpha_opaque) against the reference's
recorded answers and the host emulator, over the case table of tests/analysis_cases.py; error HRESULTs; the determinism contract
(batches, repeats, devices, host versus device variant); a full-size BC7 comparison."""
import ctypes as C

import numpy as np
import pytest

from directxtex_b200 import capi, formats as F, synth
from tests import analysis_cases as AC
from tests import analysis_lib
from tests.analysis_lib import analysis_oracle, analysis_emul  # noqa: F401  (fixtures)
from tests.test_cpu_analysis import check_vs_reference

pytestmark = pytest.mark.gpu
GAMMA = 0x1 | 0x2


def _img(buf, fmt, w, h, pitch=0):
    return capi.make_image(buf.ctypes.data, w, h, fmt, pitch)


def _uses_powf(fa, fb, fl):
    """the gamma flags (given or implied) and the sRGB curve of Decompress on BC*_SRGB data go through powf, which differs by a few
    ulp between CUDA and glibc: those cases agree with the emulator to 1e-6 relative, all others bit for bit"""
    srgb = (29, 91, 93, 72, 75, 78, 99)
    return bool(fl & GAMMA) or fa in srgb or fb in srgb


def gpu_mse(a, fa, b, fb, w, h, fl, pa=0, pb=0):
    hr, mse, mse_v = capi.compute_mse_images([_img(a, fa, w, h, pa)], [_img(b, fb, w, h, pb)], fl)
    return hr, np.concatenate([mse, mse_v[0]]).astype(np.float32)


@pytest.mark.parametrize("case", AC.mse_cases(), ids=lambda c: c[0])
def test_mse_matches_reference_and_emulator(case, analysis_oracle, analysis_emul):
    cid, fa, fb, w, h, fl, pad = case
    a, b = AC.mse_inputs(case)
    hr, want = analysis_oracle.compute_mse(a, fa, b, fb, w, h, fl, full=True)
    assert hr == 0
    pa, pitch_a = AC.padded(a, fa, w, h, pad)
    pb, pitch_b = AC.padded(b, fb, w, h, pad)
    hr, got = gpu_mse(pa, fa, pb, fb, w, h, fl, pitch_a, pitch_b)
    assert hr == 0
    check_vs_reference(got, want)
    hr, em = analysis_emul.compute_mse(pa, fa, pb, fb, w, h, fl, pitch_a, pitch_b)
    if _uses_powf(fa, fb, fl):
        assert np.all(np.abs(got.astype(np.float64) - em) <= 1e-6 * np.abs(em.astype(np.float64)) + 1e-30), (got, em)
    else:
        assert got.tobytes() == em.tobytes(), (got, em)


@pytest.mark.parametrize("case", AC.opaque_cases(), ids=lambda c: c[0])
def test_alpha_scan_matches_reference(case, analysis_oracle, analysis_emul, mirror):
    cid, fmt, w, h, levels, px = case
    hr, want = analysis_oracle.is_alpha_all_opaque(px, fmt, w, h, 1, levels)
    assert hr == 0
    layout = AC.opaque_layout(fmt, w, h, levels)
    scan = capi.is_alpha_all_opaque(px, layout, fmt)
    assert (1 if fmt in AC.NO_ALPHA else int(scan)) == want
    assert int(scan) == analysis_emul.is_alpha_all_opaque(px, layout, fmt)[1]
    # the C++ mirror's ScratchImage::IsAlphaAllOpaque (HasAlpha first, then the scan on the device) answers as the reference's member
    assert mirror.is_alpha_all_opaque(px, fmt, w, h, 1, levels) == (0, want)


@pytest.fixture(scope="module")
def mirror():
    return analysis_lib.Probe(analysis_lib.build_probe(False))


@pytest.mark.parametrize("cid", ["pair_28_28", "bc_98_vs_rgba32f", "flags_80", "size_rgba8_256x256"])
def test_mirror_compute_mse_equals_the_c_abi(cid, mirror):
    case = [c for c in AC.mse_cases() if c[0] == cid][0]
    _, fa, fb, w, h, fl, _ = case
    a, b = AC.mse_inputs(case)
    hr, got = mirror.compute_mse(a, fa, b, fb, w, h, fl)
    assert hr == 0 and got.tobytes() == gpu_mse(a, fa, b, fb, w, h, fl)[1].tobytes()


def test_error_hresults():
    a = np.zeros(64 * 4, np.uint8)
    E_POINTER, E_INVALIDARG, NOT_SUPPORTED = 0x80004003, 0x80070057, 0x80070032
    ok = _img(a, 28, 8, 8)
    null = capi.Image(8, 8, 28, 32, 256, None)
    assert capi.compute_mse_images([null], [ok])[0] == E_POINTER
    assert capi.compute_mse_images([ok], [_img(a, 28, 8, 4)])[0] == E_INVALIDARG               # size mismatch
    assert capi.compute_mse_images([ok], [capi.Image(8, 8, 250, 32, 256, a.ctypes.data)])[0] == E_INVALIDARG      # invalid format
    for f in (27, 130, 103, 111):                                   # typeless, planar (NV12), video (YUY2), palettized / not implemented
        assert capi.compute_mse_images([ok], [capi.Image(8, 8, f, 32, 256, a.ctypes.data)])[0] == NOT_SUPPORTED, f
    assert capi.is_alpha_all_opaque_images([null])[0] == E_POINTER
    assert capi.is_alpha_all_opaque_images([capi.Image(8, 8, 27, 32, 256, a.ctypes.data)])[0] == NOT_SUPPORTED
    assert capi.is_alpha_all_opaque_images([capi.Image(8, 8, 0, 32, 256, a.ctypes.data)])[0] == E_INVALIDARG


def _batch():
    cases = [c for c in AC.mse_cases() if c[0] in ("pair_28_28", "size_rgba8_5x7", "size_rgba8_256x256", "size_rgba8_1x1", "flags_80")]
    return [(c, AC.mse_inputs(c)) for c in cases]


def test_batch_of_mixed_sizes_and_kinds_equals_single_calls():
    items = [(c, ab) for c, ab in _batch()] + [(c, AC.mse_inputs(c)) for c in AC.mse_cases() if c[0] in ("bc_98_vs_rgba32f", "bc_77_vs_71", "size_bc7_5x7")]
    singles = [gpu_mse(a, c[1], b, c[2], c[3], c[4], 0)[1] for c, (a, b) in items]
    hr, mse, mse_v = capi.compute_mse_images([_img(a, c[1], c[3], c[4]) for c, (a, b) in items], [_img(b, c[2], c[3], c[4]) for c, (a, b) in items], 0)
    assert hr == 0
    for i, s in enumerate(singles):
        assert np.concatenate([mse[i:i + 1], mse_v[i]]).tobytes() == s.tobytes(), items[i][0][0]
    again = capi.compute_mse_images([_img(a, c[1], c[3], c[4]) for c, (a, b) in items], [_img(b, c[2], c[3], c[4]) for c, (a, b) in items], 0)
    assert again[1].tobytes() == mse.tobytes() and again[2].tobytes() == mse_v.tobytes()


def test_device_variants_equal_host_variants():
    torch = pytest.importorskip("torch")
    items = [(c, AC.mse_inputs(c)) for c in AC.mse_cases() if c[0] in ("pair_28_28", "bc_98_vs_rgba32f", "bc_77_vs_71", "flags_1", "size_rgba8_256x256")]
    da = [torch.from_numpy(np.ascontiguousarray(a).view(np.uint8).reshape(-1).copy()).cuda() for c, (a, b) in items]
    db = [torch.from_numpy(np.ascontiguousarray(b).view(np.uint8).reshape(-1).copy()).cuda() for c, (a, b) in items]
    out = torch.zeros(5 * len(items), dtype=torch.float32, device="cuda")
    ia = [capi.make_image(t.data_ptr(), c[3], c[4], c[1]) for t, (c, _) in zip(da, items)]
    ib = [capi.make_image(t.data_ptr(), c[3], c[4], c[2]) for t, (c, _) in zip(db, items)]
    stream = torch.cuda.current_stream().cuda_stream
    assert capi.compute_mse_device(ia, ib, 0, out.data_ptr(), C.c_void_p(stream)) == 0
    torch.cuda.synchronize()
    got = out.cpu().numpy().reshape(-1, 5)
    for i, (c, (a, b)) in enumerate(items):
        assert got[i].tobytes() == gpu_mse(a, c[1], b, c[2], c[3], c[4], 0)[1].tobytes(), c[0]
    flag = torch.zeros(1, dtype=torch.int32, device="cuda")
    for cid, fmt, w, h, levels, px in AC.opaque_cases():
        layout = AC.opaque_layout(fmt, w, h, levels)
        t = torch.from_numpy(px.copy()).cuda()
        imgs = [capi.Image(lw, lh, fmt, row, sl, t.data_ptr() + off) for (off, lw, lh, row, sl) in layout]
        assert capi.is_alpha_all_opaque_device(imgs, flag.data_ptr(), C.c_void_p(stream)) == 0
        torch.cuda.synchronize()
        assert int(flag.item()) == int(capi.is_alpha_all_opaque(px, layout, fmt)), cid


def test_full_size_c2_bc7_equals_emulator_and_fp64_bound(emul, analysis_emul):
    """the GPU's BC7 encoding of the C2 image (4096^2 RGBA32F) against its source: GPU and emulator agree bit for bit and mseV is within
    4 ulp of float(fp64 sum of the fp32 squares) / float(w*h)"""
    w = h = 4096
    src = synth.c2_rgba32f(w, h, seed=2)
    blocks = capi.compress(src, w, h, 2, 98)
    mse, mse_v = capi.compute_mse(blocks, 98, src, 2, w, h)
    hr, em = analysis_emul.compute_mse(blocks, 98, src, 2, w, h, 0)
    assert hr == 0 and np.concatenate([[mse], mse_v]).astype(np.float32).tobytes() == em.tobytes()
    dec = emul.decode_blocks(98, blocks, w, h).reshape(-1, 4)
    d = (dec - src.reshape(-1, 4)).astype(np.float32)
    want = ((d * d).astype(np.float32).astype(np.float64).sum(0)).astype(np.float32) / np.float32(w * h)
    assert np.all(np.abs(mse_v.astype(np.float64) - want) <= 4 * np.spacing(np.abs(want)))
    # repeat calls and the bands of a large host image give the same bits
    assert capi.compute_mse(blocks, 98, src, 2, w, h)[1].tobytes() == mse_v.tobytes()


def test_one_versus_two_devices_identical():
    n = capi.lib.dxb200_device_count()
    c = [c for c in AC.mse_cases() if c[0] == "size_rgba8_256x256"][0]
    big = synth.c1_rgba8(4096, 4096, seed=3)
    other = synth.c1_rgba8(4096, 4096, seed=4)
    one = capi.compute_mse(big, 28, other, 28, 4096, 4096)
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    capi.init_devices(list(range(n)))
    two = capi.compute_mse(big, 28, other, 28, 4096, 4096)
    assert one[1].tobytes() == two[1].tobytes() and one[0] == two[0]
    assert c is not None
