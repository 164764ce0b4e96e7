"""GPU suite: the CUDA path (through the C ABI) against the oracle = the unmodified reference sources.
Bit-exact for BC1-BC5, Convert and the mip filters; BC7 within the stated MSE tolerance and bit-identical
to the host lock-step emulator of the same source."""
import ctypes as C

import numpy as np
import pytest

from directxtex_b200 import capi, formats as F, synth
from tests import golden_util, oracle_lib, tolerance
from tests.oracle_lib import same, same_concat

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module", autouse=True)
def _init():
    assert capi.lib.dxb200_init(0) == 0


def test_bc15_golden():
    n0 = capi.launch_count()
    for name, src, meta, exp in golden_util.cases("compress_"):
        w, h, sf, df, flags = (int(v) for v in meta)
        got = capi.compress(src, w, h, sf, df, flags)
        assert same(got, exp), name
    assert capi.launch_count() > n0          # the CUDA kernels really ran


def test_config1_bc1_matches_reference_hash():
    img = synth.c1_rgba8(256, 256)
    got = capi.compress(img, 256, 256, 28, 71)
    assert same(got, golden_util.load()["config1_bc1_out"])


@pytest.mark.parametrize("df", [71, 74, 77, 80, 81, 83, 84])
def test_bc15_vs_oracle_random(oracle, df):
    rng = np.random.default_rng(200 + df)
    for (w, h, sf) in [(256, 128, 28), (31, 17, 28), (1, 1, 28), (2, 3, 28), (5, 7, 2), (64, 64, 2), (48, 24, 10),
                       (128, 32, 61), (16, 16, 31), (20, 12, 41), (36, 20, 87), (12, 12, 11)]:
        src = oracle_lib.random_image(sf, w, h, rng)
        for flags in (0, F.TEX_COMPRESS_UNIFORM, F.TEX_COMPRESS_DITHER, F.TEX_COMPRESS_PARALLEL):
            hr, want = oracle.compress(src, w, h, sf, df, flags & ~F.TEX_COMPRESS_PARALLEL)
            got = capi.compress(src, w, h, sf, df, flags)
            assert hr == 0 and same(got, want), (w, h, sf, df, hex(flags))


def test_bc1_threshold_and_structured(oracle):
    img = synth.c1_rgba8(128, 128, seed=5)
    for thr in (0.0, 0.25, 0.5, 0.75, 1.0):
        hr, want = oracle.compress(img, 128, 128, 28, 71, 0, threshold=thr)
        got = capi.compress(img, 128, 128, 28, 71, 0, threshold=thr)
        assert hr == 0 and same(got, want), thr


def test_compress_array_batch(oracle):
    rng = np.random.default_rng(9)
    srcs = [oracle_lib.random_image(28, 40, 24, rng) for _ in range(7)]
    outs = capi.compress_array(srcs, 40, 24, 28, 77)
    for s, o in zip(srcs, outs):
        hr, want = oracle.compress(s, 40, 24, 28, 77)
        assert hr == 0 and same(o, want)


def test_bc7_bc6h_array_batch_equals_single_images(emul):
    """BC7 / BC6H encode two consecutive blocks per warp over the whole batch, so a pair can straddle two images (15
    blocks per image here); the halves are independent, so every image must equal its single-image (emulator) result."""
    rng = np.random.default_rng(19)
    w, h = 20, 12
    srcs = [rng.random((h, w, 4), dtype=np.float32) for _ in range(5)]
    srcs[2][..., 3] = 1.0
    for dfmt in (98, 95):
        outs = capi.compress_array(srcs, w, h, 2, dfmt)
        for s_, o in zip(srcs, outs):
            he, want = emul.compress(s_, w, h, 2, dfmt)
            assert he == 0 and same(o, want), dfmt


def test_convert_golden_and_random(oracle):
    for name, src, meta, exp in golden_util.cases("convert_"):
        w, h, sf, df, fl = (int(v) for v in meta)
        got = capi.convert(src, w, h, sf, df, fl)
        assert same(got, exp), name
    rng = np.random.default_rng(4)
    for (sf, df) in [(61, 41), (41, 61), (28, 2), (2, 28), (10, 28), (2, 10), (28, 87)]:
        src = oracle_lib.random_image(sf, 257, 63, rng)
        hr, want = oracle.convert(src, 257, 63, sf, df)
        got = capi.convert(src, 257, 63, sf, df)
        assert hr == 0 and same(got, want), (sf, df)


def test_convert_ordered_dither(oracle):
    """TEX_FILTER_DITHER (ordered 4x4 matrix, StoreScanlineDither): bit-exact for every destination format with a dither case,
    including a host-staged image that is split into several bands (the matrix phase must survive the split)."""
    rng = np.random.default_rng(31)
    for sf in (2, 10, 28):
        for df in (11, 13, 24, 28, 29, 31, 35, 37, 49, 51, 56, 58, 61, 63, 65, 87, 88, 91, 93, 41):
            if sf == df:
                continue
            src = oracle_lib.random_image(sf, 37, 9, rng)
            hr, want = oracle.convert(src, 37, 9, sf, df, F.TEX_FILTER_DITHER)
            got = capi.convert(src, 37, 9, sf, df, F.TEX_FILTER_DITHER)
            assert hr == 0 and same(got, want), (sf, df)
    src = rng.random((1102, 2048, 4), dtype=np.float32)
    hr, want = oracle.convert(src, 2048, 1102, 2, 28, F.TEX_FILTER_DITHER)
    got = capi.convert(src, 2048, 1102, 2, 28, F.TEX_FILTER_DITHER)
    assert hr == 0 and same(got, want)


def test_convert_error_diffusion_dither(oracle):
    """TEX_FILTER_DITHER_DIFFUSION (Floyd-Steinberg, serpentine): serial over an image, one GPU thread per image; bit-exact,
    including the reference's behaviour of adding store-order errors to the un-swizzled source for BGR formats."""
    rng = np.random.default_rng(37)
    for fl in (F.TEX_FILTER_DITHER_DIFFUSION, F.TEX_FILTER_DITHER | F.TEX_FILTER_DITHER_DIFFUSION):
        for sf, df in [(2, 28), (2, 87), (2, 88), (10, 24), (2, 11), (2, 13), (28, 61), (2, 31), (2, 49), (2, 65), (28, 10)]:
            for (w, h) in [(37, 9), (1, 5), (64, 64)]:
                src = oracle_lib.random_image(sf, w, h, rng)
                hr, want = oracle.convert(src, w, h, sf, df, fl)
                got = capi.convert(src, w, h, sf, df, fl)
                assert hr == 0 and same(got, want), (sf, df, w, h, hex(fl))


def test_convert_exhaustive_small_domains(oracle):
    """every value of the 8/16-bit scalar formats (they use a 3-op exact division instead of an IEEE divide)"""
    for sf, dtype, n in ((61, np.uint8, 256), (63, np.int8, 256), (65, np.uint8, 256), (56, np.uint16, 65536), (58, np.int16, 65536)):
        vals = np.arange(n, dtype=np.int64).astype(dtype) if dtype in (np.uint8, np.uint16) else (np.arange(n, dtype=np.int64) - n // 2).astype(dtype)
        w, h = (256, n // 256)
        src = vals.reshape(h, w)
        for df in (2, 41):
            hr, want = oracle.convert(src, w, h, sf, df)
            got = capi.convert(src, w, h, sf, df)
            assert hr == 0 and same(got, want), (sf, df)


def test_convert_srgb_within_one_code(oracle):
    rng = np.random.default_rng(5)
    src = oracle_lib.random_image(29, 64, 16, rng)
    hr, want = oracle.convert(src, 64, 16, 29, 28, full=True)
    got = capi.convert(src, 64, 16, 29, 28)
    assert hr == 0 and np.abs(got.astype(int) - want.astype(int)).max() <= 1


def test_mips_golden():
    for name, src, meta, exp in golden_util.cases("mips_"):
        w, h, fmt, fl = (int(v) for v in meta)
        if h == 1 and (fl & 0xF00000) == F.TEX_FILTER_BOX:
            continue
        got, _ = capi.generate_mipmaps(src, w, h, fmt, fl)
        assert same(got, exp), name


@pytest.mark.parametrize("fl", [F.TEX_FILTER_BOX, F.TEX_FILTER_LINEAR, F.TEX_FILTER_CUBIC, F.TEX_FILTER_TRIANGLE, F.TEX_FILTER_POINT, 0,
                                F.TEX_FILTER_LINEAR | F.TEX_FILTER_WRAP])
def test_mips_vs_oracle(oracle, fl):
    rng = np.random.default_rng(6)
    # sizes above 64 that divide by 8 take the fused three-level BOX / LINEAR kernel, the others the per-level / tail kernels
    for (fmt, w, h) in [(28, 256, 256), (10, 128, 64), (2, 64, 64), (61, 256, 64), (28, 100, 60), (2, 128, 128), (87, 256, 128), (41, 512, 8)]:
        if (fl == F.TEX_FILTER_BOX) and (w & (w - 1) or h & (h - 1)):
            continue
        src = oracle_lib.random_image(fmt, w, h, rng)
        hr, want = oracle.generate_mipmaps(src, w, h, fmt, fl)
        got, _ = capi.generate_mipmaps(src, w, h, fmt, fl)
        assert hr == 0 and same(got, want), (fmt, w, h, hex(fl))


@pytest.mark.parametrize("fl", [0, F.TEX_FILTER_POINT, F.TEX_FILTER_BOX, F.TEX_FILTER_LINEAR, F.TEX_FILTER_CUBIC, F.TEX_FILTER_TRIANGLE,
                                F.TEX_FILTER_LINEAR | F.TEX_FILTER_WRAP, F.TEX_FILTER_CUBIC | F.TEX_FILTER_MIRROR])
def test_resize_vs_oracle(oracle, fl):
    """SURVEY 8(f) rank 2: DirectX::Resize with the custom filters, bit-exact vs the reference (down-, up-scaling, odd sizes)."""
    rng = np.random.default_rng(16)
    for (fmt, w, h, nw, nh) in [(28, 64, 64, 32, 32), (28, 100, 60, 37, 91), (2, 48, 32, 96, 80), (10, 33, 17, 16, 8),
                                (61, 128, 16, 64, 8), (87, 40, 40, 40, 13)]:
        if (fl & 0xF00000) == F.TEX_FILTER_BOX and (nw * 2 != w or nh * 2 != h):
            continue
        src = oracle_lib.random_image(fmt, w, h, rng)
        hr, want = oracle.resize(src, w, h, fmt, nw, nh, fl)
        got = capi.resize(src, w, h, fmt, nw, nh, fl)
        assert hr == 0 and same(got, want), (fmt, w, h, nw, nh, hex(fl))


@pytest.mark.parametrize("flags", [0, 0x1, 0x2, 0x3])
def test_premultiply_alpha_vs_oracle(oracle, flags):
    """SURVEY 8(f) rank 4 (first part): DirectX::PremultiplyAlpha / demultiply, bit-exact vs the reference for non-sRGB formats;
    sRGB formats without IGNORE_SRGB go through powf and are held to +-1 code."""
    rng = np.random.default_rng(23)
    for (fmt, w, h) in [(28, 64, 32), (87, 37, 5), (2, 33, 9), (10, 40, 8), (11, 16, 16), (24, 24, 8), (29, 64, 16)]:
        src = oracle_lib.random_image(fmt, w, h, rng)
        hr, want = oracle.premultiply_alpha(src, w, h, fmt, flags, full=(fmt == 29 and not (flags & 1)))
        got = capi.premultiply_alpha(src, w, h, fmt, flags)
        assert hr == 0
        if fmt == 29 and not (flags & 1):
            assert np.abs(got.astype(np.int32) - want.astype(np.int32)).max() <= 1, (fmt, flags)
        else:
            assert same(got, want), (fmt, w, h, flags)
    with pytest.raises(capi.DxTexError) as e:
        capi.premultiply_alpha(np.zeros((8, 8), np.uint8), 8, 8, 61, 0)            # R8 has no alpha
    assert e.value.hr == F.HRESULT_E_NOT_SUPPORTED


def _alpha_test_image(fmt, w, h, rng):
    yy, xx = np.mgrid[0:h, 0:w]
    a = np.clip(0.5 + 0.4 * np.sin(xx * 0.4) * np.cos(yy * 0.3) + rng.normal(0, 0.12, (h, w)), 0, 1)
    if fmt in (28, 29, 87):
        img = rng.integers(0, 256, (h, w, 4), dtype=np.uint8)
        img[..., 3] = (a * 255).astype(np.uint8)
        return img
    img = rng.random((h, w, 4), dtype=np.float32)
    img[..., 3] = a
    return img.astype(np.float16) if fmt == 10 else img


def test_scale_mipmaps_alpha_for_coverage(oracle, emul):
    """SURVEY 8(f) rank 4: GenerateMipMaps -> ScaleMipMapsAlphaForCoverage (texconv -keepcoverage), bit-exact vs the reference."""
    rng = np.random.default_rng(47)
    for fmt, w, h in [(28, 128, 128), (28, 48, 20), (2, 32, 32), (87, 16, 64), (10, 33, 17), (29, 64, 64)]:
        img = _alpha_test_image(fmt, w, h, rng)
        for ref in (0.5, 0.25):
            hr, plain, want = oracle.mips_alpha_coverage(img, w, h, fmt, ref)
            hp, chain = emul.generate_mipmaps(img, w, h, fmt)       # the reference's plain chain, bit for bit
            got = capi.scale_mipmaps_alpha_for_coverage(chain, w, h, fmt, ref)
            assert hr == 0 and hp == 0 and same(chain, plain) and same(got, want), (fmt, w, h, ref)


def test_bc7_equals_emulator_and_quality(emul):
    """GPU BC7 == host lock-step emulator (same source, explicit fmaf, -fmad=false) bit for bit, and
    MSE <= 1.02 x the reference CPU encoder's MSE (golden anchor) on each test image."""
    z = golden_util.load()
    for j in range(3):
        w, h, seed = (int(v) for v in z["bc7_%d_meta" % j])
        kind = bytes(z["bc7_%d_kind" % j]).decode()
        img = synth.c2_rgba32f(w, h, seed) if kind == "c2" else synth.photo_rgba32f(w, h, seed, alpha=(kind == "alpha"))
        got = capi.compress(img, w, h, 2, 98)
        he, em = emul.compress(img, w, h, 2, 98)
        assert he == 0
        nd = int((got.reshape(-1, 16) != em.reshape(-1, 16)).any(1).sum())
        mse = oracle_lib.mse255(emul.decode_blocks(98, got, w, h), img)
        ref_mse = float(z["bc7_%d_refmse" % j][0])
        assert mse <= ref_mse * 1.02, (kind, mse, ref_mse)
        assert nd == 0, "%d of %d blocks differ from the emulator" % (nd, got.size // 16)


@pytest.mark.parametrize("kind,flags", tolerance.bc7_cases())
def test_bc7_contract_per_class_on_device(emul, kind, flags):
    """Every content class of the tolerance corpus at 256^2: the CUDA encoder's blocks are bit-identical to the host emulator's
    and meet the BC7 contract (tests/tolerance.py) against the reference encoder's per-block errors (committed golden)."""
    n = tolerance.SIZE
    img = synth.content_ldr(kind, n, n, tolerance.SEED)
    got = capi.compress(img, n, n, 2, 98, flags)
    he, em = emul.compress(img, n, n, 2, 98, flags)
    assert he == 0
    nd = int((got.reshape(-1, 16) != em.reshape(-1, 16)).any(1).sum())
    assert nd == 0, "%s: %d of %d blocks differ from the emulator" % (kind, nd, got.size // 16)
    tolerance.check_bc7(emul, kind, flags, got)


@pytest.mark.parametrize("kind,fmt", tolerance.bc6h_cases())
def test_bc6h_contract_per_class_on_device(emul, kind, fmt):
    """As above for BC6H_UF16 / BC6H_SF16, including the float-domain bounds (sign-crossing content)."""
    n = tolerance.SIZE
    img = synth.content_hdr(kind, n, n, tolerance.SEED)
    got = capi.compress(img, n, n, 2, fmt)
    he, em = emul.compress(img, n, n, 2, fmt)
    assert he == 0
    nd = int((got.reshape(-1, 16) != em.reshape(-1, 16)).any(1).sum())
    assert nd == 0, "%s: %d blocks differ from the emulator" % (kind, nd)
    tolerance.check_bc6h(emul, kind, fmt, got)


@pytest.mark.parametrize("kind", ["cutout", "alpha_photo", "gradient", "c2"])
def test_bc7_device_equals_emulator_512(emul, kind):
    """16384 blocks per class: the packed-fp32 (FFMA2) code paths must round exactly like the scalar host emulator.  (ptxas
    contracts a packed multiply feeding a packed add; two such sites differed in 1 of ~15000 blocks until the fused form was
    written explicitly, dxb_portable.h.)"""
    img = synth.content_ldr(kind, 512, 512, tolerance.SEED)
    got = capi.compress(img, 512, 512, 2, 98)
    he, em = emul.compress(img, 512, 512, 2, 98)
    assert he == 0
    nd = int((got.reshape(-1, 16) != em.reshape(-1, 16)).any(1).sum())
    assert nd == 0, "%s: %d of %d blocks differ from the emulator" % (kind, nd, got.size // 16)


def test_full_size_c2_bc7_mse_vs_reference_on_crop(oracle, emul):
    """BASELINE configs[1] "bit-check vs ref BC7 MSE": the 4096^2 image is compressed on the GPU; on a 512^2 aligned crop (16384
    blocks: the blocks of a crop are the blocks of the full image, test_full_size_c2_bc7_properties) the reference encoder runs
    here on the host and both streams are decoded by the reference decoder: MSE_gpu <= 1.02 x MSE_ref, < 1 % of blocks worse
    than 2 x + 16."""
    img = synth.c2_rgba32f(4096, 4096)
    a = capi.compress(img, 4096, 4096, 2, 98).reshape(1024, 1024, 16)
    y0, x0, s = 1536, 512, 512
    crop = np.ascontiguousarray(img[y0:y0 + s, x0:x0 + s])
    gpu_blocks = np.ascontiguousarray(a[y0 // 4:(y0 + s) // 4, x0 // 4:(x0 + s) // 4]).reshape(-1)
    hr, theirs = oracle.bc7_block_sse(crop, s, s, 0, full=True)
    assert hr == 0
    ours, theirs = tolerance.bc7_block_sse(emul, gpu_blocks, crop), theirs.astype(np.float64)
    assert ours.sum() <= 1.02 * theirs.sum(), ours.sum() / theirs.sum()
    assert float((ours > 2.0 * theirs + 16.0).mean()) < 0.01


def test_bc7_rgba8_source_partial_blocks_and_quick(emul):
    rng = np.random.default_rng(8)
    for (w, h) in [(5, 7), (1, 1), (30, 18)]:
        src = oracle_lib.random_image(28, w, h, rng)
        for flags in (0, F.TEX_COMPRESS_BC7_QUICK):
            got = capi.compress(src, w, h, 28, 98, flags)
            he, em = emul.compress(src, w, h, 28, 98, flags)
            assert he == 0 and same(got, em), (w, h, flags)
            dec = emul.decode_blocks(98, got, w, h)      # decodable (the decoder is bit-exact to the reference's)
            assert np.isfinite(dec).all()


def test_bc7_tma_fed_kernel_equals_emulator(emul):
    """RGBA32F sources made of full 4x4 blocks go through k_compress_bc7_tma (persistent CTAs, one TMA box of 64 x 4 pixels per
    tile): widths that end in a partial, zero-filled tile, a single tile, more tiles than resident CTAs, the three-subset
    instantiation, and an array at a constant pointer stride (rank-3 tensor map) on the device API -- all must equal the emulator,
    as must a source whose rows are not 16-byte aligned for the tensor map (pitch padded by 4 bytes: the direct kernel)."""
    torch = pytest.importorskip("torch")
    rng = np.random.default_rng(23)
    before, feed = capi.tma_launch_count(), capi.lib.dxb200_get_option(capi.OPT_BC7_FEED)
    assert capi.lib.dxb200_set_option(capi.OPT_BC7_FEED, 1) == 0          # the default (4) takes the direct kernel for single images
    try:
        _tma_cases(emul, torch, rng)
    finally:
        capi.lib.dxb200_set_option(capi.OPT_BC7_FEED, feed)
    assert capi.tma_launch_count() >= before + 7                           # six single images + the stride-aligned array went through TMA


def _tma_cases(emul, torch, rng):
    for (w, h, flags) in [(100, 52, 0), (64, 4, 0), (4, 4, 0), (260, 8, 0), (1024, 512, 0), (72, 20, F.TEX_COMPRESS_BC7_USE_3SUBSETS)]:
        img = rng.random((h, w, 4), dtype=np.float32)
        if w == 100:
            img[:, :48, 3] = 1.0
        got = capi.compress(img, w, h, 2, 98, flags)
        he, em = emul.compress(img, w, h, 2, 98, flags)
        assert he == 0 and same(got, em), (w, h, flags)
    w, h, n = 72, 20, 3
    imgs = rng.random((n, h, w, 4), dtype=np.float32)
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    row, sl = F.compute_pitch(98, w, h)
    for pad in (0, 4):
        pitch = w * 16 + pad
        buf = np.zeros((n, h, pitch), np.uint8)
        buf[:, :, :w * 16] = imgs.view(np.uint8).reshape(n, h, w * 16)
        d_in = torch.from_numpy(buf.reshape(-1)).cuda()
        d_out = torch.zeros(n * sl, dtype=torch.uint8, device="cuda")
        s = capi.images([capi.Image(w, h, 2, pitch, pitch * h, d_in.data_ptr() + i * pitch * h) for i in range(n)])
        d = capi.images([capi.Image(w, h, 98, row, sl, d_out.data_ptr() + i * sl) for i in range(n)])
        assert capi.lib.dxb200_compress_device(s, n, 98, 0, 0.5, 1.0, d, st) == 0
        torch.cuda.synchronize()
        out = d_out.cpu().numpy().reshape(n, sl)
        for i in range(n):
            he, em = emul.compress(imgs[i], w, h, 2, 98, 0)
            assert he == 0 and same(out[i], em), (pad, i)


def test_device_api_with_torch_pointers(oracle):
    torch = pytest.importorskip("torch")
    img = synth.c1_rgba8(128, 64, seed=2)
    d_in = torch.from_numpy(img.reshape(-1)).cuda()
    row, sl = F.compute_pitch(77, 128, 64)
    d_out = torch.zeros(sl, dtype=torch.uint8, device="cuda")
    s = capi.images([capi.Image(128, 64, 28, 128 * 4, 128 * 64 * 4, d_in.data_ptr())])
    d = capi.images([capi.Image(128, 64, 77, row, sl, d_out.data_ptr())])
    st = torch.cuda.current_stream()
    assert capi.lib.dxb200_compress_device(s, 1, 77, 0, 0.5, 1.0, d, C.c_void_p(st.cuda_stream)) == 0
    torch.cuda.synchronize()
    hr, want = oracle.compress(img, 128, 64, 28, 77)
    assert hr == 0 and same(d_out.cpu().numpy(), want)


def test_full_size_c2_bc7_properties(emul):
    """BASELINE configs[1] at full size (4096^2 RGBA32F -> BC7): size-independent properties.
    determinism; locality (the blocks of an aligned crop are identical to the same blocks of the full image);
    the crop equals the emulator; whole-image MSE sane (PSNR > 30 dB)."""
    img = synth.c2_rgba32f(4096, 4096)
    a = capi.compress(img, 4096, 4096, 2, 98)
    b = capi.compress(img, 4096, 4096, 2, 98)
    assert same(a, b)
    y0, x0, s = 1024, 2048, 128
    crop = np.ascontiguousarray(img[y0:y0 + s, x0:x0 + s])
    cb = capi.compress(crop, s, s, 2, 98).reshape(s // 4, s // 4, 16)
    full = a.reshape(1024, 1024, 16)[y0 // 4:(y0 + s) // 4, x0 // 4:(x0 + s) // 4]
    assert same(cb, full)
    he, em = emul.compress(crop, s, s, 2, 98)
    assert he == 0 and same(cb.reshape(-1), em)
    step = 8
    sub = a.reshape(1024, 1024, 16)[::step, ::step].reshape(-1, 16).copy()
    n = sub.shape[0]
    dec = emul.decode_blocks(98, sub, 4 * n, 4).reshape(4, n, 4, 4).transpose(1, 0, 2, 3).reshape(n, 16, 4)
    src_blocks = img.reshape(1024, 4, 1024, 4, 4).transpose(0, 2, 1, 3, 4)[::step, ::step].reshape(-1, 16, 4)
    mse = float(((dec.astype(np.float64) * 255.0 - oracle_lib.bc7_ldr(src_blocks)) ** 2).mean())
    assert oracle_lib.psnr(mse) > 30.0, mse


def test_full_size_c5_bc4_and_convert_roundtrip(oracle):
    """BASELINE configs[4]: 8192^2 R8 -> BC4 bit-exact on sampled block rows; R8 -> R32F -> R8 is the identity."""
    img = synth.c5_r8(8192, 8192)
    got = capi.compress(img, 8192, 8192, 61, 80).reshape(2048, 2048, 8)
    for by in (0, 777, 2047):
        rows = np.ascontiguousarray(img[by * 4:by * 4 + 4])
        hr, want = oracle.compress(rows, 8192, 4, 61, 80)
        assert hr == 0 and same(got[by].reshape(-1), want), by
    f = capi.convert(img, 8192, 8192, 61, 41)
    assert same(f.view(np.float32), (img.reshape(-1).astype(np.float32) / np.float32(255.0)))
    back = capi.convert(f, 8192, 8192, 41, 61)
    assert same(back, img.reshape(-1))


def test_bc6h_equals_emulator_and_quality(emul):
    """GPU BC6H == host lock-step emulator bit for bit; error (reference metric) <= 1.02 x the reference CPU encoder's."""
    z = golden_util.load()
    for j in range(4):
        w, h, seed, fmt = (int(v) for v in z["bc6h_%d_meta" % j])
        kind = bytes(z["bc6h_%d_kind" % j]).decode()
        img = oracle_lib.bc6h_test_image(kind, w, h, seed)
        got = capi.compress(img, w, h, 2, fmt)
        he, em = emul.compress(img, w, h, 2, fmt)
        assert he == 0
        err = oracle_lib.bc6h_int_mse(emul.decode_blocks(fmt, got, w, h), img, fmt == 96)
        assert err <= float(z["bc6h_%d_referr" % j][0]) * 1.02, (kind, err)
        nd = int((got.reshape(-1, 16) != em.reshape(-1, 16)).any(1).sum())
        assert nd == 0, "%d blocks differ from the emulator" % nd


def test_config3_rgba16f_cubic_chain_bc6h(oracle, emul):
    """BASELINE configs[2] at reduced size: RGBA16F -> full CUBIC mip chain (bit-exact vs oracle) -> BC6H_UF16 of every
    level (== emulator; top level within tolerance of the reference encoder)."""
    w = h = 256
    img = synth.c3_rgba16f(w, h)
    chain, layout = capi.generate_mipmaps(img, w, h, 10, F.TEX_FILTER_CUBIC)
    hr, want = oracle.generate_mipmaps(img, w, h, 10, F.TEX_FILTER_CUBIC)
    assert hr == 0 and same(chain, want)
    for (off, lw, lh, row, sl) in layout[:4]:
        level = chain[off:off + sl]
        got = capi.compress(level, lw, lh, 10, 95)
        he, em = emul.compress(level, lw, lh, 10, 95)
        assert he == 0 and same(got, em)


DECOMPRESS_CASES = ((71, (28, 2)), (74, (28,)), (77, (28, 2)), (80, (61, 41)), (81, (63, 41)), (83, (49, 16)), (84, (51,)),
                    (98, (28, 2, 87)), (95, (2, 10)), (96, (2, 10)))


def _bc_inputs(oracle, bc, w, h, rng):
    """random bytes (every mode / invalid mode of the format) and a block stream produced by the reference encoder"""
    nb = ((w + 3) // 4) * ((h + 3) // 4)
    yield rng.integers(0, 256, nb * F.BLOCK_BYTES[bc], dtype=np.uint8)
    src = rng.random((h, w, 4)).astype(np.float32) * (4.0 if bc in (95, 96) else 1.0) - (1.0 if bc in (81, 84, 96) else 0.0)
    hr, blocks = oracle.compress(src, w, h, 2, bc, 0, full=True)
    assert hr == 0
    yield blocks


def test_decompress_bit_exact(oracle):
    rng = np.random.default_rng(22)
    for bc, dsts in DECOMPRESS_CASES:
        for (w, h) in ((64, 32), (5, 7), (13, 9)):
            for blocks in _bc_inputs(oracle, bc, w, h, rng):
                for df in dsts:
                    hr, want = oracle.decompress(blocks, w, h, bc, df)
                    got = capi.decompress(blocks, w, h, bc, df)
                    assert hr == 0 and same(got, want), (bc, df, w, h)


def test_compress_decompress_round_trip_full_size():
    """size-independent property at full size: GPU encode -> GPU decode of 4096^2 stays within the BC7 error budget"""
    img = synth.c2_rgba32f(4096, 4096)
    blocks = capi.compress(img, 4096, 4096, 2, 98)
    back = capi.decompress(blocks, 4096, 4096, 98, 28).reshape(4096, 4096, 4).astype(np.float32)
    mse = float(((back - oracle_lib.bc7_ldr(img)) ** 2).mean())
    assert oracle_lib.psnr(mse) > 30.0


def test_mipmaps_compress_equals_two_calls_and_reference(oracle):
    """dxb200_mipmaps_compress (the chain stays in HBM) == dxb200_generate_mipmaps + dxb200_compress == the reference, bit for bit
    (BASELINE configs[3] shape: RGBA8 -> default-filter chain -> BC3), including a non-power-of-two size (LINEAR default)."""
    rng = np.random.default_rng(41)
    for (w, h, n) in [(256, 256, 5), (96, 40, 3)]:
        srcs = [oracle_lib.random_image(28, w, h, rng) for _ in range(n)]
        outs = capi.mipmaps_compress(srcs, w, h, 28, 77)
        for src, got in zip(srcs, outs):
            chain, layout = capi.generate_mipmaps(src, w, h, 28, 0)
            hr, rchain = oracle.generate_mipmaps(src, w, h, 28, 0)
            assert hr == 0 and same(chain, rchain)
            want = [oracle.compress(chain[off:off + sl], lw, lh, 28, 77)[1] for (off, lw, lh, row, sl) in layout]
            assert same_concat(got, want, [F.compute_pitch(77, lw, lh)[1] for (off, lw, lh, row, sl) in layout]), (w, h)


def test_concurrent_host_calls_from_threads(oracle):
    """entry points are callable concurrently: each host-pointer call takes its own staging lane (streams + buffers)"""
    import threading
    rng = np.random.default_rng(43)
    srcs = [oracle_lib.random_image(28, 512, 256, rng) for _ in range(6)]
    res = [None] * len(srcs)

    def work(i):
        res[i] = capi.compress(srcs[i], 512, 256, 28, 77 if i % 2 else 71)
    th = [threading.Thread(target=work, args=(i,)) for i in range(len(srcs))]
    for t in th:
        t.start()
    for t in th:
        t.join()
    for i, s_ in enumerate(srcs):
        hr, want = oracle.compress(s_, 512, 256, 28, 77 if i % 2 else 71)
        assert hr == 0 and same(res[i], want), i


def test_multi_device_sharding_inside_the_library(oracle, emul):
    """dxb200_init_devices: array calls and mip chains are sharded over the GPUs inside one process; results unchanged"""
    rng = np.random.default_rng(47)
    srcs = [oracle_lib.random_image(28, 128, 64, rng) for _ in range(17)]       # 2 n + 1 images for up to 8 GPUs
    layout, _ = F.mip_chain_layout(28, 128, 64, 0)
    want_bc3 = [oracle.compress(s_, 128, 64, 28, 77) for s_ in srcs]
    want_chain = [oracle.generate_mipmaps(s_, 128, 64, 28, 0) for s_ in srcs]
    chains = [emul.generate_mipmaps(s_, 128, 64, 28, 0)[1] for s_ in srcs]        # equal to the reference's chains (asserted below)
    want_bc1 = [[oracle.compress(c[off:off + sl], lw, lh, 28, 71)[1] for (off, lw, lh, row, sl) in layout] for c in chains]
    n = capi.lib.dxb200_device_count()
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    srcs = srcs[:2 * n + 1]
    capi.init_devices(list(range(n)))
    outs = capi.compress_array(srcs, 128, 64, 28, 77)
    for (hr, want), o in zip(want_bc3, outs):
        assert hr == 0 and same(o, want)
    outs = capi.mipmaps_compress(srcs, 128, 64, 28, 71)
    for (hr, rchain), c, want, o in zip(want_chain, chains, want_bc1, outs):
        assert hr == 0 and same(c, rchain)
        assert same_concat(o, want, [F.compute_pitch(71, lw, lh)[1] for (off, lw, lh, row, sl) in layout])


def test_next_tier_formats_vs_oracle(oracle):
    """R11G11B10_FLOAT, R9G9B9E5_SHAREDEXP, B5G6R5, B5G5R5A1, B4G4R4A4 through the C ABI: Convert both ways (incl. x2 bias and the alpha
    threshold), mip chains, BC compression; dithered stores to the 16-bit packed formats are refused (HRESULT_E_NOT_SUPPORTED)."""
    from tests.test_cpu_oracle import NEXT_TIER, NEXT_TIER_PAIRS
    rng = np.random.default_rng(79)
    for sf, df in NEXT_TIER_PAIRS:
        src = oracle_lib.random_image(sf, 133, 21, rng)
        for fl in (0, F.TEX_FILTER_FLOAT_X2BIAS):
            hr, want = oracle.convert(src, 133, 21, sf, df, fl)
            got = capi.convert(src, 133, 21, sf, df, fl)
            assert hr == 0 and same(got, want), (sf, df, hex(fl))
    src = oracle_lib.random_image(2, 64, 8, rng)
    for thr in (0.0, 0.25, 0.9):
        hr, want = oracle.convert(src, 64, 8, 2, 86, 0, threshold=thr)
        got = capi.convert(src, 64, 8, 2, 86, 0, threshold=thr)
        assert hr == 0 and same(got, want), thr
    for fmt in NEXT_TIER:
        src = oracle_lib.random_image(fmt, 40, 24, rng)
        for fl in (F.TEX_FILTER_POINT, F.TEX_FILTER_LINEAR, F.TEX_FILTER_CUBIC, F.TEX_FILTER_TRIANGLE, 0):
            hr, want = oracle.generate_mipmaps(src, 40, 24, fmt, fl)
            got, _ = capi.generate_mipmaps(src, 40, 24, fmt, fl)
            assert hr == 0 and same(got, want), (fmt, hex(fl))
        for bc in (71, 77, 80, 83):
            hr, want = oracle.compress(src, 40, 24, fmt, bc)
            assert hr == 0 and same(capi.compress(src, 40, 24, fmt, bc), want), (fmt, bc)
    with pytest.raises(capi.DxTexError) as e:
        capi.convert(oracle_lib.random_image(28, 16, 16, rng), 16, 16, 28, 85, F.TEX_FILTER_DITHER)
    assert e.value.hr == F.HRESULT_E_NOT_SUPPORTED
