"""CPU suite, part 1: the oracle (unmodified reference sources built by oracle/Makefile) against the committed
golden vectors, and the host lock-step emulator of our kernels' arithmetic against the oracle.
Nothing here runs product code paths; no GPU needed."""
import numpy as np
import pytest

from directxtex_b200 import formats as F, synth
from tests import golden_util, oracle_lib
from tests.oracle_lib import same


def test_oracle_matches_golden_compress(oracle):
    n = 0
    for name, src, meta, exp in golden_util.cases("compress_"):
        w, h, sf, df, flags = (int(v) for v in meta)
        hr, out = oracle.compress(src, w, h, sf, df, flags)
        assert hr == 0
        assert same(out, exp), name
        n += 1
    assert n > 100


def test_oracle_config1_bc1(oracle):
    """BASELINE.json configs[0]: single 256x256 RGBA8 -> BC1 via the reference CPU Compress() on a Linux build."""
    img = synth.c1_rgba8(256, 256)
    hr, out = oracle.compress(img, 256, 256, F.DXGI_FORMAT_R8G8B8A8_UNORM, F.DXGI_FORMAT_BC1_UNORM, 0, parallel=False)
    assert hr == 0 and out.nbytes == 32768
    assert same(out, golden_util.load()["config1_bc1_out"])
    hr2, out2 = oracle.compress(img, 256, 256, 28, 71, 0, parallel=True)      # OpenMP path gives the same bytes
    assert hr2 == 0 and same(out, out2)


def test_oracle_matches_golden_convert_and_mips(oracle):
    for name, src, meta, exp in golden_util.cases("convert_"):
        w, h, sf, df, fl = (int(v) for v in meta)
        hr, out = oracle.convert(src, w, h, sf, df, fl)
        assert hr == 0 and same(out, exp), name
    for name, src, meta, exp in golden_util.cases("mips_"):
        w, h, fmt, fl = (int(v) for v in meta)
        hr, out = oracle.generate_mipmaps(src, w, h, fmt, fl)
        assert hr == 0 and same(out, exp), name


def test_emulator_bc15_bit_exact_vs_golden(emul):
    for name, src, meta, exp in golden_util.cases("compress_"):
        w, h, sf, df, flags = (int(v) for v in meta)
        hr, out = emul.compress(src, w, h, sf, df, flags)
        assert hr == 0
        assert same(out, exp), name


@pytest.mark.parametrize("df", [71, 74, 77, 80, 81, 83, 84])
def test_emulator_bc15_bit_exact_vs_oracle_random(oracle, emul, df):
    rng = np.random.default_rng(100 + df)
    for (w, h, sf) in [(96, 64, 28), (31, 17, 28), (40, 40, 2), (24, 24, 10), (64, 16, 61), (16, 16, 31), (20, 12, 41)]:
        src = oracle_lib.random_image(sf, w, h, rng)
        for flags in (0, F.TEX_COMPRESS_UNIFORM, F.TEX_COMPRESS_DITHER):
            hr, a = oracle.compress(src, w, h, sf, df, flags)
            he, b = emul.compress(src, w, h, sf, df, flags)
            assert hr == 0 and he == 0
            assert same(a, b), (w, h, sf, df, hex(flags))


def test_emulator_convert_bit_exact(oracle, emul):
    for name, src, meta, exp in golden_util.cases("convert_"):
        w, h, sf, df, fl = (int(v) for v in meta)
        he, out = emul.convert(src, w, h, sf, df, fl)
        assert he == 0 and same(out, exp), name


def test_emulator_convert_exhaustive_small_domains(oracle, emul):
    """all values of the 8/16-bit scalar formats: the 3-op exact division equals the reference's IEEE divide"""
    for sf, dtype, n in ((61, np.uint8, 256), (63, np.int8, 256), (65, np.uint8, 256), (56, np.uint16, 65536), (58, np.int16, 65536)):
        vals = np.arange(n, dtype=np.int64).astype(dtype) if dtype in (np.uint8, np.uint16) else (np.arange(n, dtype=np.int64) - n // 2).astype(dtype)
        w, h = (256, n // 256)
        src = vals.reshape(h, w)
        for df in (2, 41):
            hr, want = oracle.convert(src, w, h, sf, df)
            he, got = emul.convert(src, w, h, sf, df)
            assert hr == 0 and he == 0 and same(got, want), (sf, df)


def test_emulator_mips_bit_exact(oracle, emul):
    for name, src, meta, exp in golden_util.cases("mips_"):
        w, h, fmt, fl = (int(v) for v in meta)
        if h == 1 and (fl & 0xF00000) == F.TEX_FILTER_BOX:
            continue   # reference reads uninitialised memory for height-1 top levels (DESIGN.md, box filter quirk)
        he, out = emul.generate_mipmaps(src, w, h, fmt, fl)
        assert he == 0 and same(out, exp), name


def test_emulator_srgb_within_one_code(oracle, emul):
    """sRGB formats go through powf: glibc vs CUDA libm differ in the last ulp, so the contract is +-1 code (SURVEY A.7)."""
    rng = np.random.default_rng(7)
    src = oracle_lib.random_image(29, 32, 16, rng)
    hr, a = oracle.generate_mipmaps(src, 32, 16, 29, F.TEX_FILTER_LINEAR, full=True)
    he, b = emul.generate_mipmaps(src, 32, 16, 29, F.TEX_FILTER_LINEAR)
    assert hr == 0 and he == 0
    assert np.abs(a.astype(int) - b.astype(int)).max() <= 1


def test_emulator_bc7_quality_vs_reference(emul):
    """BC7 tolerance (DESIGN.md): RGBA MSE of our encoder <= 1.02 x the reference CPU encoder's MSE on the same
    input (i.e. PSNR no more than 0.09 dB below), every block decodable by the reference decoder."""
    z = golden_util.load()
    for j in range(3):
        w, h, seed = (int(v) for v in z["bc7_%d_meta" % j])
        kind = bytes(z["bc7_%d_kind" % j]).decode()
        img = synth.c2_rgba32f(w, h, seed) if kind == "c2" else synth.photo_rgba32f(w, h, seed, alpha=(kind == "alpha"))
        ref_mse = float(z["bc7_%d_refmse" % j][0])
        # golden self-check: decoding the stored reference blocks reproduces the stored MSE
        assert abs(oracle_lib.mse255(emul.decode_blocks(98, z["bc7_%d_blocks" % j], w, h), img) - ref_mse) < 1e-6
        he, blocks = emul.compress(img, w, h, 2, 98, 0)
        assert he == 0
        mse = oracle_lib.mse255(emul.decode_blocks(98, blocks, w, h), img)
        assert mse <= ref_mse * 1.02, (kind, mse, ref_mse)


def test_emulator_bc7_special_blocks(emul):
    """solid, two-colour, fully transparent, extreme values, partial blocks: decodable and near-lossless where possible"""
    img = np.zeros((16, 16, 4), np.float32)
    img[0:4, 0:4] = [0.2, 0.4, 0.6, 1.0]
    img[0:4, 4:8] = 0.0
    img[0:4, 8:12] = 1.0
    img[4:8, 0:4, :] = np.where((np.arange(4)[:, None] + np.arange(4)[None]) % 2 == 0, 1.0, 0.0)[..., None]
    img[4:8, 4:8] = [1.0, 0.0, 0.0, 0.0]
    img[8:12, :, :3] = np.linspace(0, 1, 16)[None, :, None]
    img[8:12, :, 3] = 1.0
    img[12:16, :, 3] = np.linspace(0, 1, 16)[None, :]
    he, blocks = emul.compress(img, 16, 16, 2, 98, 0)
    assert he == 0
    dec = emul.decode_blocks(98, blocks, 16, 16)
    ldr = oracle_lib.bc7_ldr(img)
    err = np.abs(dec * 255.0 - ldr)
    assert err[0:4, 0:12].max() <= 1.01          # solid blocks reproduce within one code
    assert err[4:8, 0:4].max() <= 1.01           # two-colour checkerboard (b/w) is exact up to endpoint precision
    assert err.max() <= 24.0
    # partial blocks
    for (w, h) in [(5, 7), (1, 1), (2, 3)]:
        sub = np.ascontiguousarray(img[:h, :w])
        he, blocks = emul.compress(sub, w, h, 2, 98, 0)
        assert he == 0 and blocks.nbytes == ((w + 3) // 4) * ((h + 3) // 4) * 16
        dec = emul.decode_blocks(98, blocks, w, h)
        assert np.abs(dec * 255.0 - oracle_lib.bc7_ldr(sub)).max() <= 24.0


def test_emulator_bc7_quick_flag_uses_mode6_only(emul):
    img = synth.photo_rgba32f(32, 32, 3)
    he, blocks = emul.compress(img, 32, 32, 2, 98, F.TEX_COMPRESS_BC7_QUICK)
    assert he == 0
    first = blocks.reshape(-1, 16)[:, 0]
    assert np.all((first & 0x7F) == 0x40)      # mode 6: six zero bits then a one


def test_emulator_bc6h_quality_vs_reference(emul):
    """BC6H tolerance (DESIGN.md): error in the reference encoder's own metric (squared half-float bit-pattern
    differences over RGB) <= 1.02 x the reference CPU encoder's on the same input; decodable by the reference decoder."""
    z = golden_util.load()
    for j in range(4):
        w, h, seed, fmt = (int(v) for v in z["bc6h_%d_meta" % j])
        kind = bytes(z["bc6h_%d_kind" % j]).decode()
        img = oracle_lib.bc6h_test_image(kind, w, h, seed)
        ref_err = float(z["bc6h_%d_referr" % j][0])
        assert abs(oracle_lib.bc6h_int_mse(emul.decode_blocks(fmt, z["bc6h_%d_blocks" % j], w, h), img, fmt == 96) - ref_err) <= 1e-6 * max(ref_err, 1)
        he, blocks = emul.compress(img, w, h, 2, fmt, 0)
        assert he == 0
        err = oracle_lib.bc6h_int_mse(emul.decode_blocks(fmt, blocks, w, h), img, fmt == 96)
        assert err <= ref_err * 1.02, (kind, fmt, err, ref_err)


def test_emulator_bc6h_special_blocks(emul):
    img = np.zeros((12, 16, 4), np.float32)
    img[..., 3] = 1
    img[0:4, 0:4, :3] = 0.0
    img[0:4, 4:8, :3] = 65504.0
    img[0:4, 8:12, :3] = [1.0, 0.5, 0.25]
    img[4:8, :, :3] = np.exp2(np.linspace(-8, 8, 16))[None, :, None]
    img[8:12, :, 0] = 1000.0
    for (w, h) in [(16, 12), (5, 7), (1, 1)]:
        sub = np.ascontiguousarray(img[:h, :w])
        he, blocks = emul.compress(sub, w, h, 2, 95, 0)
        assert he == 0
        dec = emul.decode_blocks(95, blocks, w, h)
        assert np.isfinite(dec).all()
        rel = np.abs(dec[..., :3] - sub[..., :3]) / np.maximum(np.abs(sub[..., :3]), 1e-3)
        assert rel[:4, :min(w, 12)].max() <= 0.02 if h >= 4 and w >= 12 else True      # solid blocks are near exact


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


def test_emulator_decompress_bit_exact(oracle, emul):
    rng = np.random.default_rng(21)
    for bc, dsts in DECOMPRESS_CASES:
        for (w, h) in ((32, 32), (5, 7), (13, 9)):
            for blocks in _bc_inputs(oracle, bc, w, h, rng):
                for df in dsts:
                    hr, want = oracle.decompress(blocks, w, h, bc, df)
                    he, got = emul.decompress(blocks, w, h, bc, df)
                    assert hr == 0 and he == 0 and same(got, want), (bc, df, w, h)


def test_emulator_dither_matches_reference(oracle, emul):
    """The ordered-dither and error-diffusion stores of dxb_pixel.cuh (compiled for the host by tests/emul) against the reference's StoreScanlineDither."""
    rng = np.random.default_rng(41)
    for sf in (2, 28):
        for df in (11, 13, 24, 28, 31, 35, 49, 51, 56, 58, 61, 63, 65, 87, 88):
            if sf == df:
                continue
            src = oracle_lib.random_image(sf, 21, 6, rng)
            for fl in (F.TEX_FILTER_DITHER, F.TEX_FILTER_DITHER_DIFFUSION):
                hr, want = oracle.convert(src, 21, 6, sf, df, fl)
                he, got = emul.convert(src, 21, 6, sf, df, fl)
                assert hr == 0 and he == 0 and same(got, want), (sf, df, hex(fl))


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


def test_emulator_alpha_coverage_matches_reference(oracle, emul):
    """ScaleMipMapsAlphaForCoverage: coverage counting (with the reference's sequential sub-sample quirk), the 10-step bisection
    and ScaleAlpha, compiled for the host from the device sources, against the reference."""
    rng = np.random.default_rng(43)
    for fmt, w, h in [(28, 64, 64), (28, 48, 20), (2, 32, 32), (87, 16, 64), (10, 33, 17)]:
        img = _alpha_test_image(fmt, w, h, rng)
        for ref in (0.5, 0.25):
            hr, plain, want = oracle.mips_alpha_coverage(img, w, h, fmt, ref)
            hp, chain = emul.generate_mipmaps(img, w, h, fmt)       # the reference's plain chain, bit for bit
            he, got = emul.scale_mips_alpha(chain, w, h, fmt, ref)
            assert hr == 0 and hp == 0 and he == 0 and same(chain, plain) and same(got, want) and not same(want, plain), (fmt, w, h, ref)


def test_emulator_bc6h_flat_and_two_colour_blocks(oracle, emul):
    """Flat and two-colour HDR blocks: the reference reproduces flat blocks exactly; the warp encoder must stay within a
    fraction of a half-float code of that (mode 14 with 16-bit endpoints) and within 2 % + 1 on two-colour blocks."""
    rng = np.random.default_rng(61)
    blocks = []
    for k in range(96):
        c0 = np.exp2(rng.uniform(-6, 6, 3))
        if k < 48:
            b = np.tile(c0, (4, 4, 1))
        else:
            b = np.where(rng.integers(0, 2, (4, 4, 1)), c0, np.exp2(rng.uniform(-6, 6, 3)))
        blocks.append(np.concatenate([b, np.ones((4, 4, 1))], -1).astype(np.float32))
    img = np.ascontiguousarray(np.concatenate(blocks, axis=1))
    h, w = 4, 4 * len(blocks)
    for fmt in (95, 96):
        he, eb = emul.compress(img, w, h, 2, fmt)
        hr, rb = oracle.compress(img, w, h, 2, fmt, full=True)
        assert he == 0 and hr == 0
        src = oracle_lib.bc6h_to_int(img[..., :3], fmt == 96)
        err = []
        for bl in (eb, rb):
            d = oracle_lib.bc6h_to_int(emul.decode_blocks(fmt, bl, w, h).reshape(h, w, 4)[..., :3], fmt == 96)
            e = (d.astype(np.float64) - src) ** 2
            err.append(e.reshape(4, len(blocks), 4, 3).transpose(1, 0, 2, 3).reshape(len(blocks), -1).mean(1))
        ours, ref = err
        assert ours[:48].mean() <= ref[:48].mean() + 1.0, (fmt, ours[:48].mean(), ref[:48].mean())
        assert ours[48:].mean() <= ref[48:].mean() * 1.02 + 1.0, (fmt, ours[48:].mean(), ref[48:].mean())


NEXT_TIER = (26, 67, 85, 86, 115)          # R11G11B10_FLOAT, R9G9B9E5_SHAREDEXP, B5G6R5, B5G5R5A1, B4G4R4A4
NEXT_TIER_PAIRS = [(85, 28), (86, 28), (115, 28), (28, 85), (28, 86), (28, 115), (2, 85), (2, 86), (2, 115), (26, 2), (67, 2), (2, 26), (2, 67),
                   (10, 26), (28, 26), (26, 28), (67, 28), (31, 26), (26, 31), (85, 86), (26, 67), (67, 26), (87, 85), (115, 10)]


def test_emulator_next_tier_formats_bit_exact(oracle, emul):
    """R11G11B10_FLOAT, R9G9B9E5_SHAREDEXP, B5G6R5, B5G5R5A1 (alpha threshold 0.5), B4G4R4A4 (DirectXTexConvert.cpp:906, 1189, 1227, 1244, 1511 /
    1756, 2057, 2096, 2116, 2399; CONVF_POS_ONLY x2-bias cases :3469-3583): Convert in both directions, mip chains and BC compression from them."""
    rng = np.random.default_rng(77)
    for sf, df in NEXT_TIER_PAIRS:
        src = oracle_lib.random_image(sf, 37, 9, rng)
        for fl in (0, F.TEX_FILTER_FLOAT_X2BIAS, F.TEX_FILTER_RGB_COPY_GREEN):
            hr, want = oracle.convert(src, 37, 9, sf, df, fl)
            he, got = emul.convert(src, 37, 9, sf, df, fl)
            assert hr == 0 and he == 0 and same(got, want), (sf, df, hex(fl))
    for fmt in NEXT_TIER:
        src = oracle_lib.random_image(fmt, 20, 12, rng)
        for fl in (F.TEX_FILTER_POINT, F.TEX_FILTER_LINEAR, F.TEX_FILTER_CUBIC, F.TEX_FILTER_TRIANGLE, 0):
            hr, want = oracle.generate_mipmaps(src, 20, 12, fmt, fl)
            he, got = emul.generate_mipmaps(src, 20, 12, fmt, fl)
            assert hr == 0 and he == 0 and same(got, want), (fmt, hex(fl))
        for bc in (71, 77, 80, 83):
            hr, want = oracle.compress(src, 20, 12, fmt, bc)
            he, got = emul.compress(src, 20, 12, fmt, bc)
            assert hr == 0 and he == 0 and same(got, want), (fmt, bc)
