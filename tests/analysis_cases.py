"""TEST INFRASTRUCTURE: the seeded case table of ComputeMSE and IsAlphaAllOpaque that tests/test_cpu_analysis.py and
tests/test_gpu_analysis.py both iterate, so that every reference call the GPU test replays is recorded by the CPU test."""
import zlib

import numpy as np

from directxtex_b200 import formats as F
from tests import oracle_lib

BC_FORMATS = (71, 72, 74, 75, 77, 78, 80, 81, 83, 84, 95, 96, 98, 99)
CMSE_ALL = (0x1, 0x2, 0x10, 0x20, 0x40, 0x80, 0x100, 0x200)


def _image(fmt, w, h, rng):
    if fmt in F.BLOCK_BYTES:
        return rng.integers(0, 256, F.compute_pitch(fmt, w, h)[1], dtype=np.uint8)
    return oracle_lib.random_image(fmt, w, h, rng)


def _padded(img, fmt, w, h, pad):
    """the same rows at a row pitch `pad` bytes larger"""
    row, _ = F.compute_pitch(fmt, w, h)
    rows = max(1, (h + 3) // 4) if fmt in F.BLOCK_BYTES else h
    out = np.full((rows, row + pad), 0xA5, np.uint8)
    out[:, :row] = np.ascontiguousarray(img).view(np.uint8).reshape(rows, row)
    return out.reshape(-1), row + pad


def mse_cases():
    """[(id, fmt_a, fmt_b, w, h, flags, pad)]: pad > 0 = both images at a row pitch that many bytes larger"""
    c = []
    for fa, fb in ((28, 28), (29, 28), (88, 28), (2, 10), (61, 41), (24, 11)):
        c.append(("pair_%d_%d" % (fa, fb), fa, fb, 61, 37, 0, 0))
    for fl in (0x100, 0x200):
        c.append(("snorm_bias_%x" % fl, 31, 28, 61, 37, fl, 0))
    for fb in BC_FORMATS:
        c.append(("bc_%d_vs_rgba32f" % fb, 2, fb, 61, 37, 0, 0))
    c.append(("bc_77_vs_71", 77, 71, 61, 37, 0, 0))
    c.append(("bc_99_vs_98", 99, 98, 61, 37, 0, 0))
    for fl in CMSE_ALL + (0x1 | 0x80, 0x10 | 0x40 | 0x200):
        c.append(("flags_%x" % fl, 28, 28, 61, 37, fl, 0))
    c.append(("flags_bc_rgba8_%x" % 0x101, 28, 98, 61, 37, 0x101, 0))
    for w, h in ((1, 1), (2, 3), (5, 7), (256, 256)):
        c.append(("size_rgba8_%dx%d" % (w, h), 28, 28, w, h, 0, 0))
        c.append(("size_bc7_%dx%d" % (w, h), 98, 2, w, h, 0, 0))
    c.append(("size_f16_256", 2, 10, 256, 256, 0, 0))
    c.append(("size_bc1_256", 71, 2, 256, 256, 0, 0))
    c.append(("pitch_rgba8", 28, 28, 61, 37, 0, 12))
    c.append(("pitch_bc3", 77, 28, 61, 37, 0, 32))
    return c


def mse_inputs(case):
    """(a, b) tightly packed, deterministic per case id"""
    cid, fa, fb, w, h, fl, pad = case
    rng = np.random.default_rng(zlib.crc32(cid.encode()))
    return _image(fa, w, h, rng), _image(fb, w, h, rng)


def padded(img, fmt, w, h, pad):
    if not pad:
        return np.ascontiguousarray(img).view(np.uint8).reshape(-1), 0
    return _padded(img, fmt, w, h, pad)


# ---- IsAlphaAllOpaque ------------------------------------------------------------------------------------------------------
def _bc3_block(a0, a1, alpha_idx, rng):
    """one BC3 block: alpha endpoints a0 / a1, 16 alpha indices, colour half random"""
    bits = 0
    for i, k in enumerate(alpha_idx):
        bits |= int(k) << (3 * i)
    return np.concatenate([np.array([a0, a1], np.uint8), np.frombuffer(bits.to_bytes(6, "little"), np.uint8), rng.integers(0, 256, 8, dtype=np.uint8)])


def _bc1_block(three_colour, idx, rng):
    c = sorted(int(v) for v in rng.integers(0, 65536, 2))
    if c[0] == c[1]:
        c[1] = (c[1] + 1) & 0xFFFF
        c = sorted(c)
    c0, c1 = (c[0], c[1]) if three_colour else (c[1], c[0])        # c0 <= c1: 3 colours + transparent
    bits = 0
    for i, k in enumerate(idx):
        bits |= int(k) << (2 * i)
    return np.frombuffer(np.array([c0, c1], np.uint16).tobytes() + bits.to_bytes(4, "little"), np.uint8)


def _bc7_blocks(n, modes, rng):
    b = rng.integers(0, 256, (n, 16), dtype=np.uint8)
    m = rng.choice(modes, n)
    b[:, 0] = (b[:, 0] & ~((2 << m) - 1).astype(np.uint8)) | (1 << m).astype(np.uint8)
    return b.reshape(-1)


def opaque_cases():
    """[(id, fmt, w, h, levels, pixels packed as ScratchImage::Initialize2D(fmt, w, h, 1, levels) lays them out)]"""
    rng = np.random.default_rng(77)
    out = []

    def chain(fmt, w, h, levels, alpha_fn=None):
        layout, total = F.mip_chain_layout(fmt, w, h, levels)
        px = np.zeros(total, np.uint8)
        for off, lw, lh, row, sl in layout:
            px[off:off + sl] = _image(fmt, lw, lh, rng)
        return layout, px

    layout, px = chain(28, 61, 37, 0)
    for off, lw, lh, row, sl in layout:
        px[off + 3:off + sl:4] = 255
    out.append(("rgba8_opaque_chain", 28, 61, 37, len(layout), px.copy()))
    px[layout[-1][0] + 3] = 0                                          # only the last level (1x1) is not opaque
    out.append(("rgba8_last_level", 28, 61, 37, len(layout), px.copy()))
    px = np.full((5 * 7 * 4,), 255, np.uint8)
    px[4 * 17 + 3] = 254
    out.append(("rgba8_254", 28, 5, 7, 1, px))
    img = np.ones((7, 5, 4), np.float32)
    img[..., 3] = np.float32(0.997)
    out.append(("rgba32f_0997", 2, 5, 7, 1, img.reshape(-1).view(np.uint8).copy()))
    img[3, 2, 3] = np.nextafter(np.float32(0.997), np.float32(0))
    out.append(("rgba32f_below_0997", 2, 5, 7, 1, img.reshape(-1).view(np.uint8).copy()))
    for a in (252, 253):
        blocks = np.concatenate([_bc3_block(255, 255, [0] * 16, rng) for _ in range(5)] + [_bc3_block(a, a, [0] * 16, rng)])
        out.append(("bc3_alpha_%d" % a, 77, 12, 8, 1, blocks))
    edge = [0] * 16
    edge[15] = 1                                                       # pixel (3, 3) of the block: outside a 6x6 image
    blocks = np.concatenate([_bc3_block(255, 0, [0] * 16, rng) for _ in range(3)] + [_bc3_block(255, 0, edge, rng)])
    out.append(("bc3_padding_only", 77, 6, 6, 1, blocks))
    blocks = np.concatenate([_bc1_block(False, rng.integers(0, 4, 16), rng) for _ in range(5)] + [_bc1_block(True, [0] * 15 + [3], rng)])
    out.append(("bc1_transparent_index", 71, 12, 8, 1, blocks))
    blocks = np.concatenate([_bc1_block(False, rng.integers(0, 4, 16), rng) for _ in range(6)])
    out.append(("bc1_four_colour", 71, 12, 8, 1, blocks))
    out.append(("bc7_modes_0_3", 98, 16, 12, 1, _bc7_blocks(12, [0, 1, 2, 3], rng)))
    for m in (4, 5, 6, 7):
        out.append(("bc7_mode_%d" % m, 98, 16, 12, 1, _bc7_blocks(12, [m], rng)))
    out.append(("r8_no_alpha", 61, 9, 5, 1, _image(61, 9, 5, rng)))
    out.append(("b5g6r5_no_alpha", 85, 9, 5, 1, _image(85, 9, 5, rng)))
    for f in (80, 83, 95):
        out.append(("bc_%d_no_alpha" % f, f, 12, 8, 1, _image(f, 12, 8, rng)))
    return out


NO_ALPHA = (61, 85, 80, 83, 95)        # HasAlpha() false: ScratchImage::IsAlphaAllOpaque answers true before any scan


def opaque_layout(fmt, w, h, levels):
    return F.mip_chain_layout(fmt, w, h, levels)[0]
