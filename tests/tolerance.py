"""TEST INFRASTRUCTURE: the tolerance contract of the two non-bit-exact codecs (BC7, BC6H), shared by the CPU tests (host
emulator of the CUDA encoder), the GPU tests (the CUDA encoder through the C ABI) and tests/golden/make_golden_bc67.py.

Contract (DESIGN.md section 3), per content class at 256x256, against the UNMODIFIED reference encoder on the same input:
  BC7   image:  RGBA MSE (8-bit codes)           <= 1.02 x the reference's
        blocks: fewer than 1 % of the blocks worse than 2 x the reference's block error + 16
  BC6H  image:  error in the reference encoder's own metric (half bit patterns, RGB)   <= 1.02 x the reference's (+ 0.5 absolute,
                the reference reproduces flat blocks exactly)
        blocks: fewer than 1 % of the blocks worse than 2 x the reference's block error + 768  (16 squared codes per value)
        floats: MSE of the decoded float values <= 1.5 x the reference's, largest absolute float error <= 2 x the reference's
                (+ 2^-10 of the image's largest magnitude): the bit-pattern metric is logarithmic and says nothing about outliers.
"""
import hashlib
import os

import numpy as np

from directxtex_b200 import formats as F, synth
from tests import oracle_lib

SIZE = 256
SEED = 1
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "golden_bc67_v2.npz")
_z = {}


def golden():
    if "z" not in _z:
        _z["z"] = np.load(GOLDEN)
    return _z["z"]


def bc7_cases():
    """(class, TEX_COMPRESS flags)"""
    # default flags on every class; TEX_COMPRESS_BC7_USE_3SUBSETS (modes 0 / 2) on the classes where the reference gains from it
    return [(k, 0) for k in synth.LDR_CLASSES] + [(k, F.TEX_COMPRESS_BC7_USE_3SUBSETS) for k in ("noise", "cluster3", "cluster4", "chan_uncorr", "photo", "c2", "text")]


def bc6h_cases():
    return [(k, 95) for k in synth.HDR_CLASSES] + [(k, 96) for k in synth.HDR_SIGNED_CLASSES] + [("c3", 96), ("smooth", 96)]


def bc7_key(kind, flags):
    return "bc7_%s_%x" % (kind, flags)


def bc6h_key(kind, fmt):
    return "bc6h_%s_%d" % (kind, fmt)


def _blocks(a, n):
    return a.reshape(n // 4, 4, n // 4, 4, -1).sum((1, 3, 4))


def bc7_block_sse(decoder, blocks, img):
    n = img.shape[0]
    dec = decoder.decode_blocks(98, blocks, n, n).astype(np.float64) * 255.0
    src = oracle_lib.bc7_ldr(img).astype(np.float64)
    return _blocks((dec - src) ** 2, n)


def bc6h_block_errors(decoder, blocks, img, fmt):
    n = img.shape[0]
    signed = fmt == 96
    dec = decoder.decode_blocks(fmt, blocks, n, n)
    clip = np.clip(img[..., :3], -65504 if signed else 0, 65504)
    a = oracle_lib.bc6h_to_int(dec[..., :3], signed).astype(np.float64)
    s = oracle_lib.bc6h_to_int(clip, signed).astype(np.float64)
    s16 = clip.astype(np.float16).astype(np.float64)
    fd = (dec[..., :3].astype(np.float64) - s16)
    assert np.isfinite(fd).all()
    return _blocks((a - s) ** 2, n), _blocks(fd ** 2, n), float(np.abs(fd).max())


def bc7_input(kind):
    img = synth.content_ldr(kind, SIZE, SIZE, SEED)
    return img


def check_input(key, img):
    assert bytes(golden()[key + "_sha1"]) == hashlib.sha1(img.tobytes()).digest(), "regenerated input differs from the golden's: " + key


def check_bc7(decoder, kind, flags, blocks):
    """asserts the BC7 contract for `blocks` (our encoder's output for class `kind`, decoded by `decoder`); returns (ratio, bad fraction)"""
    key = bc7_key(kind, flags)
    img = synth.content_ldr(kind, SIZE, SIZE, SEED)
    check_input(key, img)
    ours = bc7_block_sse(decoder, blocks, img)
    theirs = golden()[key + "_sse"].astype(np.float64)
    ratio = ours.sum() / max(theirs.sum(), 1e-9)
    bad = float((ours > 2.0 * theirs + 16.0).mean())
    assert ours.sum() <= 1.02 * theirs.sum() + 1e-6, (key, ratio)
    assert bad < 0.01, (key, bad)
    return ratio, bad


def check_bc6h(decoder, kind, fmt, blocks):
    key = bc6h_key(kind, fmt)
    img = synth.content_hdr(kind, SIZE, SIZE, SEED)
    check_input(key, img)
    z = golden()
    isse, fsse, fmax = bc6h_block_errors(decoder, blocks, img, fmt)
    risse, rfsse, rfmax = z[key + "_isse"], z[key + "_fsse"], float(z[key + "_fmax"][0])
    npx = SIZE * SIZE * 3
    ratio = isse.sum() / max(risse.sum(), 1e-9)
    assert isse.sum() / npx <= 1.02 * risse.sum() / npx + 0.5, (key, ratio)
    bad = float((isse > 2.0 * risse + 768.0).mean())
    assert bad < 0.01, (key, bad)
    scale = float(np.abs(np.clip(img[..., :3], -65504, 65504)).max())
    assert fsse.sum() <= 1.5 * rfsse.sum() + npx * (scale * 2.0 ** -10) ** 2, (key, fsse.sum() / max(rfsse.sum(), 1e-30))
    assert fmax <= 2.0 * rfmax + scale * 2.0 ** -10, (key, fmax, rfmax)
    return ratio, bad, fsse.sum() / max(rfsse.sum(), 1e-30)
