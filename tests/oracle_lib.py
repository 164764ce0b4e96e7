"""TEST INFRASTRUCTURE: the reference's answers to the calls the tests make (tests/golden/reference_calls.npz, replayed by
`Recorded`), ctypes access to the oracle that recorded them (oracle/_ref/libdxtex_ref.so = the unmodified reference sources,
`Ref`) and the host lock-step emulator of our own kernels (tests/emul).  Never imported by the product."""
import ctypes as C
import hashlib
import json
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_SO = os.path.join(ROOT, "oracle", "_ref", "libdxtex_ref.so")
EMUL_SO = os.path.join(ROOT, "tests", "emul", "_build", "libdxb_emul.so")
CALLS = os.path.join(ROOT, "tests", "golden", "reference_calls.npz")

from directxtex_b200 import formats as F


def build_ref():
    if not os.path.exists(REF_SO):
        raise RuntimeError("oracle/_ref/libdxtex_ref.so missing: build it with `make -C oracle REF=<DirectXTex checkout>`")
    return REF_SO


def build_emul(force=False):
    srcs = [os.path.join(ROOT, "tests", "emul", "emul.cpp")]
    cs = os.path.join(ROOT, "directxtex_b200", "csrc")
    srcs += [os.path.join(cs, f) for f in os.listdir(cs)]
    stale = (not os.path.exists(EMUL_SO)) or any(os.path.getmtime(s) > os.path.getmtime(EMUL_SO) for s in srcs)
    if force or stale:
        subprocess.run([os.path.join(ROOT, "tests", "emul", "build.sh")], check=True, stdout=subprocess.DEVNULL)
    return EMUL_SO


class Ref:
    def __init__(self, path):
        L = self.L = C.CDLL(path)
        sz, u32, vp, f32 = C.c_size_t, C.c_uint32, C.c_void_p, C.c_float
        L.ref_compress.argtypes = [vp, sz, sz, u32, sz, u32, u32, f32, vp, sz]
        L.ref_compress_timed.argtypes = [vp, sz, sz, u32, sz, u32, u32, f32]
        L.ref_compress_timed.restype = C.c_double
        L.ref_decompress.argtypes = [vp, sz, sz, u32, u32, vp, sz]
        L.ref_convert.argtypes = [vp, sz, sz, u32, sz, u32, u32, f32, vp, sz]
        L.ref_convert_timed.argtypes = [vp, sz, sz, u32, u32, u32, f32]
        L.ref_convert_timed.restype = C.c_double
        L.ref_generate_mipmaps.argtypes = [vp, sz, sz, u32, sz, u32, sz, vp, sz, C.POINTER(sz), C.POINTER(sz)]
        L.ref_generate_mipmaps_timed.argtypes = [vp, sz, sz, u32, u32, sz]
        L.ref_resize.argtypes = [vp, sz, sz, u32, sz, sz, sz, u32, vp, sz]
        L.ref_premultiply_alpha.argtypes = [vp, sz, sz, u32, sz, u32, vp, sz]
        L.ref_mips_alpha_coverage.argtypes = [vp, sz, sz, u32, u32, C.c_float, vp, sz, vp]
        L.ref_dds_save.argtypes = [vp, sz, vp, u32, vp, sz, C.POINTER(sz)]
        L.ref_dds_load.argtypes = [vp, sz, u32, vp, vp, sz, C.POINTER(sz)]
        L.ref_generate_mipmaps_timed.restype = C.c_double
        L.ref_compute_mse.argtypes = [vp, u32, vp, u32, sz, sz, C.POINTER(f32), C.POINTER(f32), u32]
        L.ref_encode_block.argtypes = [u32, vp, u32, f32, vp]
        L.ref_decode_blocks.argtypes = [u32, vp, sz, vp]
        L.ref_compute_pitch.argtypes = [u32, sz, sz, C.POINTER(sz), C.POINTER(sz)]
        L.ref_omp_set_threads.argtypes = [C.c_int]

    def threads(self):
        return self.L.ref_omp_max_threads()

    def compute_pitch(self, fmt, w, h):
        r, s = C.c_size_t(), C.c_size_t()
        hr = self.L.ref_compute_pitch(fmt, w, h, r, s)
        return hr, r.value, s.value

    def compress(self, src, w, h, src_fmt, dst_fmt, flags=0, threshold=0.5, parallel=True):
        src = np.ascontiguousarray(src)
        _, sl = F.compute_pitch(dst_fmt, w, h)
        out = np.zeros(sl, np.uint8)
        hr = self.L.ref_compress(src.ctypes.data, w, h, src_fmt, 0, dst_fmt, flags | (F.TEX_COMPRESS_PARALLEL if parallel else 0),
                                 threshold, out.ctypes.data, out.nbytes)
        return F.hr_u32(hr), out

    def compress_seconds(self, src, w, h, src_fmt, dst_fmt, flags=0, threshold=0.5, parallel=True):
        src = np.ascontiguousarray(src)
        return self.L.ref_compress_timed(src.ctypes.data, w, h, src_fmt, 0, dst_fmt,
                                         flags | (F.TEX_COMPRESS_PARALLEL if parallel else 0), threshold)

    def convert(self, src, w, h, src_fmt, dst_fmt, filter=0, threshold=0.5):
        src = np.ascontiguousarray(src)
        n = w * h * F.BYTES_PER_PIXEL.get(dst_fmt, 16)
        out = np.zeros(n, np.uint8)
        hr = self.L.ref_convert(src.ctypes.data, w, h, src_fmt, 0, dst_fmt, filter, threshold, out.ctypes.data, n)
        return F.hr_u32(hr), out

    def generate_mipmaps(self, src, w, h, fmt, filter=0, levels=0):
        src = np.ascontiguousarray(src)
        _, total = F.mip_chain_layout(fmt, w, h, levels)
        out = np.zeros(total, np.uint8)
        nl, nb = C.c_size_t(), C.c_size_t()
        hr = self.L.ref_generate_mipmaps(src.ctypes.data, w, h, fmt, 0, filter, levels, out.ctypes.data, total, nl, nb)
        return F.hr_u32(hr), out

    def resize(self, src, w, h, fmt, width, height, filter=0):
        src = np.ascontiguousarray(src)
        n = width * height * F.BYTES_PER_PIXEL[fmt]
        out = np.zeros(n, np.uint8)
        hr = self.L.ref_resize(src.ctypes.data, w, h, fmt, 0, width, height, filter, out.ctypes.data, n)
        return F.hr_u32(hr), out

    def premultiply_alpha(self, src, w, h, fmt, flags=0):
        src = np.ascontiguousarray(src)
        n = w * h * F.BYTES_PER_PIXEL[fmt]
        out = np.zeros(n, np.uint8)
        hr = self.L.ref_premultiply_alpha(src.ctypes.data, w, h, fmt, 0, flags, out.ctypes.data, n)
        return F.hr_u32(hr), out

    def mips_alpha_coverage(self, src, w, h, fmt, alpha_ref, filter=0):
        """(hr, plain GenerateMipMaps chain, chain after ScaleMipMapsAlphaForCoverage)"""
        src = np.ascontiguousarray(src)
        _, total = F.mip_chain_layout(fmt, w, h, 0)
        out, plain = np.zeros(total, np.uint8), np.zeros(total, np.uint8)
        hr = self.L.ref_mips_alpha_coverage(src.ctypes.data, w, h, fmt, filter, alpha_ref, out.ctypes.data, total, plain.ctypes.data)
        return F.hr_u32(hr), plain, out

    def dds_save(self, pixels, fmt, w, h, array_size=1, mip_levels=1, misc_flags=0, misc_flags2=0, flags=0):
        pixels = np.ascontiguousarray(pixels).view(np.uint8).reshape(-1)
        meta = np.array([w, h, array_size, mip_levels, fmt, misc_flags, misc_flags2], np.uint64)
        out = np.zeros(pixels.size + 256, np.uint8)
        n = C.c_size_t()
        hr = self.L.ref_dds_save(pixels.ctypes.data, pixels.size, meta.ctypes.data, flags, out.ctypes.data, out.size, n)
        return F.hr_u32(hr), out[:n.value]

    def dds_load(self, data, flags=0):
        data = np.ascontiguousarray(data).view(np.uint8).reshape(-1)
        meta = np.zeros(7, np.uint64)
        out = np.zeros(data.size * 2 + 64, np.uint8)
        n = C.c_size_t()
        hr = self.L.ref_dds_load(data.ctypes.data, data.size, flags, meta.ctypes.data, out.ctypes.data, out.size, n)
        return F.hr_u32(hr), [int(v) for v in meta], out[:n.value]

    def decompress(self, blocks, w, h, bc_fmt, dst_fmt):
        blocks = np.ascontiguousarray(blocks)
        n = w * h * F.BYTES_PER_PIXEL[dst_fmt]
        out = np.zeros(n, np.uint8)
        hr = self.L.ref_decompress(blocks.ctypes.data, w, h, bc_fmt, dst_fmt, out.ctypes.data, n)
        return F.hr_u32(hr), out

    def decode_blocks(self, fmt, blocks, w, h):
        """BC blocks (row-major block order) -> float32 image (h4*4, w4*4, 4) via D3DXDecodeBC*."""
        nbx, nby = (w + 3) // 4, (h + 3) // 4
        blocks = np.ascontiguousarray(blocks)
        dec = np.zeros((nbx * nby, 16, 4), np.float32)
        hr = self.L.ref_decode_blocks(fmt, blocks.ctypes.data, nbx * nby, dec.ctypes.data)
        assert hr == 0
        return dec.reshape(nby, nbx, 4, 4, 4).transpose(0, 2, 1, 3, 4).reshape(nby * 4, nbx * 4, 4)[:h, :w]

    def encode_block(self, fmt, rgba16x4, bcflags=0, threshold=0.5):
        px = np.ascontiguousarray(rgba16x4, np.float32)
        out = np.zeros(16, np.uint8)
        hr = self.L.ref_encode_block(fmt, px.ctypes.data, bcflags, threshold, out.ctypes.data)
        assert hr == 0
        return out[:F.BLOCK_BYTES[fmt]]

    def mipchain_layout(self, fmt, w, h, levels=0):
        """(hr, level count, total bytes, [(offset, width, height, row pitch) per level])"""
        A = C.c_size_t * 16
        nl, tot = C.c_size_t(), C.c_size_t()
        off, ws, hs, ps = A(), A(), A(), A()
        self.L.ref_mipchain_layout.argtypes = [C.c_uint32, C.c_size_t, C.c_size_t, C.c_size_t, C.POINTER(C.c_size_t), C.POINTER(C.c_size_t)] + [C.POINTER(C.c_size_t)] * 4 + [C.c_size_t]
        hr = self.L.ref_mipchain_layout(fmt, w, h, levels, nl, tot, off, ws, hs, ps, 16)
        return F.hr_u32(hr), nl.value, tot.value, [[off[i], ws[i], hs[i], ps[i]] for i in range(nl.value)]

    def bc7_block_sse(self, src_f32, w, h, flags=0):
        """(hr, per-block sum of squared 8-bit RGBA differences of the reference encoder's BC7 blocks, float32 (h/4, w/4))"""
        hr, blocks = self.compress(src_f32, w, h, 2, 98, flags)
        d = self.decode_blocks(98, blocks, w, h).astype(np.float64) * 255.0 - bc7_ldr(src_f32).astype(np.float64)
        return hr, (d ** 2).reshape(h // 4, 4, w // 4, 4, 4).sum((1, 3, 4)).astype(np.float32)


def _digest(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()[:16]


class Digest:
    """A reference output (bytes) kept as a SHA-256 prefix and its length instead of the bytes: `same` compares an array with it."""

    def __init__(self, hexdigest, nbytes):
        self.hex, self.nbytes, self.size = hexdigest, nbytes, nbytes

    def __repr__(self):
        return "Digest(%s)" % self.hex


def same(a, b):
    """np.array_equal for arrays; byte equality of the other side where one side is a Digest"""
    if isinstance(a, Digest) or isinstance(b, Digest):
        return (a.hex if isinstance(a, Digest) else _digest(a)) == (b.hex if isinstance(b, Digest) else _digest(b))
    return np.array_equal(a, b)


def same_concat(got, wants, sizes):
    """`same` for an output made of consecutive pieces of the given byte sizes"""
    offs = np.cumsum([0] + list(sizes))
    return got.size == offs[-1] and all(same(got[o:o + n], w) for o, n, w in zip(offs, sizes, wants))


def _call_key(name, args, kwargs):
    h = hashlib.sha256(name.encode())
    for a in list(args) + [kwargs[k] for k in sorted(kwargs)]:
        if isinstance(a, np.ndarray):
            a = np.ascontiguousarray(a)
            h.update(("%s%s" % (a.dtype.str, a.shape)).encode())
            h.update(a.tobytes())
        elif isinstance(a, (float, np.floating)):
            h.update(repr(float(a)).encode())
        else:
            h.update(repr(int(a)).encode())
    h.update(repr(sorted(kwargs)).encode())
    return h.hexdigest()[:16]


def _encode(v, full, arrays):
    if isinstance(v, np.ndarray):
        d = _digest(v)
        if full:
            arrays["a_" + d] = v
            return {"a": d}
        return {"d": d, "n": int(v.nbytes)}
    if isinstance(v, (list, tuple)):
        return [_encode(x, full, arrays) for x in v]
    return int(v)


def _decode(v, z):
    if isinstance(v, dict):
        return z["a_" + v["a"]] if "a" in v else Digest(v["d"], v["n"])
    if isinstance(v, list):
        return [_decode(x, z) for x in v]
    return v


class Recorded:
    """The reference's answers, replayed from tests/golden/reference_calls.npz: the same methods as `Ref`, looked up by a hash
    of the method name and every argument.  Array outputs come back as `Digest`s, or as arrays where the caller passes
    full=True (the tests that measure a difference instead of asserting equality)."""

    def __init__(self, path=CALLS):
        self.z = np.load(path)
        self.calls = json.loads(bytes(self.z["calls"]).decode())

    def __getattr__(self, name):
        if name.startswith("_") or name in ("z", "calls"):
            raise AttributeError(name)

        def call(*args, full=False, **kwargs):
            key = _call_key(name, args, kwargs)
            if key not in self.calls:
                raise KeyError("no recorded reference answer for %s with these arguments (tests/golden/reference_calls.npz is recorded "
                               "by running the suite with DXB_RECORD_REFERENCE set, see tests/conftest.py)" % name)
            return tuple(_decode(v, self.z) for v in self.calls[key])
        return call


class Recorder:
    """Wraps the live `Ref` and records each call as `Recorded` will replay it; `save` writes the file.  Callers get what the
    replay gives, so a recording run exercises the same comparisons as a replay."""

    def __init__(self, ref):
        self.ref, self.calls, self.arrays = ref, {}, {}

    def __getattr__(self, name):
        if name.startswith("_") or name in ("ref", "calls", "arrays"):
            raise AttributeError(name)

        def call(*args, full=False, **kwargs):
            rec = [_encode(v, full, self.arrays) for v in getattr(self.ref, name)(*args, **kwargs)]
            self.calls[_call_key(name, args, kwargs)] = rec
            return tuple(_decode(v, self.arrays) for v in rec)
        return call

    def save(self, path):
        old = Recorded(path) if os.path.exists(path) else None
        calls = dict(old.calls) if old else {}
        arrays = {k: old.z[k] for k in old.z.files if k.startswith("a_")} if old else {}
        calls.update(self.calls)
        arrays.update(self.arrays)
        used = {"a_" + v["a"] for rec in calls.values() for v in _flat(rec) if isinstance(v, dict) and "a" in v}
        np.savez_compressed(path, calls=np.frombuffer(json.dumps(calls, sort_keys=True).encode(), np.uint8),
                            **{k: v for k, v in arrays.items() if k in used})


def _flat(v):
    if isinstance(v, list):
        for x in v:
            yield from _flat(x)
    else:
        yield v


class Emul:
    def __init__(self, path):
        L = self.L = C.CDLL(path)
        sz, u32, vp, f32 = C.c_size_t, C.c_uint32, C.c_void_p, C.c_float
        L.emul_compress.argtypes = [vp, sz, sz, u32, sz, u32, u32, f32, vp]
        L.emul_convert.argtypes = [vp, sz, sz, u32, sz, u32, sz, u32, vp]
        L.emul_generate_mipmaps.argtypes = [vp] + [C.POINTER(sz)] * 4 + [sz, u32, u32]
        L.emul_scale_mips_alpha.argtypes = [vp, vp] + [C.POINTER(sz)] * 4 + [sz, u32, C.c_float]
        L.emul_decompress.argtypes = [vp, sz, sz, u32, u32, vp]

    def compress(self, src, w, h, src_fmt, dst_fmt, flags=0, threshold=0.5):
        src = np.ascontiguousarray(src)
        _, sl = F.compute_pitch(dst_fmt, w, h)
        out = np.zeros(sl, np.uint8)
        hr = self.L.emul_compress(src.ctypes.data, w, h, src_fmt, 0, dst_fmt, flags, threshold, out.ctypes.data)
        return F.hr_u32(hr), out

    def convert(self, src, w, h, src_fmt, dst_fmt, filter=0):
        src = np.ascontiguousarray(src)
        out = np.zeros(w * h * F.BYTES_PER_PIXEL[dst_fmt], np.uint8)
        hr = self.L.emul_convert(src.ctypes.data, w, h, src_fmt, 0, dst_fmt, 0, filter, out.ctypes.data)
        return F.hr_u32(hr), out

    def decompress(self, blocks, w, h, bc_fmt, dst_fmt):
        blocks = np.ascontiguousarray(blocks)
        out = np.zeros(w * h * F.BYTES_PER_PIXEL[dst_fmt], np.uint8)
        hr = self.L.emul_decompress(blocks.ctypes.data, w, h, bc_fmt, dst_fmt, out.ctypes.data)
        return F.hr_u32(hr), out

    def decode_blocks(self, fmt, blocks, w, h):
        """BC blocks -> float32 image (h, w, 4): Decompress to R32G32B32A32_FLOAT, which the tests hold bit-exact to the reference
        decoder (test_emulator_decompress_bit_exact)"""
        hr, out = self.decompress(blocks, w, h, fmt, F.DXGI_FORMAT_R32G32B32A32_FLOAT)
        assert hr == 0
        return out.view(np.float32).reshape(h, w, 4)

    def generate_mipmaps(self, src, w, h, fmt, filter=0, levels=0):
        layout, total = F.mip_chain_layout(fmt, w, h, levels)
        chain = np.zeros(total, np.uint8)
        s = np.ascontiguousarray(src).view(np.uint8).reshape(-1)
        chain[:layout[0][4]] = s[:layout[0][4]]
        A = C.c_size_t * len(layout)
        off, ws, hs, ps = A(*[l[0] for l in layout]), A(*[l[1] for l in layout]), A(*[l[2] for l in layout]), A(*[l[3] for l in layout])
        hr = self.L.emul_generate_mipmaps(chain.ctypes.data, off, ws, hs, ps, len(layout), fmt, filter)
        return F.hr_u32(hr), chain

    def scale_mips_alpha(self, chain, w, h, fmt, alpha_ref):
        layout, total = F.mip_chain_layout(fmt, w, h, 0)
        chain = np.ascontiguousarray(chain).view(np.uint8).reshape(-1)
        out = np.zeros(total, np.uint8)
        A = C.c_size_t * len(layout)
        off, ws, hs, ps = A(*[l[0] for l in layout]), A(*[l[1] for l in layout]), A(*[l[2] for l in layout]), A(*[l[3] for l in layout])
        hr = self.L.emul_scale_mips_alpha(chain.ctypes.data, out.ctypes.data, off, ws, hs, ps, len(layout), fmt, alpha_ref)
        return F.hr_u32(hr), out


def load_ref():
    return Ref(build_ref())


def load_reference_answers():
    """`Recorded`, or a `Recorder` on the reference build when DXB_RECORD_REFERENCE names the file to record into"""
    path = os.environ.get("DXB_RECORD_REFERENCE")
    return Recorder(load_ref()) if path else Recorded()


def load_emul():
    return Emul(build_emul())


# ---- shared helpers ---------------------------------------------------------------------------------
def bc7_ldr(img_f32):
    """the reference's LDR staging (BC6HBC7.cpp:2794-2797) as float 0..255"""
    t = img_f32.astype(np.float32) * np.float32(255.0) + np.float32(0.01)
    return np.floor(np.clip(t, 0, 255)).astype(np.float32)


def mse255(decoded01, src_f32):
    d = decoded01.astype(np.float64) * 255.0
    s = bc7_ldr(src_f32).astype(np.float64)
    return float(((d - s) ** 2).mean())


def psnr(mse):
    return 10.0 * np.log10(255.0 ** 2 / max(mse, 1e-12))


def random_image(fmt, w, h, rng):
    bpp = F.BYTES_PER_PIXEL[fmt]
    n = w * h * bpp
    if fmt == 26:       # R11G11B10_FLOAT: every bit pattern except Inf / NaN (exponent 31): outside the parity contract like NaN inputs elsewhere
        v = rng.integers(0, 1 << 32, w * h, dtype=np.uint64).astype(np.uint32)
        return (v & ~np.uint32((1 << 10) | (1 << 21) | (1 << 31))).view(np.uint8)
    if fmt in (2, 6, 16, 41):
        return (rng.random(n // 4).astype(np.float32) * 1.4 - 0.2).view(np.uint8)
    if fmt in (10, 34, 54):
        return (rng.random(n // 2) * 1.4 - 0.2).astype(np.float16).view(np.uint8)
    return rng.integers(0, 256, n, dtype=np.uint8)


def bc6h_to_int(img_f, signed=False):
    """the reference's INTColor domain (F16ToINT, BC6HBC7.cpp:534-552) of an RGB(A) float image"""
    h = np.asarray(img_f, np.float32).astype(np.float16).view(np.uint16).astype(np.int64)
    if signed:
        m = np.minimum(h & 0x7FFF, 0x7BFF)
        return np.where(h & 0x8000, -m, m)
    return np.where(h & 0x8000, 0, h)


def bc6h_int_mse(decoded, src_f32, signed=False):
    """mean squared difference of half-float bit patterns over RGB: the reference encoder's own error metric"""
    a = bc6h_to_int(decoded[..., :3], signed)
    b = bc6h_to_int(np.clip(src_f32[..., :3], -65504 if signed else 0, 65504), signed)
    return float(((a - b).astype(np.float64) ** 2).mean())


def bc6h_test_image(kind, w, h, seed):
    from directxtex_b200 import synth
    rng = np.random.default_rng(seed)
    y, x = np.mgrid[0:h, 0:w].astype(np.float32)
    if kind == "c3":
        return np.ascontiguousarray(synth.c3_rgba16f(w, h, seed=seed).astype(np.float32))
    smooth = np.stack([np.exp2(4 * np.sin(x * 0.05) + 2 * np.cos(y * 0.03)), np.exp2(3 * np.cos(x * 0.02 + y * 0.04)),
                       np.exp2(2 * np.sin(y * 0.06)), np.ones_like(x)], -1).astype(np.float32)
    if kind == "smooth":
        return np.ascontiguousarray((smooth * (1 + 0.02 * rng.normal(size=smooth.shape))).astype(np.float32))
    if kind == "edges":
        e = np.where(((x // 4 + y // 4) % 3 == 0)[..., None] & ((x % 4) < 2)[..., None], np.float32(50.0), smooth)
        return np.ascontiguousarray(e.astype(np.float32))
    if kind == "signed":
        v = smooth - np.float32(3.0)
        v[..., 3] = 1
        return np.ascontiguousarray(v.astype(np.float32))
    raise ValueError(kind)
