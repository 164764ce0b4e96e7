"""ctypes binding of include/dxtex_b200.h.  No codec logic here; no fallback path."""
import ctypes as C
import os
import numpy as np

from . import formats as F

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("DXTEX_B200_LIB") or os.path.join(_HERE, "_lib", "libdxtex_b200.so")     # env override: kernel-variant experiments

SYMBOLS = [
    "dxb200_version", "dxb200_init", "dxb200_init_devices", "dxb200_initialized_devices", "dxb200_shutdown", "dxb200_device_count", "dxb200_launch_count", "dxb200_tma_launch_count", "dxb200_set_option", "dxb200_get_option", "dxb200_last_error",
    "dxb200_host_alloc", "dxb200_host_free", "dxb200_compute_pitch", "dxb200_calculate_mip_levels",
    "dxb200_compress", "dxb200_compress_ex", "dxb200_compress_device", "dxb200_convert_ex", "dxb200_mipmaps_compress", "dxb200_decompress", "dxb200_decompress_device",
    "dxb200_convert", "dxb200_convert_device", "dxb200_generate_mipmaps", "dxb200_generate_mipmaps_device",
    "dxb200_resize", "dxb200_resize_device", "dxb200_premultiply_alpha", "dxb200_premultiply_alpha_device",
    "dxb200_scale_mipmaps_alpha_for_coverage", "dxb200_scale_mipmaps_alpha_for_coverage_device",
    "dxb200_dds_encode_header", "dxb200_dds_save_memory", "dxb200_dds_get_metadata", "dxb200_dds_load_memory",
    "dxb200_compute_mse", "dxb200_compute_mse_device", "dxb200_is_alpha_all_opaque", "dxb200_is_alpha_all_opaque_device",
]


class Image(C.Structure):
    """dxb200_image == DirectX::Image (DirectXTex.h:437-445)."""
    _fields_ = [("width", C.c_size_t), ("height", C.c_size_t), ("format", C.c_uint32),
                ("rowPitch", C.c_size_t), ("slicePitch", C.c_size_t), ("pixels", C.c_void_p)]


class Metadata(C.Structure):
    """dxb200_metadata == DirectX::TexMetadata (DirectXTex.h:187-216)."""
    _fields_ = [("width", C.c_size_t), ("height", C.c_size_t), ("depth", C.c_size_t), ("arraySize", C.c_size_t), ("mipLevels", C.c_size_t),
                ("miscFlags", C.c_uint32), ("miscFlags2", C.c_uint32), ("format", C.c_uint32), ("dimension", C.c_uint32)]


STATUS_FN = C.CFUNCTYPE(C.c_int, C.c_size_t, C.c_size_t, C.c_void_p)      # dxb200_status_fn


class DxTexError(RuntimeError):
    def __init__(self, hr, what):
        self.hr = F.hr_u32(hr)
        super().__init__("%s failed: HRESULT 0x%08X (%s)" % (what, self.hr, last_error()))


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError("libdxtex_b200.so is not built (%s); run `python -c 'import __graft_entry__ as g; g.build()'`. "
                          "There is no CPU fallback." % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    missing = [n for n in SYMBOLS if not hasattr(lib, n)]
    if missing:
        raise ImportError("%s is stale (missing %s); rebuild with `python -c 'import __graft_entry__ as g; g.build()'`" % (LIB_PATH, ", ".join(missing)))
    IP = C.POINTER(Image)
    lib.dxb200_version.restype = C.c_char_p
    lib.dxb200_last_error.restype = C.c_char_p
    lib.dxb200_launch_count.restype = C.c_uint64
    lib.dxb200_tma_launch_count.restype = C.c_uint64
    lib.dxb200_set_option.argtypes = [C.c_uint32, C.c_int32]
    lib.dxb200_get_option.argtypes = [C.c_uint32]
    lib.dxb200_host_alloc.restype = C.c_void_p
    lib.dxb200_host_alloc.argtypes = [C.c_size_t]
    lib.dxb200_host_free.argtypes = [C.c_void_p]
    lib.dxb200_init.argtypes = [C.c_int]
    lib.dxb200_init_devices.argtypes = [C.c_int, C.POINTER(C.c_int)]
    lib.dxb200_initialized_devices.argtypes = [C.POINTER(C.c_int), C.c_int]
    lib.dxb200_compress_ex.argtypes = [IP, C.c_size_t, C.c_uint32, C.c_uint32, C.c_float, C.c_float, IP, STATUS_FN, C.c_void_p]
    lib.dxb200_convert_ex.argtypes = [IP, C.c_size_t, C.c_uint32, C.c_uint32, C.c_float, IP, STATUS_FN, C.c_void_p]
    lib.dxb200_mipmaps_compress.argtypes = [IP, C.c_size_t, C.c_size_t, C.c_uint32, C.c_uint32, C.c_uint32, C.c_float, C.c_float, IP]
    lib.dxb200_compute_pitch.argtypes = [C.c_uint32, C.c_size_t, C.c_size_t, C.POINTER(C.c_size_t), C.POINTER(C.c_size_t)]
    lib.dxb200_calculate_mip_levels.argtypes = [C.c_size_t, C.c_size_t, C.POINTER(C.c_size_t)]
    lib.dxb200_compress.argtypes = [IP, C.c_size_t, C.c_uint32, C.c_uint32, C.c_float, C.c_float, IP]
    lib.dxb200_compress_device.argtypes = [IP, C.c_size_t, C.c_uint32, C.c_uint32, C.c_float, C.c_float, IP, C.c_void_p]
    lib.dxb200_decompress.argtypes = [IP, C.c_size_t, C.c_uint32, IP]
    lib.dxb200_decompress_device.argtypes = [IP, C.c_size_t, C.c_uint32, IP, C.c_void_p]
    lib.dxb200_convert.argtypes = [IP, C.c_size_t, C.c_uint32, C.c_uint32, C.c_float, IP]
    lib.dxb200_convert_device.argtypes = [IP, C.c_size_t, C.c_uint32, C.c_uint32, C.c_float, IP, C.c_void_p]
    lib.dxb200_generate_mipmaps.argtypes = [IP, C.c_size_t, C.c_size_t, C.c_uint32]
    lib.dxb200_generate_mipmaps_device.argtypes = [IP, C.c_size_t, C.c_size_t, C.c_uint32, C.c_void_p]
    lib.dxb200_resize.argtypes = [IP, C.c_size_t, C.c_uint32, IP]
    lib.dxb200_resize_device.argtypes = [IP, C.c_size_t, C.c_uint32, IP, C.c_void_p]
    lib.dxb200_premultiply_alpha.argtypes = [IP, C.c_size_t, C.c_uint32, IP]
    lib.dxb200_premultiply_alpha_device.argtypes = [IP, C.c_size_t, C.c_uint32, IP, C.c_void_p]
    lib.dxb200_scale_mipmaps_alpha_for_coverage.argtypes = [IP, C.c_size_t, C.c_float, IP]
    lib.dxb200_scale_mipmaps_alpha_for_coverage_device.argtypes = [IP, C.c_size_t, C.c_float, IP, C.c_void_p]
    lib.dxb200_scale_mipmaps_alpha_for_coverage.restype = C.c_int32
    lib.dxb200_scale_mipmaps_alpha_for_coverage_device.restype = C.c_int32
    MP, SP = C.POINTER(Metadata), C.POINTER(C.c_size_t)
    lib.dxb200_dds_encode_header.argtypes = [MP, C.c_uint32, C.c_void_p, C.c_size_t, SP]
    lib.dxb200_dds_save_memory.argtypes = [IP, C.c_size_t, MP, C.c_uint32, C.c_void_p, C.c_size_t, SP]
    lib.dxb200_dds_get_metadata.argtypes = [C.c_void_p, C.c_size_t, C.c_uint32, MP, SP]
    lib.dxb200_dds_load_memory.argtypes = [C.c_void_p, C.c_size_t, C.c_uint32, IP, C.c_size_t]
    FP = C.POINTER(C.c_float)
    lib.dxb200_compute_mse.argtypes = [IP, IP, C.c_size_t, C.c_uint32, FP, FP]
    lib.dxb200_compute_mse_device.argtypes = [IP, IP, C.c_size_t, C.c_uint32, C.c_void_p, C.c_void_p]
    lib.dxb200_is_alpha_all_opaque.argtypes = [IP, C.c_size_t, C.POINTER(C.c_int32)]
    lib.dxb200_is_alpha_all_opaque_device.argtypes = [IP, C.c_size_t, C.c_void_p, C.c_void_p]
    for name in ("dxb200_compute_mse", "dxb200_compute_mse_device", "dxb200_is_alpha_all_opaque", "dxb200_is_alpha_all_opaque_device",
                 "dxb200_dds_encode_header", "dxb200_dds_save_memory", "dxb200_dds_get_metadata", "dxb200_dds_load_memory"):
        getattr(lib, name).restype = C.c_int32
    for name in ("dxb200_init", "dxb200_init_devices", "dxb200_initialized_devices", "dxb200_compress_ex", "dxb200_convert_ex", "dxb200_mipmaps_compress", "dxb200_device_count", "dxb200_compute_pitch", "dxb200_calculate_mip_levels", "dxb200_compress",
                 "dxb200_compress_device", "dxb200_decompress", "dxb200_decompress_device", "dxb200_convert",
                 "dxb200_convert_device", "dxb200_generate_mipmaps", "dxb200_generate_mipmaps_device", "dxb200_resize", "dxb200_resize_device", "dxb200_premultiply_alpha", "dxb200_premultiply_alpha_device"):
        getattr(lib, name).restype = C.c_int32
    return lib


lib = _load()


def last_error():
    return (lib.dxb200_last_error() or b"").decode()


def launch_count():
    return int(lib.dxb200_launch_count())


OPT_BC7_FEED = 1


def tma_launch_count():
    return int(lib.dxb200_tma_launch_count())


def make_image(ptr, w, h, fmt, row_pitch=0):
    row, sl = F.compute_pitch(fmt, w, h)
    if row_pitch and row_pitch != row:
        sl = row_pitch * (max(1, (h + 3) // 4) if fmt in F.BLOCK_BYTES else h)
        row = row_pitch
    return Image(w, h, fmt, row, sl, ptr)


def images(seq):
    arr = (Image * len(seq))(*seq)
    return arr


def _np_ptr(a):
    return a.ctypes.data


# ------------------------------------------------------------------------------------------------
# host-pointer calls (numpy in / numpy out) — what a DirectX::Compress caller sees
def compress(src, w, h, src_fmt, dst_fmt, flags=0, threshold=0.5, alpha_weight=1.0):
    """src: C-contiguous numpy array holding the image rows; returns uint8 array of blocks."""
    src = np.ascontiguousarray(src)
    _, sl = F.compute_pitch(dst_fmt, w, h) if dst_fmt in F.BLOCK_BYTES else (0, 0)
    out = np.zeros(max(sl, 1), np.uint8)
    s = images([make_image(_np_ptr(src), w, h, src_fmt)])
    d = images([Image(w, h, dst_fmt, *(F.compute_pitch(dst_fmt, w, h) if dst_fmt in F.BLOCK_BYTES else (0, 0)), _np_ptr(out))])
    hr = lib.dxb200_compress(s, 1, dst_fmt, flags, threshold, alpha_weight, d)
    if hr != 0:
        raise DxTexError(hr, "dxb200_compress")
    return out[:sl]


def init_devices(devices):
    arr = (C.c_int * len(devices))(*devices)
    hr = lib.dxb200_init_devices(len(devices), arr)
    if hr != 0:
        raise DxTexError(hr, "dxb200_init_devices")


def compress_with_status(src, w, h, src_fmt, dst_fmt, callback, flags=0):
    """dxb200_compress_ex of one image; callback(done, total) -> bool (False aborts).  Returns (hr, blocks)."""
    src = np.ascontiguousarray(src)
    row, sl = F.compute_pitch(dst_fmt, w, h)
    out = np.zeros(sl, np.uint8)
    s = images([make_image(_np_ptr(src), w, h, src_fmt)])
    d = images([Image(w, h, dst_fmt, row, sl, _np_ptr(out))])
    cb = STATUS_FN(lambda done, total, user: 1 if callback(done, total) else 0)
    hr = lib.dxb200_compress_ex(s, 1, dst_fmt, flags, 0.5, 1.0, d, cb, None)
    return F.hr_u32(hr), out


def mipmaps_compress(srcs, w, h, src_fmt, dst_fmt, filter=0, levels=0, flags=0):
    """dxb200_mipmaps_compress of an array of equally sized host images; returns one packed BC chain (bytes) per image."""
    srcs = [np.ascontiguousarray(a).view(np.uint8).reshape(-1) for a in srcs]
    levels = levels or F.count_mips(w, h)
    olayout, total = texture_layout(dst_fmt, w, h, 1, levels)
    row, sl = F.compute_pitch(src_fmt, w, h)
    outs = [np.zeros(total, np.uint8) for _ in srcs]
    s = images([Image(w, h, src_fmt, row, sl, _np_ptr(a)) for a in srcs])
    d = images([Image(lw, lh, dst_fmt, r, sp, _np_ptr(o) + off) for o in outs for (off, lw, lh, r, sp) in olayout])
    hr = lib.dxb200_mipmaps_compress(s, len(srcs), levels, filter, dst_fmt, flags, 0.5, 1.0, d)
    if hr != 0:
        raise DxTexError(hr, "dxb200_mipmaps_compress")
    return outs


def compress_array(srcs, w, h, src_fmt, dst_fmt, flags=0, threshold=0.5):
    srcs = [np.ascontiguousarray(s) for s in srcs]
    row, sl = F.compute_pitch(dst_fmt, w, h)
    outs = [np.zeros(sl, np.uint8) for _ in srcs]
    s = images([make_image(_np_ptr(a), w, h, src_fmt) for a in srcs])
    d = images([Image(w, h, dst_fmt, row, sl, _np_ptr(o)) for o in outs])
    hr = lib.dxb200_compress(s, len(srcs), dst_fmt, flags, threshold, 1.0, d)
    if hr != 0:
        raise DxTexError(hr, "dxb200_compress")
    return outs


def convert(src, w, h, src_fmt, dst_fmt, filter=0, threshold=0.5):
    src = np.ascontiguousarray(src)
    if dst_fmt not in F.BYTES_PER_PIXEL:
        out = np.zeros(16, np.uint8)
        d = images([Image(w, h, dst_fmt, 0, 0, _np_ptr(out))])
    else:
        row, sl = F.compute_pitch(dst_fmt, w, h)
        out = np.zeros(sl, np.uint8)
        d = images([Image(w, h, dst_fmt, row, sl, _np_ptr(out))])
    s = images([make_image(_np_ptr(src), w, h, src_fmt) if src_fmt in F.BYTES_PER_PIXEL or src_fmt in F.BLOCK_BYTES
                else Image(w, h, src_fmt, 0, 0, _np_ptr(src))])
    hr = lib.dxb200_convert(s, 1, dst_fmt, filter, threshold, d)
    if hr != 0:
        raise DxTexError(hr, "dxb200_convert")
    return out


def generate_mipmaps(src, w, h, fmt, filter=0, levels=0):
    """Returns (chain bytes laid out as a ScratchImage would, layout list)."""
    src = np.ascontiguousarray(src).view(np.uint8).reshape(-1)
    layout, total = F.mip_chain_layout(fmt, w, h, levels)
    chain = np.zeros(total, np.uint8)
    chain[:layout[0][4]] = src[:layout[0][4]]
    imgs = images([Image(lw, lh, fmt, row, sl, _np_ptr(chain) + off) for (off, lw, lh, row, sl) in layout])
    hr = lib.dxb200_generate_mipmaps(imgs, 1, len(layout), filter)
    if hr != 0:
        raise DxTexError(hr, "dxb200_generate_mipmaps")
    return chain, layout


def resize(src, w, h, fmt, width, height, filter=0):
    """DirectX::Resize of one image; returns the width x height result as tightly packed bytes."""
    src = np.ascontiguousarray(src).view(np.uint8).reshape(-1)
    srow, ssl = F.compute_pitch(fmt, w, h)
    drow, dsl = F.compute_pitch(fmt, width, height)
    out = np.zeros(dsl, np.uint8)
    s = images([Image(w, h, fmt, srow, ssl, _np_ptr(src))])
    d = images([Image(width, height, fmt, drow, dsl, _np_ptr(out))])
    hr = lib.dxb200_resize(s, 1, filter, d)
    if hr != 0:
        raise DxTexError(hr, "dxb200_resize")
    return out


def premultiply_alpha(src, w, h, fmt, flags=0):
    """DirectX::PremultiplyAlpha of one image (flags = TEX_PMALPHA_FLAGS); returns the result bytes."""
    src = np.ascontiguousarray(src).view(np.uint8).reshape(-1)
    row, sl = F.compute_pitch(fmt, w, h)
    out = np.zeros(sl, np.uint8)
    s = images([Image(w, h, fmt, row, sl, _np_ptr(src))])
    d = images([Image(w, h, fmt, row, sl, _np_ptr(out))])
    hr = lib.dxb200_premultiply_alpha(s, 1, flags, d)
    if hr != 0:
        raise DxTexError(hr, "dxb200_premultiply_alpha")
    return out


def texture_layout(fmt, w, h, array_size=1, mip_levels=1):
    """(list of (offset, w, h, rowPitch, slicePitch) item-major / mip-minor, total bytes) as ScratchImage::Initialize lays it out."""
    out, off = [], 0
    for _ in range(array_size):
        lw, lh = w, h
        for _ in range(mip_levels):
            row, sl = F.compute_pitch(fmt, lw, lh)
            out.append((off, lw, lh, row, sl))
            off += sl
            lw, lh = max(1, lw >> 1), max(1, lh >> 1)
    return out, off


def dds_save(pixels, fmt, w, h, array_size=1, mip_levels=1, misc_flags=0, misc_flags2=0, flags=0):
    """SaveToDDSMemory of a 2D texture whose images are packed in `pixels` in ScratchImage order; returns the file bytes."""
    pixels = np.ascontiguousarray(pixels).view(np.uint8).reshape(-1)
    layout, total = texture_layout(fmt, w, h, array_size, mip_levels)
    assert pixels.size == total
    imgs = images([Image(lw, lh, fmt, row, sl, _np_ptr(pixels) + off) for (off, lw, lh, row, sl) in layout])
    md = Metadata(w, h, 1, array_size, mip_levels, misc_flags, misc_flags2, fmt, 3)
    need = C.c_size_t()
    hr = lib.dxb200_dds_save_memory(imgs, len(layout), C.byref(md), flags, None, 0, C.byref(need))
    if hr != 0:
        raise DxTexError(hr, "dxb200_dds_save_memory")
    out = np.zeros(need.value, np.uint8)
    hr = lib.dxb200_dds_save_memory(imgs, len(layout), C.byref(md), flags, _np_ptr(out), out.size, C.byref(need))
    if hr != 0:
        raise DxTexError(hr, "dxb200_dds_save_memory")
    return out


def dds_load(data, flags=0):
    """LoadFromDDSMemory; returns (Metadata, pixels packed in ScratchImage order)."""
    data = np.ascontiguousarray(data).view(np.uint8).reshape(-1)
    md = Metadata()
    off = C.c_size_t()
    hr = lib.dxb200_dds_get_metadata(_np_ptr(data), data.size, flags, C.byref(md), C.byref(off))
    if hr != 0:
        raise DxTexError(hr, "dxb200_dds_get_metadata")
    layout, total = texture_layout(md.format, md.width, md.height, md.arraySize, md.mipLevels)
    pixels = np.zeros(total, np.uint8)
    imgs = images([Image(lw, lh, md.format, row, sl, _np_ptr(pixels) + o) for (o, lw, lh, row, sl) in layout])
    hr = lib.dxb200_dds_load_memory(_np_ptr(data), data.size, flags, imgs, len(layout))
    if hr != 0:
        raise DxTexError(hr, "dxb200_dds_load_memory")
    return md, pixels


def scale_mipmaps_alpha_for_coverage(chain, w, h, fmt, alpha_ref):
    """DirectX::ScaleMipMapsAlphaForCoverage on one mip chain (bytes in ScratchImage layout); returns the new chain."""
    chain = np.ascontiguousarray(chain).view(np.uint8).reshape(-1)
    layout, total = F.mip_chain_layout(fmt, w, h, 0)
    out = np.zeros(total, np.uint8)
    s = images([Image(lw, lh, fmt, row, sl, _np_ptr(chain) + off) for (off, lw, lh, row, sl) in layout])
    d = images([Image(lw, lh, fmt, row, sl, _np_ptr(out) + off) for (off, lw, lh, row, sl) in layout])
    hr = lib.dxb200_scale_mipmaps_alpha_for_coverage(s, len(layout), alpha_ref, d)
    if hr != 0:
        raise DxTexError(hr, "dxb200_scale_mipmaps_alpha_for_coverage")
    return out


def decompress(blocks, w, h, bc_fmt, dst_fmt):
    blocks = np.ascontiguousarray(blocks)
    row, sl = F.compute_pitch(dst_fmt, w, h) if dst_fmt in F.BYTES_PER_PIXEL else (0, 0)
    out = np.zeros(max(sl, 1), np.uint8)
    s = images([make_image(_np_ptr(blocks), w, h, bc_fmt) if bc_fmt in F.BLOCK_BYTES else Image(w, h, bc_fmt, 0, 0, _np_ptr(blocks))])
    d = images([Image(w, h, dst_fmt, row, sl, _np_ptr(out))])
    hr = lib.dxb200_decompress(s, 1, dst_fmt, d)
    if hr != 0:
        raise DxTexError(hr, "dxb200_decompress")
    return out[:sl]


# ------------------------------------------------------------------------------------------------
# ComputeMSE / IsAlphaAllOpaque
CMSE_DEFAULT, CMSE_IMAGE1_SRGB, CMSE_IMAGE2_SRGB = 0, 0x1, 0x2
CMSE_IGNORE_RED, CMSE_IGNORE_GREEN, CMSE_IGNORE_BLUE, CMSE_IGNORE_ALPHA = 0x10, 0x20, 0x40, 0x80
CMSE_IMAGE1_X2_BIAS, CMSE_IMAGE2_X2_BIAS = 0x100, 0x200


def compute_mse_images(a, b, flags=0):
    """dxb200_compute_mse of prepared Image structs (lists of equal length): returns (hr, mse float32[n], mseV float32[n, 4])."""
    n = len(a)
    mse, mse_v = np.zeros(n, np.float32), np.zeros((n, 4), np.float32)
    hr = lib.dxb200_compute_mse(images(a), images(b), n, flags, mse.ctypes.data_as(C.POINTER(C.c_float)), mse_v.ctypes.data_as(C.POINTER(C.c_float)))
    return F.hr_u32(hr), mse, mse_v


def compute_mse(a, fmt_a, b, fmt_b, w, h, flags=0, pitch_a=0, pitch_b=0):
    """DirectX::ComputeMSE of two host images (numpy buffers holding the rows); returns (mse, mseV[4]) as float32."""
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    hr, mse, mse_v = compute_mse_images([make_image(_np_ptr(a), w, h, fmt_a, pitch_a)], [make_image(_np_ptr(b), w, h, fmt_b, pitch_b)], flags)
    if hr != 0:
        raise DxTexError(hr, "dxb200_compute_mse")
    return mse[0], mse_v[0]


def compute_mse_device(a, b, flags, out_ptr, stream=None):
    """dxb200_compute_mse_device: a / b = Image structs holding device pointers, out_ptr = device float[5 n]; returns the HRESULT."""
    return F.hr_u32(lib.dxb200_compute_mse_device(images(a), images(b), len(a), flags, out_ptr, stream))


def is_alpha_all_opaque_images(imgs):
    """dxb200_is_alpha_all_opaque of prepared Image structs (one format): returns (hr, opaque bool)."""
    v = C.c_int32(-1)
    hr = lib.dxb200_is_alpha_all_opaque(images(imgs), len(imgs), C.byref(v))
    return F.hr_u32(hr), v.value == 1


def is_alpha_all_opaque(pixels, layout, fmt):
    """The IsAlphaAllOpaque scan of the images of one texture held in `pixels` at the (offset, w, h, rowPitch, slicePitch) entries
    of `layout` (texture_layout / formats.mip_chain_layout); returns True / False."""
    pixels = np.ascontiguousarray(pixels).view(np.uint8).reshape(-1)
    hr, v = is_alpha_all_opaque_images([Image(lw, lh, fmt, row, sl, _np_ptr(pixels) + off) for (off, lw, lh, row, sl) in layout])
    if hr != 0:
        raise DxTexError(hr, "dxb200_is_alpha_all_opaque")
    return v


def is_alpha_all_opaque_device(imgs, out_ptr, stream=None):
    """dxb200_is_alpha_all_opaque_device: imgs = Image structs holding device pointers, out_ptr = device int32; returns the HRESULT."""
    return F.hr_u32(lib.dxb200_is_alpha_all_opaque_device(images(imgs), len(imgs), out_ptr, stream))
