/* dxtex_b200.h — C ABI of libdxtex_b200.so, the B200 (sm_100a) backend for the DirectXTex hot path:
 * DirectX::Compress / Decompress-side block codecs, DirectX::Convert, DirectX::GenerateMipMaps, DirectX::ComputeMSE.
 *
 * Every entry point names the reference interface it replaces (paths relative to the reference
 * repository microsoft/DirectXTex @ 0bb96f0).  The design precedent inside the reference for an
 * accelerator boundary at per-image granularity is GPUCompressBC::{Initialize,Prepare,Compress}
 * (DirectXTex/BCDirectCompute.cpp:109, 203, 373), used by DirectX::Compress(ID3D11Device*, ...)
 * (DirectXTex/DirectXTexCompressGPU.cpp:249-319).
 *
 * Conventions
 *   - plain C: pointers + sizes, no C++/torch types; all functions return an HRESULT bit pattern
 *     (S_OK = 0; E_INVALIDARG, E_POINTER, E_OUTOFMEMORY, E_FAIL, HRESULT_E_NOT_SUPPORTED as in
 *     DirectXTexP.h:210-234 / SURVEY.md 8(b)).  CUDA failures map to E_FAIL / E_OUTOFMEMORY.
 *   - there is NO CPU fallback: without a CUDA device every compute entry point fails with E_FAIL,
 *     and format pairs the kernels do not implement fail with HRESULT_E_NOT_SUPPORTED.
 *   - `dxb200_image` mirrors DirectX::Image (DirectXTex/DirectXTex.h:437-445) field for field.
 *   - the host-pointer entry points never allocate caller-visible memory: the caller sizes the
 *     destination exactly as ScratchImage::Initialize2D would (DirectXTexImage.cpp:405-455; pitches
 *     from dxb200_compute_pitch == ComputePitch, DirectXTexUtil.cpp:961-1183) and the call fills it.
 *   - `_device` variants take device pointers in the same struct and a CUstream/cudaStream_t
 *     (as void*, may be NULL for the default stream); they only enqueue work.
 *   - thread safety: entry points may be called concurrently from several host threads; each host-pointer call takes one of a
 *     device's two staging lanes (own streams and buffers), so two calls per device really overlap; more wait.
 */
#ifndef DXTEX_B200_H
#define DXTEX_B200_H

#include <stddef.h>
#include <stdint.h>

#if defined(__GNUC__)
#define DXB200_API __attribute__((visibility("default")))
#else
#define DXB200_API
#endif

#ifdef __cplusplus
extern "C" {
#endif

typedef struct dxb200_image
{
    size_t   width;
    size_t   height;
    uint32_t format;      /* DXGI_FORMAT value */
    size_t   rowPitch;
    size_t   slicePitch;
    uint8_t* pixels;
} dxb200_image;

/* library / device management (GPUCompressBC::Initialize, BCDirectCompute.cpp:109) */
DXB200_API const char* dxb200_version(void);
DXB200_API int32_t  dxb200_init(int device);                 /* = dxb200_init_devices(1, &device); idempotent */
/* Multi-GPU inside the library (SURVEY.md 8(b), 8(e); the reference parallelises inside the call too: CompressBC_Parallel,
 * DirectXTexCompress.cpp:210-372).  After dxb200_init_devices(n, devs) every host-pointer entry point shards its work over
 * the n devices: contiguous ranges of images (array calls, mip chains: a chain never spans devices) or of block-row bands
 * (one large image), one host thread and one stream set per device, no collective.  `_device` variants always run on the
 * device that owns the caller's pointers.  Devices can be added by further calls; idempotent per device. */
DXB200_API int32_t  dxb200_init_devices(int ndev, const int* devices);
DXB200_API int32_t  dxb200_initialized_devices(int* devices, int maxDevices);   /* returns how many are initialised */
DXB200_API void     dxb200_shutdown(void);                   /* release cached device / pinned buffers */
DXB200_API int32_t  dxb200_device_count(void);
DXB200_API uint64_t dxb200_launch_count(void);               /* number of kernels this library has launched so far */
DXB200_API uint64_t dxb200_tma_launch_count(void);           /* ... of which fed by TMA tensor-map tile loads (k_compress_bc7_tma) */
/* process-wide tuning options (no reference counterpart; results never depend on them).
 *   DXB200_OPT_BC7_FEED  how k_compress_bc7 gets RGBA32F sources made of full blocks: 0 = direct vector loads, one CTA per 16 blocks,
 *                        1 = persistent CTAs fed by TMA tensor-map tile loads with an atomic tile counter, 2 = the same with statically
 *                        strided tiles, 3 = TMA with one CTA per tile, 4 = automatic (default): 1 for batches of images, 0 for a single
 *                        image -- whichever measured faster.  Initial value: environment variable DXB200_BC7_TMA. */
#define DXB200_OPT_BC7_FEED 1u
DXB200_API int32_t  dxb200_set_option(uint32_t option, int32_t value);      /* E_INVALIDARG for an unknown option */
DXB200_API int32_t  dxb200_get_option(uint32_t option);                     /* -1 for an unknown option */
DXB200_API const char* dxb200_last_error(void);              /* text of the last CUDA error seen by the calling thread's call */

/* pinned host allocations for callers that want full-rate H2D/D2H (optional; any host pointer works) */
DXB200_API void*    dxb200_host_alloc(size_t bytes);
DXB200_API void     dxb200_host_free(void* p);

/* ComputePitch (DirectXTexUtil.cpp:961-1183), CP_FLAGS_NONE, for the implemented formats */
DXB200_API int32_t  dxb200_compute_pitch(uint32_t format, size_t width, size_t height, size_t* rowPitch, size_t* slicePitch);
/* CalculateMipLevels (DirectXTexMipmaps.cpp:359-380): *levels==0 -> full chain */
DXB200_API int32_t  dxb200_calculate_mip_levels(size_t width, size_t height, size_t* levels);

/* DirectX::Compress / CompressEx, single image and array overloads
 * (DirectXTexCompress.cpp:632-845; block walk CompressBC :72-205).
 *   flags     = TEX_COMPRESS_FLAGS (DirectXTex.h:887-917); TEX_COMPRESS_PARALLEL is accepted and ignored
 *   threshold = BC1 alpha threshold (TEX_THRESHOLD_DEFAULT 0.5)
 * src[i] and dst[i] must have equal width/height; dst[i].format == dstFormat, pitches per dxb200_compute_pitch. */
DXB200_API int32_t  dxb200_compress(const dxb200_image* src, size_t nimages, uint32_t dstFormat,
                         uint32_t flags, float threshold, float alphaWeight, const dxb200_image* dst);
DXB200_API int32_t  dxb200_compress_device(const dxb200_image* src, size_t nimages, uint32_t dstFormat,
                                uint32_t flags, float threshold, float alphaWeight, const dxb200_image* dst, void* stream);
/* CompressEx / ConvertEx status callback (DirectXTex.h:929-944; DirectXTexCompress.cpp:115-121, 356-360, 785-837): called with
 * (done, total) before every band of work rows goes to the device -- pixel rows of a single image, images of an array --
 * and with (total, total) at the end; returning 0 stops the call between bands with E_ABORT (0x80004004).  With several
 * devices the callback is serialised but may come from worker threads. */
typedef int (*dxb200_status_fn)(size_t done, size_t total, void* user);
DXB200_API int32_t  dxb200_compress_ex(const dxb200_image* src, size_t nimages, uint32_t dstFormat, uint32_t flags, float threshold,
                            float alphaWeight, const dxb200_image* dst, dxb200_status_fn status, void* user);

/* DirectX::Decompress (DirectXTexCompress.cpp:852-979; DecompressBC :425-535) */
DXB200_API int32_t  dxb200_decompress(const dxb200_image* src, size_t nimages, uint32_t dstFormat, const dxb200_image* dst);
DXB200_API int32_t  dxb200_decompress_device(const dxb200_image* src, size_t nimages, uint32_t dstFormat, const dxb200_image* dst, void* stream);

/* DirectX::Convert / ConvertEx (DirectXTexConvert.cpp:5091-5404; ConvertCustom no-dither path :4888-4908).
 *   filter = TEX_FILTER_FLAGS; TEX_FILTER_DITHER = ordered dithering (StoreScanlineDither :4049-4567 without diffusion errors);
 *   TEX_FILTER_DITHER_DIFFUSION = Floyd-Steinberg error diffusion (serial per image; ConvertCustom :4815-4858) */
DXB200_API int32_t  dxb200_convert(const dxb200_image* src, size_t nimages, uint32_t dstFormat,
                        uint32_t filter, float threshold, const dxb200_image* dst);
DXB200_API int32_t  dxb200_convert_device(const dxb200_image* src, size_t nimages, uint32_t dstFormat,
                               uint32_t filter, float threshold, const dxb200_image* dst, void* stream);
DXB200_API int32_t  dxb200_convert_ex(const dxb200_image* src, size_t nimages, uint32_t dstFormat, uint32_t filter, float threshold,
                           const dxb200_image* dst, dxb200_status_fn status, void* user);

/* DirectX::GenerateMipMaps (DirectXTexMipmaps.cpp:2828-3247; Generate2DMips{Point,Box,Linear,Cubic,Triangle}Filter :907-1602).
 *   chain = items*levels images laid out item-major, mip-minor (TexMetadata::ComputeIndex, DirectXTexUtil.cpp:1695-1741);
 *   level 0 of every item is filled by the caller, levels 1.. are written.
 *   filter = TEX_FILTER_FLAGS; mode 0 selects BOX for power-of-two sizes else LINEAR (:3169-3174). */
DXB200_API int32_t  dxb200_generate_mipmaps(const dxb200_image* chain, size_t items, size_t levels, uint32_t filter);
DXB200_API int32_t  dxb200_generate_mipmaps_device(const dxb200_image* chain, size_t items, size_t levels, uint32_t filter, void* stream);

/* GenerateMipMaps followed by Compress (what texconv does, Texconv/texconv.cpp -m / -f) as ONE call whose mip chain never leaves
 * HBM: base[i] = level 0 of item i (host), dst[i * levels + l] = the compressed image of level l of item i (host, sized by the
 * caller as ScratchImage::Initialize2D(dstFormat, w, h, items, levels) would).  Results are identical to
 * dxb200_generate_mipmaps + dxb200_compress (same kernels); host<->device traffic drops from (1 + 2 x 1.33) x source bytes up/down
 * to the source up and the blocks down.  filter as dxb200_generate_mipmaps, flags / threshold as dxb200_compress. */
DXB200_API int32_t  dxb200_mipmaps_compress(const dxb200_image* base, size_t items, size_t levels, uint32_t filter, uint32_t dstFormat,
                                 uint32_t flags, float threshold, float alphaWeight, const dxb200_image* dst);

/* DirectX::Resize (DirectXTexResize.cpp:854-935 single image, :942-1120 arrays; custom filters ResizePointFilter /
 * ResizeBoxFilter / ResizeLinearFilter / ResizeCubicFilter / ResizeTriangleFilter :255-798, selection :805-837).
 *   src[i] -> dst[i], i < nimages; all sources share one size and format, all destinations share one size and the
 *   source format.  filter = TEX_FILTER_FLAGS; mode 0 selects BOX when the target is exactly half the source in both
 *   directions, else LINEAR (:812-817); BOX on any other ratio -> E_FAIL (:318-319); compressed formats ->
 *   HRESULT_E_NOT_SUPPORTED (:875-879).  (SURVEY 8(f) rank 2: the texconv step in front of Convert.) */
DXB200_API int32_t  dxb200_resize(const dxb200_image* src, size_t nimages, uint32_t filter, const dxb200_image* dst);
DXB200_API int32_t  dxb200_resize_device(const dxb200_image* src, size_t nimages, uint32_t filter, const dxb200_image* dst, void* stream);

/* DirectX::PremultiplyAlpha (DirectXTexPMAlpha.cpp:214-344; PremultiplyAlpha_ / PremultiplyAlphaLinear / DemultiplyAlpha /
 * DemultiplyAlphaLinear :30-208).  src[i] -> dst[i], same size and format; flags = TEX_PMALPHA_FLAGS (DirectXTex.h:860-879):
 * 0x1 IGNORE_SRGB, 0x2 REVERSE (premultiplied -> straight), 0x1000000 / 0x2000000 SRGB_IN / SRGB_OUT.
 * Formats without alpha or compressed -> HRESULT_E_NOT_SUPPORTED (:224-229).  (SURVEY 8(f) rank 4, first part.) */
DXB200_API int32_t  dxb200_premultiply_alpha(const dxb200_image* src, size_t nimages, uint32_t flags, const dxb200_image* dst);
DXB200_API int32_t  dxb200_premultiply_alpha_device(const dxb200_image* src, size_t nimages, uint32_t flags, const dxb200_image* dst, void* stream);

/* DirectX::ScaleMipMapsAlphaForCoverage (DirectXTexMipmaps.cpp:3483-3552; CalculateAlphaCoverage :213-308,
 * EstimateAlphaScaleForCoverage :310-355, ScaleAlpha :143-193) for ONE array item: src[0..nlevels) = its mip levels as
 * GenerateMipMaps produced them, dst[0..nlevels) = the same levels of the result.  Level 0 is copied; every other level's
 * alpha is scaled so that its alpha-test coverage at `alphaReference` matches level 0's (10-step bisection).
 * (SURVEY 8(f) rank 4.)  The _device variant synchronises `stream` internally (the bisection reads counts back). */
DXB200_API int32_t  dxb200_scale_mipmaps_alpha_for_coverage(const dxb200_image* src, size_t nlevels, float alphaReference, const dxb200_image* dst);
DXB200_API int32_t  dxb200_scale_mipmaps_alpha_for_coverage_device(const dxb200_image* src, size_t nlevels, float alphaReference,
                                                                   const dxb200_image* dst, void* stream);

/* DirectX::ComputeMSE (DirectXTexMisc.cpp:388-468) for n pairs a[i] vs b[i] (same width / height per pair; any implemented format on
 * either side, BC included: BC data is decoded in the kernel exactly as Decompress(..., R32G32B32A32_FLOAT) would).
 *   flags = CMSE_FLAGS (DirectXTex.h:1022-1038); the flags implied by the formats (:46-91) are added per pair.
 *   mse[i] and mseV[4 * i .. 4 * i + 3] (mseV may be NULL) as the reference returns them.
 * Per-pixel squares are the reference's fp32 values (up to a few ulp of powf with the sRGB flags); they are summed in fp64 over a
 * reduction tree fixed by the image geometry (dxb_analyze.cuh), so mseV is within 4 fp32 ulp of the exact mean of those squares
 * and bit-identical across calls, batch compositions, device counts and the host / device variants.  The reference's running
 * fp32 sum drifts from the exact value as images grow (~1e-3 relative at 1024^2).
 * Errors: NULL pixels -> E_POINTER; size mismatch or invalid format -> E_INVALIDARG; typeless / planar / palettized or any
 * other valid format this backend does not implement -> HRESULT_E_NOT_SUPPORTED; no device -> E_FAIL.
 * _device: device images, out = 5 floats per pair on the device (mse, then mseV); only enqueues work on `stream`. */
DXB200_API int32_t  dxb200_compute_mse(const dxb200_image* a, const dxb200_image* b, size_t n, uint32_t flags, float* mse, float* mseV);
DXB200_API int32_t  dxb200_compute_mse_device(const dxb200_image* a, const dxb200_image* b, size_t n, uint32_t flags, float* out, void* stream);
/* The image scan of ScratchImage::IsAlphaAllOpaque (DirectXTexImage.cpp:800-852; IsAlphaAllOpaqueBC, DirectXTexCompress.cpp:539-620) over
 * n images of one format: *opaque = 1 when no in-image pixel has alpha < 0.997 (uncompressed, after load) or < 0.99 (BC1/2/3/7, after
 * decode), else 0; BC4 / BC5 / BC6H give 0 as IsAlphaAllOpaqueBC does (the HasAlpha test of the ScratchImage member comes first in
 * the C++ mirror).  Errors as dxb200_compute_mse.  _device: device images and a device int32; only enqueues work. */
DXB200_API int32_t  dxb200_is_alpha_all_opaque(const dxb200_image* images, size_t n, int32_t* opaque);
DXB200_API int32_t  dxb200_is_alpha_all_opaque_device(const dxb200_image* images, size_t n, int32_t* opaque, void* stream);

/* ---- DDS container (host-side only, no GPU work; SURVEY 8(f) rank 3) ------------------------------------------------
 * dxb200_metadata is a field-for-field mirror of DirectX::TexMetadata (DirectXTex.h:187-216).
 * EncodeDDSHeader (DirectXTexDDS.cpp:711-1043), SaveToDDSMemory (:2403-2620), GetMetadataFromDDSMemory / DecodeDDSHeader
 * (:319-683, 1960-2003), LoadFromDDSMemory (:2008-2100).  TEXTURE2D resources (arrays, cubemaps, mip chains) in the
 * formats this library implements; flags = DDS_FLAGS (DirectXTex.h:232-279): FORCE_DX10_EXT, FORCE_DX10_EXT_MISC2,
 * FORCE_DX9_LEGACY, FORCE_DXT5_RXGB, IGNORE_MIPS, ALLOW_LARGE_FILES are honoured (HRESULT_E_CANNOT_MAKE as in the
 * reference when a format has no legacy encoding); load-side conversion / legacy-expansion flags -> HRESULT_E_NOT_SUPPORTED.
 * save/encode: dst == NULL only computes *required.  load: `images` describes the destination (item-major, mip-minor)
 * as ScratchImage::Initialize(metadata) lays it out. */
typedef struct dxb200_metadata
{
    size_t   width, height, depth, arraySize, mipLevels;
    uint32_t miscFlags, miscFlags2;
    uint32_t format;        /* DXGI_FORMAT */
    uint32_t dimension;     /* TEX_DIMENSION: 3 = TEXTURE2D */
} dxb200_metadata;
DXB200_API int32_t  dxb200_dds_encode_header(const dxb200_metadata* metadata, uint32_t flags, void* dst, size_t maxsize, size_t* required);
DXB200_API int32_t  dxb200_dds_save_memory(const dxb200_image* images, size_t nimages, const dxb200_metadata* metadata, uint32_t flags,
                                           void* dst, size_t maxsize, size_t* required);
DXB200_API int32_t  dxb200_dds_get_metadata(const void* src, size_t size, uint32_t flags, dxb200_metadata* metadata, size_t* dataOffset);
DXB200_API int32_t  dxb200_dds_load_memory(const void* src, size_t size, uint32_t flags, const dxb200_image* images, size_t nimages);

#ifdef __cplusplus
}
#endif
#endif /* DXTEX_B200_H */
