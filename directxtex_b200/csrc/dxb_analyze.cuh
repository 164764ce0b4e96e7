// dxb_analyze.cuh — whole-image reductions over decoded pixels, shared by k_compute_mse / k_alpha_opaque (dxb_k_analyze.cu), the
// host API (dxb_api.cu: implied flags, the image-level tree of the host-pointer variant) and the host emulator (tests/emul):
//   ComputeMSE               DirectXTexMisc.cpp:27-176 (ComputeMSE_), :388-468 (BC inputs: Decompress to R32G32B32A32_FLOAT first)
//   IsAlphaAllOpaque scan    DirectXTexImage.cpp:800-852, IsAlphaAllOpaqueBC DirectXTexCompress.cpp:539-620
//
// Numerical contract of ComputeMSE:
//   - per pixel, the reference's fp32 statements in its order: pow(v, {2.2, 2.2, 2.2, 1}) for the sRGB flags, v*2 - 1 (unfused) for
//     the X2_BIAS flags, d = v1 - v2, the IGNORE masks (a select, so a NaN channel that is ignored counts 0), d*d rounded to fp32.
//     powf differs by a few ulp between CUDA and glibc, so only the gamma flag leaves the bits of the reference's squares.
//   - the squares are summed in fp64 over a tree fixed by the image geometry alone:
//       tile  = the <= 16 in-image pixels of one 4x4 tile, summed in row order;
//       chunk = DXB_AN_TILES consecutive tiles of one tile row (the last chunk of a row is short), halving tree over the slots;
//       image = lane t (t < DXB_AN_TILES) sums chunks t, t + DXB_AN_TILES, ... in order, then the same halving tree.
//     No float atomics: the result does not depend on grid size, device count, batch composition or host versus device variant.
//   - mseV[c] = float(sum[c]) / float(w*h), mse = ((mseV[0] + mseV[1]) + mseV[2]) + mseV[3] in fp32, as the reference finishes.
//     mseV is within 4 fp32 ulp of float(exact sum of the reference's squares) / float(w*h); the reference's own running fp32 sum
//     drifts from that by up to ~1e-3 relative at 1024^2 and by percents at 4096^2.
#pragma once
#include "dxb_decode.cuh"

#define DXB_AN_TILES 256u            // tiles per chunk = threads per CTA of the analysis kernels

#if defined(__CUDACC__)
#define DXB_HD __host__ __device__ inline
#else
#define DXB_HD static inline
#endif

// CMSE_FLAGS (DirectXTex.h:1022-1038)
enum
{
    DXB_CMSE_IMAGE1_SRGB = 0x1, DXB_CMSE_IMAGE2_SRGB = 0x2,
    DXB_CMSE_IGNORE_RED = 0x10, DXB_CMSE_IGNORE_GREEN = 0x20, DXB_CMSE_IGNORE_BLUE = 0x40, DXB_CMSE_IGNORE_ALPHA = 0x80,
    DXB_CMSE_IMAGE1_X2_BIAS = 0x100, DXB_CMSE_IMAGE2_X2_BIAS = 0x200,
    DXB_CMSE_MASK = 0x3F3,
};

// flags implied by the format of the image that is compared (:46-91); a BC image is compared as its R32G32B32A32_FLOAT
// decompression, which implies nothing (so BC*_SRGB data gets no gamma, as in the reference).  second = image2's bits.
DXB_HD uint32_t dxb_cmse_implied(uint32_t fmt, bool second)
{
    const uint32_t srgb = second ? (uint32_t)DXB_CMSE_IMAGE2_SRGB : (uint32_t)DXB_CMSE_IMAGE1_SRGB;
    switch (fmt)
    {
    case DXB_FMT_B8G8R8X8_UNORM: return DXB_CMSE_IGNORE_ALPHA;
    case DXB_FMT_B8G8R8X8_UNORM_SRGB: return srgb | DXB_CMSE_IGNORE_ALPHA;
    case DXB_FMT_R8G8B8A8_UNORM_SRGB: case DXB_FMT_B8G8R8A8_UNORM_SRGB: return srgb;
    default: return 0u;
    }
}
// the same comparison with the images swapped: the IMAGE1 and IMAGE2 bits trade places (d*d does not change sign)
DXB_HD uint32_t dxb_cmse_swap(uint32_t f)
{
    return (f & ~(uint32_t)(DXB_CMSE_IMAGE1_SRGB | DXB_CMSE_IMAGE2_SRGB | DXB_CMSE_IMAGE1_X2_BIAS | DXB_CMSE_IMAGE2_X2_BIAS))
         | ((f & DXB_CMSE_IMAGE1_SRGB) << 1) | ((f & DXB_CMSE_IMAGE2_SRGB) >> 1) | ((f & DXB_CMSE_IMAGE1_X2_BIAS) << 1) | ((f & DXB_CMSE_IMAGE2_X2_BIAS) >> 1);
}

// ---- the 16 pixels of one tile of a BC image: decode, then the conversion step of Decompress(..., R32G32B32A32_FLOAT)
// (DecompressBC, DirectXTexCompress.cpp:488-528 with ConvertScanline(..., TEX_FILTER_DEFAULT) :500: sRGB data is linearised)
DXB_DEV void dxb_an_bc_tile(uint32_t fmt, const uint8_t* src, dxb_px* px)
{
#if DXB_ON_DEVICE
    __align__(16) uint8_t blk[16];
    if (dxb_bc_block_bytes(fmt) == 8u) *reinterpret_cast<uint2*>(blk) = *reinterpret_cast<const uint2*>(src);
    else *reinterpret_cast<uint4*>(blk) = *reinterpret_cast<const uint4*>(src);
#else
    alignas(16) uint8_t blk[16];
    memcpy(blk, src, dxb_bc_block_bytes(fmt));
#endif
    dxb_decode_block(fmt, blk, px);
    const uint32_t inF = dxb_convert_flags(fmt), outF = dxb_convert_flags(DXB_FMT_R32G32B32A32_FLOAT);
    const uint32_t cflags = dxb_resolve_srgb_convert(0u, fmt, DXB_FMT_R32G32B32A32_FLOAT);
    for (int i = 0; i < 16; ++i) px[i] = dxb_convert_pixel(px[i], inF, outF, cflags);
}

// ---- ComputeMSE_ per pixel (:112-153): the fp32 square of each channel
// powf out of line: its inlined copies (six per pixel) spill registers in the tile loop
#if DXB_ON_DEVICE
static __device__ __noinline__ float dxb_pow22(float v) { return powf(v, 2.2f); }
#else
static inline float dxb_pow22(float v) { return powf(v, 2.2f); }
#endif
DXB_DEV dxb_px dxb_cmse_prep(dxb_px v, bool srgb, bool bias)
{
    if (srgb) { v.x = dxb_pow22(v.x); v.y = dxb_pow22(v.y); v.z = dxb_pow22(v.z); }    // XMVectorPow(v, g_Gamma22); pow(w, 1) = w
    if (bias) { v.x = dxb_madd(v.x, 2.0f, -1.0f); v.y = dxb_madd(v.y, 2.0f, -1.0f); v.z = dxb_madd(v.z, 2.0f, -1.0f); v.w = dxb_madd(v.w, 2.0f, -1.0f); }
    return v;
}
DXB_DEV dxb_px dxb_cmse_square(dxb_px v1, dxb_px v2, uint32_t flags)
{
    v1 = dxb_cmse_prep(v1, (flags & DXB_CMSE_IMAGE1_SRGB) != 0u, (flags & DXB_CMSE_IMAGE1_X2_BIAS) != 0u);
    v2 = dxb_cmse_prep(v2, (flags & DXB_CMSE_IMAGE2_SRGB) != 0u, (flags & DXB_CMSE_IMAGE2_X2_BIAS) != 0u);
    dxb_px d = dxb_make_px(v1.x - v2.x, v1.y - v2.y, v1.z - v2.z, v1.w - v2.w);
    if (flags & DXB_CMSE_IGNORE_RED) d.x = 0.0f;
    if (flags & DXB_CMSE_IGNORE_GREEN) d.y = 0.0f;
    if (flags & DXB_CMSE_IGNORE_BLUE) d.z = 0.0f;
    if (flags & DXB_CMSE_IGNORE_ALPHA) d.w = 0.0f;
    return dxb_make_px(d.x * d.x, d.y * d.y, d.z * d.z, d.w * d.w);
}

struct dxb_sum4 { double x, y, z, w; };

// tile (bx, by): fp64 sums of the squares of its in-image pixels in row order.  BCA / BCB: the side is BC data (a / b point at
// the block rows); otherwise pixel rows.  A BC side is only ever side a when the other one is not BC (the host swaps the pair).
template <bool BCA, bool BCB>
DXB_DEV dxb_sum4 dxb_cmse_tile(const uint8_t* a, size_t pitchA, uint32_t fmtA, const uint8_t* b, size_t pitchB, uint32_t fmtB,
                               uint32_t width, uint32_t height, uint32_t bx, uint32_t by, uint32_t flags)
{
    dxb_sum4 s = { 0.0, 0.0, 0.0, 0.0 };
    const uint32_t x0 = bx * 4u, y0 = by * 4u;
    const uint32_t pw = (width - x0 < 4u) ? (width - x0) : 4u, ph = (height - y0 < 4u) ? (height - y0) : 4u;
    dxb_px pa[BCA ? 16 : 1], pb[BCB ? 16 : 1];
    if (BCA) dxb_an_bc_tile(fmtA, a + (size_t)by * pitchA + (size_t)bx * dxb_bc_block_bytes(fmtA), pa);
    if (BCB) dxb_an_bc_tile(fmtB, b + (size_t)by * pitchB + (size_t)bx * dxb_bc_block_bytes(fmtB), pb);
    #pragma unroll
    for (uint32_t t = 0; t < 4u; ++t)
    {
        if (t >= ph) break;
        const uint8_t* ra = BCA ? nullptr : a + (size_t)(y0 + t) * pitchA;
        const uint8_t* rb = BCB ? nullptr : b + (size_t)(y0 + t) * pitchB;
        #pragma unroll
        for (uint32_t s2 = 0; s2 < 4u; ++s2)
        {
            if (s2 >= pw) break;
            const dxb_px v1 = BCA ? pa[BCA ? (t * 4u + s2) : 0u] : dxb_load_pixel(fmtA, ra, x0 + s2);
            const dxb_px v2 = BCB ? pb[BCB ? (t * 4u + s2) : 0u] : dxb_load_pixel(fmtB, rb, x0 + s2);
            const dxb_px q = dxb_cmse_square(v1, v2, flags);
            s.x += (double)q.x; s.y += (double)q.y; s.z += (double)q.z; s.w += (double)q.w;
        }
    }
    return s;
}

// ---- the halving tree over DXB_AN_TILES slots (chunk level and image level); the kernels run the same steps in shared memory
DXB_HD void dxb_an_tree(double* v)        // v[DXB_AN_TILES] -> v[0]
{
    for (uint32_t s = DXB_AN_TILES / 2u; s >= 1u; s >>= 1)
        for (uint32_t t = 0; t < s; ++t) v[t] = v[t] + v[t + s];
}
// image level from the chunk partials (4 doubles per chunk, chunk order): out = { mse, mseV[0..3] }
DXB_HD void dxb_cmse_finish(const double* partials, uint32_t nchunks, uint64_t pixels, float* out)
{
    const float n = (float)pixels;
    float v[4];
    for (int c = 0; c < 4; ++c)
    {
        double lane[DXB_AN_TILES];
        for (uint32_t t = 0; t < DXB_AN_TILES; ++t)
        {
            double acc = 0.0;
            for (uint32_t k = t; k < nchunks; k += DXB_AN_TILES) acc = acc + partials[4u * k + (uint32_t)c];
            lane[t] = acc;
        }
        dxb_an_tree(lane);
        v[c] = (float)lane[0] / n;
    }
    out[0] = ((v[0] + v[1]) + v[2]) + v[3];
    out[1] = v[0]; out[2] = v[1]; out[3] = v[2]; out[4] = v[3];
}

// ---- IsAlphaAllOpaque on one tile: false when an in-image pixel is below the threshold.  Uncompressed: alpha < 0.997 after
// LoadScanline (DirectXTexImage.cpp:822-846).  BC1/2/3/7: alpha < 0.99 after the block decoder (DirectXTexCompress.cpp:578-611);
// BC4/5/6H are answered per image on the host (:569-572).  A NaN alpha compares false, as XMVector4Less does.
template <bool BC>
DXB_DEV bool dxb_opaque_tile(const uint8_t* img, size_t pitch, uint32_t fmt, uint32_t width, uint32_t height, uint32_t bx, uint32_t by)
{
    const uint32_t x0 = bx * 4u, y0 = by * 4u;
    const uint32_t pw = (width - x0 < 4u) ? (width - x0) : 4u, ph = (height - y0 < 4u) ? (height - y0) : 4u;
    bool ok = true;
    if (BC)
    {
        dxb_px px[16];
#if DXB_ON_DEVICE
        __align__(16) uint8_t blk[16];
        const uint8_t* src = img + (size_t)by * pitch + (size_t)bx * dxb_bc_block_bytes(fmt);
        if (dxb_bc_block_bytes(fmt) == 8u) *reinterpret_cast<uint2*>(blk) = *reinterpret_cast<const uint2*>(src);
        else *reinterpret_cast<uint4*>(blk) = *reinterpret_cast<const uint4*>(src);
#else
        alignas(16) uint8_t blk[16];
        memcpy(blk, img + (size_t)by * pitch + (size_t)bx * dxb_bc_block_bytes(fmt), dxb_bc_block_bytes(fmt));
#endif
        dxb_decode_block(fmt, blk, px);
        #pragma unroll
        for (uint32_t t = 0; t < 4u; ++t)
            #pragma unroll
            for (uint32_t s2 = 0; s2 < 4u; ++s2)
                if (t < ph && s2 < pw && px[t * 4u + s2].w < 0.99f) ok = false;
        return ok;
    }
    for (uint32_t t = 0; t < ph; ++t)
    {
        const uint8_t* row = img + (size_t)(y0 + t) * pitch;
        for (uint32_t s2 = 0; s2 < pw; ++s2)
            if (dxb_load_pixel(fmt, row, x0 + s2).w < 0.997f) ok = false;
    }
    return ok;
}
// the formats whose BC scan runs (IsAlphaAllOpaqueBC's decoder switch after the TYPELESS promotion)
DXB_HD bool dxb_opaque_bc_scanned(uint32_t fmt)
{
    return fmt == DXB_FMT_BC1_UNORM || fmt == DXB_FMT_BC1_UNORM_SRGB || fmt == DXB_FMT_BC2_UNORM || fmt == DXB_FMT_BC2_UNORM_SRGB ||
           fmt == DXB_FMT_BC3_UNORM || fmt == DXB_FMT_BC3_UNORM_SRGB || fmt == DXB_FMT_BC7_UNORM || fmt == DXB_FMT_BC7_UNORM_SRGB;
}
