// dxb_launch.h — job/parameter structs shared by the kernels' translation units and the host API, plus the
// host-callable launchers each kernel TU exports (hidden visibility; not part of the C ABI).
#pragma once
#include <stdint.h>
#include <stddef.h>
#include <cuda_runtime.h>
#include "dxb_mipjob.h"

struct dxb_job
{
    const uint8_t* src; uint8_t* dst;
    size_t srcPitch, dstPitch;
    uint32_t width, height;
    uint32_t nbx, nby;
    uint32_t firstUnit;
    uint32_t pad;
};

// one image pair (ComputeMSE: a vs b) or one image (IsAlphaAllOpaque: a) walked one thread per 4x4 tile; the work units are
// chunks of DXB_AN_TILES tiles of one tile row (dxb_analyze.cuh), cpr per tile row
struct dxb_pair_job
{
    const uint8_t* a; const uint8_t* b;
    size_t pitchA, pitchB;
    uint32_t width, height;
    uint32_t fmtA, fmtB;
    uint32_t flags;                // CMSE flags, the ones implied by the formats included
    uint32_t nbx, cpr;             // tiles per row, chunks per tile row
    uint32_t firstUnit;            // first chunk of this job in the launch
    uint32_t firstPartial;         // index of its first chunk partial (ComputeMSE)
    uint32_t pad;
};
// image level of ComputeMSE: chunks [firstPartial, firstPartial + nchunks) of the partials -> out[5 * index ..]
struct dxb_mse_final
{
    uint64_t pixels;
    uint32_t firstPartial, nchunks;
};

struct dxb_compress_params
{
    uint32_t srcFormat, dstFormat;
    uint32_t inF, outF, cflags, bcflags;
    float threshold;
    uint32_t totalUnits, njobs;
    // batches of equal mip chains (items x levels jobs, item-major): every item has periodJobs jobs covering periodUnits units, so a
    // unit's job is found from one division and a short forward scan instead of a 14-step binary search of dependent loads
    uint32_t periodUnits, periodJobs;     // 0 = no such structure
};

struct dxb_convert_params
{
    uint32_t srcFormat, dstFormat, inF, outF, flags;
    uint32_t totalUnits, njobs;
    float threshold;               // alpha threshold of 1-bit alpha destinations (B5G5R5A1)
};

struct dxb_mip_params
{
    uint32_t format, mode /*DXB_FILTER_* mode bits*/, filter, lflags;
    uint32_t totalUnits, njobs;
    dxb_tri_axis triX, triY;       // triangle filter only
};

#ifndef DXB_BC7_WARPS
#define DXB_BC7_WARPS 8       // warps per CTA of k_compress_bc7 (two blocks per warp, 8.6 KB dynamic shared per warp)
#endif
#ifndef DXB_BC7_MINB
#define DXB_BC7_MINB 3        // __launch_bounds__ min CTAs per SM of k_compress_bc7
#endif
#ifndef DXB_BC6H_WARPS
#define DXB_BC6H_WARPS 8      // warps per CTA of k_compress_bc6h (two blocks per warp)
#endif
#ifndef DXB_BC6H_MINB
#define DXB_BC6H_MINB 2
#endif

// launchers: `grid` CTAs on `stream`; jobs == nullptr -> `single` is used
void dxb_launch_bc15(unsigned grid, cudaStream_t stream, const dxb_job* jobs, const dxb_job& single, const dxb_compress_params& P);
void dxb_launch_bc7(unsigned grid, cudaStream_t stream, const dxb_job* jobs, const dxb_job& single, const dxb_compress_params& P);
// TMA-fed persistent variant (RGBA32F sources of full 4x4 blocks, equal images at a constant stride); false = not eligible, nothing launched
bool dxb_launch_bc7_tma(unsigned residentCtas, cudaStream_t stream, const dxb_job* hostJobs, const dxb_compress_params& P);
int dxb_bc7_get_feed();            // 0 direct kernel, 1-3 TMA-fed variants (dxb_k_bc7.cu)
void dxb_bc7_set_feed(int mode);
void dxb_launch_decompress(unsigned grid, cudaStream_t stream, const dxb_job* jobs, const dxb_job& single, const dxb_compress_params& P);
void dxb_launch_bc6h(unsigned grid, cudaStream_t stream, const dxb_job* jobs, const dxb_job& single, const dxb_compress_params& P);
// hostJobs = the same records on the host (njobs of them); jobs = device copy or nullptr when njobs == 1
void dxb_launch_convert(unsigned grid, cudaStream_t stream, const dxb_job* jobs, const dxb_job* hostJobs, const dxb_convert_params& P);
void dxb_launch_mip(unsigned grid, cudaStream_t stream, const dxb_mip_job* jobs, const dxb_mip_job* hostJobs, const dxb_mip_params& P);
// tail of a chain: levels [first, first+count) of all items in one launch (jobsDev laid out [level][item]); false = no such kernel
void dxb_launch_convert_diffuse(cudaStream_t stream, const dxb_job* jobs, const dxb_job* hostJobs, const dxb_convert_params& P, void* errors, uint32_t errStride);
void dxb_launch_alpha_coverage(unsigned grid, cudaStream_t stream, const dxb_job& j, uint32_t fmt, float scale, float ref, unsigned long long* count);
void dxb_launch_scale_alpha(unsigned grid, cudaStream_t stream, const dxb_job& j, uint32_t fmt, float scale);
void dxb_launch_pmalpha(unsigned grid, cudaStream_t stream, const dxb_job* jobs, const dxb_job* hostJobs, const dxb_convert_params& P);
bool dxb_launch_mip_box3(cudaStream_t stream, const dxb_mip_job* jobsDev, const dxb_mip_job* hostJobs, uint32_t items, const dxb_mip_params& P);
bool dxb_launch_mip_tail(cudaStream_t stream, const dxb_mip_job* jobsDev, uint32_t items, uint32_t count, const dxb_mip_params& P);
// ComputeMSE / IsAlphaAllOpaque (dxb_k_analyze.cu); every job of one launch has the same kind of sides (BC or not, BC on side a
// when only one is); partials = 4 doubles per chunk
void dxb_launch_compute_mse(unsigned grid, cudaStream_t stream, const dxb_pair_job* jobs, const dxb_pair_job& single, uint32_t njobs,
                            uint32_t totalUnits, double* partials);
void dxb_launch_mse_finish(cudaStream_t stream, const dxb_mse_final* jobs, uint32_t njobs, const double* partials, float* out);
void dxb_launch_alpha_opaque(unsigned grid, cudaStream_t stream, const dxb_pair_job* jobs, const dxb_pair_job& single, uint32_t njobs,
                             uint32_t totalUnits, int32_t* opaque);
void dxb_launch_set_i32(cudaStream_t stream, int32_t* p, int32_t value);
// resident CTAs per SM of each kernel at its block size
int dxb_occupancy_bc15();
int dxb_occupancy_bc7();
int dxb_occupancy_bc6h();

#ifdef __CUDACC__
template <typename J>
__device__ __forceinline__ const J& dxb_find_job(const J* jobs, uint32_t njobs, const J& single, uint32_t unit, uint32_t periodUnits = 0, uint32_t periodJobs = 0)
{
    if (jobs == nullptr) return single;
    if (periodUnits != 0u)
    {
        const uint32_t item = unit / periodUnits;
        uint32_t k = item * periodJobs;
        const uint32_t end = k + periodJobs - 1u;
        while (k < end && jobs[k + 1u].firstUnit <= unit) ++k;
        return jobs[k];
    }
    uint32_t lo = 0, hi = njobs;            // last job with firstUnit <= unit
    while (hi - lo > 1)
    {
        const uint32_t mid = (lo + hi) >> 1;
        if (jobs[mid].firstUnit <= unit) lo = mid; else hi = mid;
    }
    return jobs[lo];
}
#endif
