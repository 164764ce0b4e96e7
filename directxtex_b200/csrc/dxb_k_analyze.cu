// dxb_k_analyze.cu — whole-image reductions, one THREAD per 4x4 tile, one CTA per chunk of DXB_AN_TILES tiles of a tile row
// (dxb_analyze.cuh has the per-pixel arithmetic and the reduction tree):
//   k_compute_mse<BCA, BCB>   ComputeMSE: fp64 partial sums of one chunk, BC sides decoded in the kernel
//   k_mse_finish              image level of the tree: one CTA per pair -> { mse, mseV[4] }
//   k_alpha_opaque<BC>        IsAlphaAllOpaque scan; a device flag ends the scan early once a pixel is found
#include "dxb_launch.h"
#include "dxb_analyze.cuh"

// chunk `unit` of the launch -> its job and the tile this thread handles (false: past the end of the tile row)
__device__ __forceinline__ bool an_tile(const dxb_pair_job& j, uint32_t unit, uint32_t* bx, uint32_t* by)
{
    const uint32_t local = unit - j.firstUnit;
    *by = local / j.cpr;
    *bx = (local - *by * j.cpr) * DXB_AN_TILES + threadIdx.x;
    return *bx < j.nbx;
}

template <bool BCA, bool BCB>
__global__ void __launch_bounds__(DXB_AN_TILES) k_compute_mse(const dxb_pair_job* __restrict__ jobs, dxb_pair_job single, uint32_t njobs,
                                                              uint32_t totalUnits, double* __restrict__ partials)
{
    __shared__ double sm[4][DXB_AN_TILES];
    const uint32_t t = threadIdx.x;
    for (uint32_t unit = blockIdx.x; unit < totalUnits; unit += gridDim.x)
    {
        const dxb_pair_job& j = dxb_find_job(jobs, njobs, single, unit);
        uint32_t bx, by;
        dxb_sum4 s = { 0.0, 0.0, 0.0, 0.0 };
        if (an_tile(j, unit, &bx, &by))
            s = dxb_cmse_tile<BCA, BCB>(j.a, j.pitchA, j.fmtA, j.b, j.pitchB, j.fmtB, j.width, j.height, bx, by, j.flags);
        sm[0][t] = s.x; sm[1][t] = s.y; sm[2][t] = s.z; sm[3][t] = s.w;
        __syncthreads();
        #pragma unroll
        for (uint32_t h = DXB_AN_TILES / 2u; h >= 1u; h >>= 1)        // dxb_an_tree
        {
            if (t < h) { sm[0][t] = sm[0][t] + sm[0][t + h]; sm[1][t] = sm[1][t] + sm[1][t + h]; sm[2][t] = sm[2][t] + sm[2][t + h]; sm[3][t] = sm[3][t] + sm[3][t + h]; }
            __syncthreads();
        }
        if (t < 4u) partials[4u * (j.firstPartial + (unit - j.firstUnit)) + t] = sm[t][0];
        __syncthreads();
    }
}

__global__ void __launch_bounds__(DXB_AN_TILES) k_mse_finish(const dxb_mse_final* __restrict__ jobs, const double* __restrict__ partials, float* __restrict__ out)
{
    __shared__ double sm[4][DXB_AN_TILES];
    const dxb_mse_final j = jobs[blockIdx.x];
    const uint32_t t = threadIdx.x;
    double acc[4] = { 0.0, 0.0, 0.0, 0.0 };
    for (uint32_t k = t; k < j.nchunks; k += DXB_AN_TILES)
        #pragma unroll
        for (int c = 0; c < 4; ++c) acc[c] = acc[c] + partials[4u * (j.firstPartial + k) + (uint32_t)c];
    #pragma unroll
    for (int c = 0; c < 4; ++c) sm[c][t] = acc[c];
    __syncthreads();
    #pragma unroll
    for (uint32_t h = DXB_AN_TILES / 2u; h >= 1u; h >>= 1)
    {
        if (t < h) for (int c = 0; c < 4; ++c) sm[c][t] = sm[c][t] + sm[c][t + h];
        __syncthreads();
    }
    if (t == 0)
    {
        const float n = (float)j.pixels;
        const float v0 = (float)sm[0][0] / n, v1 = (float)sm[1][0] / n, v2 = (float)sm[2][0] / n, v3 = (float)sm[3][0] / n;
        float* o = out + 5u * blockIdx.x;
        o[0] = ((v0 + v1) + v2) + v3;
        o[1] = v0; o[2] = v1; o[3] = v2; o[4] = v3;
    }
}

template <bool BC>
__global__ void __launch_bounds__(DXB_AN_TILES) k_alpha_opaque(const dxb_pair_job* __restrict__ jobs, dxb_pair_job single, uint32_t njobs,
                                                               uint32_t totalUnits, int32_t* opaque)
{
    for (uint32_t unit = blockIdx.x; unit < totalUnits; unit += gridDim.x)
    {
        if (*reinterpret_cast<volatile int32_t*>(opaque) == 0) return;           // an earlier chunk found a pixel
        const dxb_pair_job& j = dxb_find_job(jobs, njobs, single, unit);
        uint32_t bx, by;
        if (an_tile(j, unit, &bx, &by) && !dxb_opaque_tile<BC>(j.a, j.pitchA, j.fmtA, j.width, j.height, bx, by)) *opaque = 0;
    }
}

__global__ void k_set_i32(int32_t* p, int32_t v) { *p = v; }

void dxb_launch_compute_mse(unsigned grid, cudaStream_t stream, const dxb_pair_job* jobs, const dxb_pair_job& single, uint32_t njobs,
                            uint32_t totalUnits, double* partials)
{
    const bool bcA = dxb_bc_block_bytes(single.fmtA) != 0u, bcB = dxb_bc_block_bytes(single.fmtB) != 0u;
    if (bcA && bcB) k_compute_mse<true, true><<<grid, DXB_AN_TILES, 0, stream>>>(jobs, single, njobs, totalUnits, partials);
    else if (bcA) k_compute_mse<true, false><<<grid, DXB_AN_TILES, 0, stream>>>(jobs, single, njobs, totalUnits, partials);
    else k_compute_mse<false, false><<<grid, DXB_AN_TILES, 0, stream>>>(jobs, single, njobs, totalUnits, partials);
}

void dxb_launch_mse_finish(cudaStream_t stream, const dxb_mse_final* jobs, uint32_t njobs, const double* partials, float* out)
{
    k_mse_finish<<<njobs, DXB_AN_TILES, 0, stream>>>(jobs, partials, out);
}

void dxb_launch_alpha_opaque(unsigned grid, cudaStream_t stream, const dxb_pair_job* jobs, const dxb_pair_job& single, uint32_t njobs,
                             uint32_t totalUnits, int32_t* opaque)
{
    if (dxb_bc_block_bytes(single.fmtA) != 0u) k_alpha_opaque<true><<<grid, DXB_AN_TILES, 0, stream>>>(jobs, single, njobs, totalUnits, opaque);
    else k_alpha_opaque<false><<<grid, DXB_AN_TILES, 0, stream>>>(jobs, single, njobs, totalUnits, opaque);
}

void dxb_launch_set_i32(cudaStream_t stream, int32_t* p, int32_t value)
{
    k_set_i32<<<1, 1, 0, stream>>>(p, value);
}
