// tests/emul/analysis_emul.cpp — TEST INFRASTRUCTURE, never shipped.
//
// Host build of ComputeMSE and the IsAlphaAllOpaque scan from the headers the kernels are compiled from (dxb_analyze.cuh: the
// same tile arithmetic and the same fp64 reduction tree as dxb_k_analyze.cu), so that the arithmetic can be rehearsed without a
// GPU and the GPU results compared with it.  Built with the flags of tests/emul/build.sh by tests/analysis_lib.py.
#include <cstdint>
#include <cstddef>
#include <cstring>
#include <cmath>
#include <vector>
#include <algorithm>
#include <utility>

#include "dxb_portable.h"
#include "dxb_formats.h"
#include "dxb_pixel.cuh"

// ---- ComputeMSE / IsAlphaAllOpaque emulation: the same tile arithmetic and the same fp64 tree as dxb_k_analyze.cu ----------------
#include "dxb_analyze.cuh"
extern "C" int32_t emul_compute_mse(const uint8_t* a, uint32_t fmtA, size_t pitchA, const uint8_t* b, uint32_t fmtB, size_t pitchB,
                                    size_t w, size_t h, uint32_t flags, float* out5)
{
    bool bcA = dxb_bc_block_bytes(fmtA) != 0, bcB = dxb_bc_block_bytes(fmtB) != 0;
    if ((!bcA && !dxb_bytes_per_pixel(fmtA)) || (!bcB && !dxb_bytes_per_pixel(fmtB))) return DXB_E_NOT_SUPPORTED;
    if (!pitchA) pitchA = bcA ? ((w + 3) / 4) * dxb_bc_block_bytes(fmtA) : w * dxb_bytes_per_pixel(fmtA);
    if (!pitchB) pitchB = bcB ? ((w + 3) / 4) * dxb_bc_block_bytes(fmtB) : w * dxb_bytes_per_pixel(fmtB);
    uint32_t f = (flags & DXB_CMSE_MASK) | dxb_cmse_implied(fmtA, false) | dxb_cmse_implied(fmtB, true);
    if (!bcA && bcB) { std::swap(a, b); std::swap(fmtA, fmtB); std::swap(pitchA, pitchB); std::swap(bcA, bcB); f = dxb_cmse_swap(f); }
    const uint32_t nbx = (uint32_t)((w + 3) / 4), nby = (uint32_t)((h + 3) / 4), cpr = (nbx + DXB_AN_TILES - 1) / DXB_AN_TILES;
    std::vector<double> partials((size_t)nby * cpr * 4);
    #pragma omp parallel for schedule(dynamic, 4)
    for (long c = 0; c < (long)nby * cpr; ++c)
    {
        const uint32_t by = (uint32_t)(c / cpr), bx0 = (uint32_t)(c % cpr) * DXB_AN_TILES;
        std::vector<double> lane(4 * DXB_AN_TILES, 0.0);
        for (uint32_t t = 0; t < DXB_AN_TILES && bx0 + t < nbx; ++t)
        {
            dxb_sum4 s;
            if (bcA && bcB) s = dxb_cmse_tile<true, true>(a, pitchA, fmtA, b, pitchB, fmtB, (uint32_t)w, (uint32_t)h, bx0 + t, by, f);
            else if (bcA) s = dxb_cmse_tile<true, false>(a, pitchA, fmtA, b, pitchB, fmtB, (uint32_t)w, (uint32_t)h, bx0 + t, by, f);
            else s = dxb_cmse_tile<false, false>(a, pitchA, fmtA, b, pitchB, fmtB, (uint32_t)w, (uint32_t)h, bx0 + t, by, f);
            lane[t] = s.x; lane[DXB_AN_TILES + t] = s.y; lane[2 * DXB_AN_TILES + t] = s.z; lane[3 * DXB_AN_TILES + t] = s.w;
        }
        for (int k = 0; k < 4; ++k) { dxb_an_tree(lane.data() + k * DXB_AN_TILES); partials[4 * c + k] = lane[k * DXB_AN_TILES]; }
    }
    dxb_cmse_finish(partials.data(), nby * cpr, (uint64_t)w * h, out5);
    return DXB_S_OK;
}

// the scan over the images of one texture held at base + offsets[i]
extern "C" int32_t emul_is_alpha_all_opaque(const uint8_t* base, const size_t* offsets, const size_t* widths, const size_t* heights,
                                            const size_t* pitches, size_t n, uint32_t fmt, int32_t* opaque)
{
    const bool bc = dxb_bc_block_bytes(fmt) != 0;
    if (!bc && !dxb_bytes_per_pixel(fmt)) return DXB_E_NOT_SUPPORTED;
    *opaque = 1;
    if (bc && !dxb_opaque_bc_scanned(fmt)) { *opaque = 0; return DXB_S_OK; }
    for (size_t i = 0; i < n; ++i)
        for (uint32_t by = 0; by < (heights[i] + 3) / 4; ++by)
            for (uint32_t bx = 0; bx < (widths[i] + 3) / 4; ++bx)
            {
                const bool ok = bc ? dxb_opaque_tile<true>(base + offsets[i], pitches[i], fmt, (uint32_t)widths[i], (uint32_t)heights[i], bx, by)
                                   : dxb_opaque_tile<false>(base + offsets[i], pitches[i], fmt, (uint32_t)widths[i], (uint32_t)heights[i], bx, by);
                if (!ok) { *opaque = 0; return DXB_S_OK; }
            }
    return DXB_S_OK;
}
