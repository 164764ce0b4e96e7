// dxb_api.cu — the extern "C" boundary of libdxtex_b200.so (see include/dxtex_b200.h) and the host
// logic behind it: argument validation with the reference's HRESULTs, pitch rules, batching,
// staging of host images through device memory, kernel launches on sm_100a.
//
// Compiled with: nvcc -gencode arch=compute_100a,code=sm_100a -fmad=false (bit-exact fp32 contract
// of the BC1-5 / convert / mip kernels) -lineinfo.  There is no host implementation of any codec in
// this file: if CUDA is unavailable every compute entry point returns E_FAIL.
#include <cuda_runtime.h>
#include <atomic>
#include <mutex>
#include <condition_variable>
#include <memory>
#include <thread>
#include <unistd.h>
#include <sys/syscall.h>
#include <vector>
#include <string>
#include <cstring>
#include <cstdio>
#include <cmath>
#include <algorithm>

#include "../../include/dxtex_b200.h"
#include "dxb_formats.h"
#include "dxb_launch.h"
#include "dxb_host_tri.h"

namespace {

constexpr int NSLOT = 3;        // (stream, device buffer pair) slots of one lane: H2D / kernel / D2H of consecutive chunks overlap
constexpr int NLANE = 2;        // host-staged calls that can be in flight on one device at the same time (each owns a lane)

std::mutex g_mu;                // guards the device table only; calls on different lanes / devices run concurrently
std::atomic<uint64_t> g_launches{0}, g_tma_launches{0};
thread_local std::string t_lastError;

struct Lane
{
    cudaStream_t streams[NSLOT] = { nullptr, nullptr, nullptr };
    void* dIn[NSLOT] = { nullptr, nullptr, nullptr };  size_t dInCap[NSLOT] = { 0, 0, 0 };
    void* dOut[NSLOT] = { nullptr, nullptr, nullptr }; size_t dOutCap[NSLOT] = { 0, 0, 0 };
    bool busy = false;
};

// one per CUDA device the library was initialised on (dxb200_init / dxb200_init_devices; SURVEY.md 8(b), 8(e))
struct Device
{
    int ordinal = 0;
    int numSMs = 148;
    int numaNode = -1;
    int gridBC15 = 0, gridBC7 = 0, gridBC6H = 0, gridRow = 0;
    std::mutex mu; std::condition_variable cv;
    Lane lanes[NLANE];
};
std::vector<std::unique_ptr<Device>> g_devs;

// the device (and, for host-staged calls, the lane) the calling thread is working on
struct View { Device* dev = nullptr; Lane* lane = nullptr; };
thread_local View t_v;

int32_t cuda_hr(cudaError_t e, const char* what)
{
    if (e == cudaSuccess) return DXB_S_OK;
    char buf[256];
    snprintf(buf, sizeof(buf), "%s: %s", what, cudaGetErrorString(e));
    t_lastError = buf;
    (void)cudaGetLastError();
    return (e == cudaErrorMemoryAllocation) ? DXB_E_OUTOFMEMORY : DXB_E_FAIL;
}
#define DXB_CUDA(call) do { const int32_t hr__ = cuda_hr((call), #call); if (hr__ != DXB_S_OK) return hr__; } while (0)

// NUMA node of a device's PCI function (sysfs), -1 if unknown
int device_numa_node(int ordinal)
{
    char bus[32] = { 0 };
    if (cudaDeviceGetPCIBusId(bus, sizeof(bus), ordinal) != cudaSuccess) { (void)cudaGetLastError(); return -1; }
    for (char* c = bus; *c; ++c) *c = (char)tolower(*c);
    char path[96];
    snprintf(path, sizeof(path), "/sys/bus/pci/devices/%s/numa_node", bus);
    FILE* f = fopen(path, "r");
    if (!f) return -1;
    int node = -1;
    if (fscanf(f, "%d", &node) != 1) node = -1;
    fclose(f);
    return node;
}

// find or create the Device record of CUDA device `ordinal`; g_mu held.  Leaves `ordinal` current.
int32_t init_device_locked(int ordinal, Device** out)
{
    for (auto& d : g_devs) if (d->ordinal == ordinal) { if (out) *out = d.get(); return DXB_S_OK; }
    int n = 0;
    DXB_CUDA(cudaGetDeviceCount(&n));
    if (n <= 0) { t_lastError = "no CUDA device"; return DXB_E_FAIL; }
    if (ordinal < 0 || ordinal >= n) { t_lastError = "device ordinal out of range"; return DXB_E_INVALIDARG; }
    DXB_CUDA(cudaSetDevice(ordinal));
    std::unique_ptr<Device> d(new Device);
    d->ordinal = ordinal;
    cudaDeviceProp prop;
    DXB_CUDA(cudaGetDeviceProperties(&prop, ordinal));
    d->numSMs = prop.multiProcessorCount;
    d->numaNode = device_numa_node(ordinal);
    for (int l = 0; l < NLANE; ++l)
        for (int i = 0; i < NSLOT; ++i) DXB_CUDA(cudaStreamCreateWithFlags(&d->lanes[l].streams[i], cudaStreamNonBlocking));
    {
        // job arrays use stream-ordered allocation: keep freed blocks in the pool across synchronisation points
        // (the default release threshold of 0 returns them to the OS, which makes the next call's cudaMallocAsync slow)
        cudaMemPool_t pool;
        if (cudaDeviceGetDefaultMemPool(&pool, ordinal) == cudaSuccess)
        {
            uint64_t keep = ~uint64_t(0);
            (void)cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
        }
        (void)cudaGetLastError();
    }
    d->gridBC15 = d->numSMs * dxb_occupancy_bc15();
    d->gridBC7 = d->numSMs * dxb_occupancy_bc7();
    d->gridBC6H = d->numSMs * dxb_occupancy_bc6h();
    d->gridRow = d->numSMs * 8;
    if (out) *out = d.get();
    g_devs.push_back(std::move(d));
    return DXB_S_OK;
}

// the devices host-pointer calls are sharded over; a process that never called dxb200_init* gets its current CUDA device
int32_t device_list(std::vector<Device*>* out)
{
    std::lock_guard<std::mutex> lk(g_mu);
    if (g_devs.empty())
    {
        int cur = 0;
        if (cudaGetDevice(&cur) != cudaSuccess) { (void)cudaGetLastError(); cur = 0; }
        const int32_t hr = init_device_locked(cur, nullptr);
        if (hr != DXB_S_OK) return hr;
    }
    out->clear();
    for (auto& d : g_devs) out->push_back(d.get());
    return DXB_S_OK;
}

// host-pointer call on device `d`: waits for one of its lanes, makes device and lane current for the calling thread
struct HostScope
{
    Device* d = nullptr; Lane* l = nullptr; int prev = -1; View saved;
    int32_t enter(Device* dev)
    {
        saved = t_v;
        if (cudaGetDevice(&prev) != cudaSuccess) { (void)cudaGetLastError(); prev = -1; }
        DXB_CUDA(cudaSetDevice(dev->ordinal));
        std::unique_lock<std::mutex> lk(dev->mu);
        for (;;)
        {
            for (int i = 0; i < NLANE && !l; ++i) if (!dev->lanes[i].busy) l = &dev->lanes[i];
            if (l) break;
            dev->cv.wait(lk);
        }
        l->busy = true; d = dev;
        t_v.dev = dev; t_v.lane = l;
        return DXB_S_OK;
    }
    ~HostScope()
    {
        if (l) { { std::lock_guard<std::mutex> lk(d->mu); l->busy = false; } d->cv.notify_one(); }
        t_v = saved;
        if (prev >= 0 && d && prev != d->ordinal) (void)cudaSetDevice(prev);
    }
};

// _device call: the work goes to the device that owns the caller's pointers, on the caller's stream
struct DevScope
{
    int prev = -1, ord = -1; View saved;
    int32_t enter(const void* p)
    {
        saved = t_v;
        if (cudaGetDevice(&prev) != cudaSuccess) { (void)cudaGetLastError(); prev = 0; }
        ord = prev;
        cudaPointerAttributes a;
        if (p && cudaPointerGetAttributes(&a, p) == cudaSuccess && (a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged)) ord = a.device;
        (void)cudaGetLastError();
        Device* dev = nullptr;
        {
            std::lock_guard<std::mutex> lk(g_mu);
            const int32_t hr = init_device_locked(ord, &dev);           // leaves `ord` current when it creates the record
            if (hr != DXB_S_OK) return hr;
        }
        DXB_CUDA(cudaSetDevice(ord));
        t_v.dev = dev; t_v.lane = nullptr;
        return DXB_S_OK;
    }
    ~DevScope()
    {
        t_v = saved;
        if (prev >= 0 && ord >= 0 && prev != ord) (void)cudaSetDevice(prev);
    }
};

// Runs fn(lo, hi) over [0, n) split into contiguous ranges of about equal weight, one range per initialised device, each on
// its own host thread (the caller's thread takes the first range).  One device or one unit: runs inline.
template <typename WeightFn, typename Fn>
int32_t run_sharded(size_t n, WeightFn weight, Fn fn)
{
    std::vector<Device*> devs;
    int32_t hr = device_list(&devs);
    if (hr != DXB_S_OK) return hr;
    const size_t nd = std::min(devs.size(), std::max<size_t>(n, 1));
    if (nd <= 1)
    {
        HostScope sc;
        hr = sc.enter(devs[0]);
        return hr != DXB_S_OK ? hr : fn(size_t(0), n);
    }
    double total = 0;
    for (size_t i = 0; i < n; ++i) total += (double)weight(i);
    std::vector<size_t> cut(nd + 1, n);
    cut[0] = 0;
    {
        double acc = 0; size_t d = 1;
        for (size_t i = 0; i < n && d < nd; ++i)
        {
            acc += (double)weight(i);
            while (d < nd && acc >= total * (double)d / (double)nd) cut[d++] = i + 1;
        }
    }
    std::vector<int32_t> hrs(nd, DXB_S_OK);
    std::vector<std::string> errs(nd);
    auto work = [&](size_t d)
    {
        if (cut[d] == cut[d + 1]) return;
        HostScope sc;
        hrs[d] = sc.enter(devs[d]);
        if (hrs[d] == DXB_S_OK) hrs[d] = fn(cut[d], cut[d + 1]);
        if (hrs[d] != DXB_S_OK) errs[d] = t_lastError;
    };
    std::vector<std::thread> th;
    for (size_t d = 1; d < nd; ++d) th.emplace_back(work, d);
    work(0);
    for (auto& t : th) t.join();
    for (size_t d = 0; d < nd; ++d) if (hrs[d] != DXB_S_OK) { t_lastError = errs[d]; return hrs[d]; }
    return DXB_S_OK;
}

// progress reporting / cancellation of the host-staged calls (the reference's statusCallback, DirectXTexCompress.cpp:115-121, 785-837)
struct Progress
{
    dxb200_status_fn fn = nullptr; void* user = nullptr;
    size_t total = 0; std::atomic<size_t> done{0}; std::atomic<bool> aborted{false};
    std::mutex mu;
    // false = the caller asked to stop
    bool report(size_t add)
    {
        if (!fn) return true;
        if (aborted.load()) return false;
        const size_t d = done.fetch_add(add);                      // units finished before this chunk, as the reference reports (:115-121)
        std::lock_guard<std::mutex> lk(mu);
        if (!fn(std::min(d, total), total, user)) aborted.store(true);
        return !aborted.load();
    }
};

int32_t ensure_buffer(void** p, size_t* cap, size_t need)
{
    if (*cap >= need) return DXB_S_OK;
    if (*p) { cudaFree(*p); *p = nullptr; *cap = 0; }
    const size_t want = (need + (size_t(1) << 20)) & ~((size_t(1) << 20) - 1);
    DXB_CUDA(cudaMalloc(p, want));
    *cap = want;
    return DXB_S_OK;
}

// ---- format predicates (DirectXTex.inl:57-130 / DirectXTexUtil.cpp), implemented subset ----------
bool is_compressed(uint32_t f) { return dxb_bc_block_bytes(f) != 0; }
bool is_supported_pixel_format(uint32_t f) { return dxb_bytes_per_pixel(f) != 0; }

int32_t compute_pitch(uint32_t fmt, size_t w, size_t h, size_t* row, size_t* slice)
{
    if (const uint32_t bs = dxb_bc_block_bytes(fmt))
    {
        const size_t nbw = std::max<size_t>(1, (w + 3) / 4), nbh = std::max<size_t>(1, (h + 3) / 4);
        *row = nbw * bs; *slice = *row * nbh;
        return DXB_S_OK;
    }
    if (const uint32_t bpp = dxb_bytes_per_pixel(fmt))
    {
        *row = w * bpp; *slice = *row * h;
        return DXB_S_OK;
    }
    return DXB_E_NOT_SUPPORTED;
}

size_t count_mips(size_t w, size_t h)
{
    size_t n = 1;
    while (h > 1 || w > 1) { if (h > 1) h >>= 1; if (w > 1) w >>= 1; ++n; }
    return n;
}

// ---- generic launch helper ------------------------------------------------------------------
template <typename J>
struct DeviceJobs
{
    J* d = nullptr; cudaStream_t s = nullptr;
    int32_t upload(const std::vector<J>& jobs, cudaStream_t stream)
    {
        s = stream;
        if (jobs.size() <= 1) return DXB_S_OK;
        DXB_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&d), jobs.size() * sizeof(J), stream));
        DXB_CUDA(cudaMemcpyAsync(d, jobs.data(), jobs.size() * sizeof(J), cudaMemcpyHostToDevice, stream));
        return DXB_S_OK;
    }
    void release() { if (d) { cudaFreeAsync(d, s); d = nullptr; } }
};

int32_t check_launch(const char* name)
{
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return cuda_hr(cudaGetLastError(), name);
}

// ---- Compress ---------------------------------------------------------------------------------
struct CompressPlan { dxb_compress_params P; bool bc7, bc6h; };

// validation + flag resolution shared by host and device variants (DirectXTexCompress.cpp:664-676, 732-749, 72-107)
int32_t plan_compress(const dxb200_image* src, size_t n, uint32_t dstFormat, uint32_t flags, float threshold,
                      const dxb200_image* dst, CompressPlan* plan)
{
    if (!src || !dst || !n) return DXB_E_INVALIDARG;
    const uint32_t srcFormat = src[0].format;
    if (is_compressed(srcFormat) || !is_compressed(dstFormat)) return DXB_E_INVALIDARG;
    if (!is_supported_pixel_format(srcFormat)) return DXB_E_NOT_SUPPORTED;        // no CPU fallback for other formats
    for (size_t i = 0; i < n; ++i)
    {
        if (!src[i].pixels || !dst[i].pixels) return DXB_E_POINTER;
        if (src[i].format != srcFormat || dst[i].format != dstFormat) return DXB_E_INVALIDARG;
        if (src[i].width != dst[i].width || src[i].height != dst[i].height) return DXB_E_FAIL;
        if (!src[i].width || !src[i].height || src[i].width > 0xFFFFFFFFull || src[i].height > 0xFFFFFFFFull) return DXB_E_INVALIDARG;
    }
    dxb_compress_params& P = plan->P;
    P.srcFormat = srcFormat; P.dstFormat = dstFormat;
    P.inF = dxb_convert_flags(srcFormat); P.outF = dxb_convert_flags(dstFormat);
    uint32_t cflags = 0;                                                       // DetermineEncoderSettings :46-68
    if (dstFormat == DXB_FMT_BC4_UNORM || dstFormat == DXB_FMT_BC4_SNORM) cflags = DXB_FILTER_RGB_COPY_RED;
    if (dstFormat == DXB_FMT_BC5_UNORM || dstFormat == DXB_FMT_BC5_SNORM) cflags = DXB_FILTER_RGB_COPY_RED | DXB_FILTER_RGB_COPY_GREEN;
    cflags |= (flags & DXB_FILTER_SRGB_MASK);                                  // GetSRGBFlags :37-44
    P.cflags = dxb_resolve_srgb_convert(cflags, srcFormat, dstFormat);
    P.bcflags = flags & (DXB_BC_FLAGS_DITHER_RGB | DXB_BC_FLAGS_DITHER_A | DXB_BC_FLAGS_UNIFORM |
                         DXB_BC_FLAGS_USE_3SUBSETS | DXB_BC_FLAGS_FORCE_BC7_MODE6);                 // GetBCFlags :26-35
    P.threshold = threshold;
    plan->bc7 = (dstFormat == DXB_FMT_BC7_UNORM || dstFormat == DXB_FMT_BC7_UNORM_SRGB);
    plan->bc6h = (dstFormat == DXB_FMT_BC6H_UF16 || dstFormat == DXB_FMT_BC6H_SF16);
    return DXB_S_OK;
}

// enqueue the kernel for images whose pixels already live on the device
int32_t launch_compress(const CompressPlan& plan, const dxb200_image* src, const dxb200_image* dst, size_t n, cudaStream_t stream)
{
    std::vector<dxb_job> jobs(n);
    uint64_t total = 0;
    for (size_t i = 0; i < n; ++i)
    {
        dxb_job& j = jobs[i];
        j.src = src[i].pixels; j.dst = dst[i].pixels;
        j.srcPitch = src[i].rowPitch; j.dstPitch = dst[i].rowPitch;
        j.width = (uint32_t)src[i].width; j.height = (uint32_t)src[i].height;
        j.nbx = (j.width + 3) / 4; j.nby = (j.height + 3) / 4;
        j.firstUnit = (uint32_t)total; j.pad = 0;
        total += (uint64_t)j.nbx * j.nby;
        if (total > 0x7FFFFFFFull) return DXB_E_INVALIDARG;                    // same 2^31-block limit as CompressBC_Parallel (:258)
    }
    dxb_compress_params P = plan.P;
    P.totalUnits = (uint32_t)total; P.njobs = (uint32_t)n;
    // (a periodic job-table lookup for batches of equal mip chains -- one division and a short scan instead of the binary
    //  search -- was measured slower on C4: 64.3 vs 60.4 ms; the binary search's loads are warp-uniform and stay in L1)
    P.periodUnits = 0; P.periodJobs = 0;
    DeviceJobs<dxb_job> dj;
    int32_t hr = dj.upload(jobs, stream);
    if (hr != DXB_S_OK) return hr;
    if (plan.bc6h)
    {
        const uint32_t need = (uint32_t)((total + 2 * DXB_BC6H_WARPS - 1) / (2 * DXB_BC6H_WARPS));
        const uint32_t grid = std::max(1u, std::min<uint32_t>(need, (uint32_t)t_v.dev->gridBC6H * 4u));
        dxb_launch_bc6h(grid, stream, dj.d, jobs[0], P);
        hr = check_launch("k_compress_bc6h");
    }
    else if (plan.bc7)
    {
        const uint32_t need = (uint32_t)((total + 2 * DXB_BC7_WARPS - 1) / (2 * DXB_BC7_WARPS));
        // one CTA per 2 * DXB_BC7_WARPS blocks (no grid-stride cap): block costs differ (alpha blocks run the separate-alpha
        // tasks), so the hardware CTA scheduler balances better than a static stride
        const uint32_t grid = std::max(1u, need);
        // RGBA32F sources of full blocks: persistent kernel fed by TMA tile loads; everything else: the direct kernel
        if (dxb_launch_bc7_tma((unsigned)t_v.dev->gridBC7, stream, jobs.data(), P)) g_tma_launches.fetch_add(1, std::memory_order_relaxed);
        else dxb_launch_bc7(grid, stream, dj.d, jobs[0], P);
        hr = check_launch("k_compress_bc7");
    }
    else
    {
        const uint32_t need = (uint32_t)((total + 127) / 128);
        const uint32_t grid = std::max(1u, std::min<uint32_t>(need, (uint32_t)t_v.dev->gridBC15 * 4u));
        dxb_launch_bc15(grid, stream, dj.d, jobs[0], P);
        hr = check_launch("k_compress_bc15");
    }
    dj.release();
    return hr;
}

// ---- host staging -------------------------------------------------------------------------------------
// Host images are cut into BANDS of whole work rows (4 pixel rows per block row on the BC side) of about 32 MiB, and the
// bands are pushed through NSLOT (stream, device buffer) slots: H2D -> kernel -> D2H of one band overlaps the other
// slots' copies and kernels (fully when the caller's memory is pinned, see dxb200_host_alloc).  Band boundaries fall on
// block rows, so the result is identical to processing the whole image at once.
struct BandSplit { std::vector<dxb200_image> src, dst; std::vector<size_t> units; };      // units = progress units a band completes

// srcRows/dstRows: pixel (or block) rows of the source/destination image consumed/produced per work row
void split_bands(const dxb200_image* src, const dxb200_image* dst, size_t n, size_t srcRows, size_t dstRows, bool srcIsBC, bool dstIsBC, BandSplit& out)
{
    const size_t BAND = size_t(32) << 20;
    for (size_t m = 0; m < n; ++m)
    {
        const size_t srcTotalRows = srcIsBC ? (src[m].height + 3) / 4 : src[m].height;
        const size_t dstTotalRows = dstIsBC ? (dst[m].height + 3) / 4 : dst[m].height;
        const size_t units = std::max<size_t>(1, (srcTotalRows + srcRows - 1) / srcRows);
        const size_t bytesPerUnit = src[m].rowPitch * srcRows + dst[m].rowPitch * dstRows;
        const size_t per = std::max<size_t>(1, BAND / std::max<size_t>(bytesPerUnit, 1));
        for (size_t u0 = 0; u0 < units; u0 += per)
        {
            const size_t u1 = std::min(units, u0 + per);
            dxb200_image s = src[m], d = dst[m];
            const size_t sr0 = u0 * srcRows, sr1 = std::min(srcTotalRows, u1 * srcRows);
            const size_t dr0 = u0 * dstRows, dr1 = std::min(dstTotalRows, u1 * dstRows);
            s.pixels = src[m].pixels + sr0 * src[m].rowPitch; s.slicePitch = (sr1 - sr0) * src[m].rowPitch;
            d.pixels = dst[m].pixels + dr0 * dst[m].rowPitch; d.slicePitch = (dr1 - dr0) * dst[m].rowPitch;
            // pixel heights of the band (the uncompressed side counts pixel rows; the BC side the same pixel rows)
            const size_t pixRows = srcIsBC ? std::min(src[m].height, sr1 * 4) - sr0 * 4 : (sr1 - sr0);
            s.height = pixRows; d.height = pixRows;
            out.src.push_back(s); out.dst.push_back(d);
            // progress as the reference reports it: pixel rows of a single image, images of an array (:115-121, 785-837)
            out.units.push_back(n == 1 ? pixRows : (u1 == units ? 1 : 0));
        }
    }
}

// dst == nullptr: the kernels write no image (IsAlphaAllOpaque); dstIn: dst[] is a second INPUT, copied up like src and not back
// (ComputeMSE)
template <typename LaunchFn>
int32_t run_staged(const dxb200_image* src, const dxb200_image* dst, size_t n, LaunchFn fn, Progress* prog = nullptr, const size_t* units = nullptr,
                   bool dstIn = false)
{
    const size_t CHUNK = size_t(48) << 20;
    size_t i = 0; int slot = 0;
    int32_t hr = DXB_S_OK;
    while (i < n && hr == DXB_S_OK)
    {
        size_t inBytes = 0, outBytes = 0, k = i;
        while (k < n)
        {
            const size_t a = (src[k].slicePitch + 255) & ~size_t(255), b = dst ? (dst[k].slicePitch + 255) & ~size_t(255) : 0;
            if (k > i && (inBytes + a + outBytes + b) > CHUNK) break;
            inBytes += a; outBytes += b; ++k;
        }
        cudaStream_t st = t_v.lane->streams[slot];
        hr = cuda_hr(cudaStreamSynchronize(st), "slot sync"); if (hr) break;
        if (prog)
        {
            size_t add = 0;
            for (size_t m = i; m < k; ++m) add += units ? units[m] : 0;
            if (!prog->report(add)) { hr = DXB_E_ABORT; break; }
        }
        hr = ensure_buffer(&t_v.lane->dIn[slot], &t_v.lane->dInCap[slot], inBytes); if (hr) break;
        hr = ensure_buffer(&t_v.lane->dOut[slot], &t_v.lane->dOutCap[slot], outBytes); if (hr) break;
        std::vector<dxb200_image> ds(src + i, src + k), dd;
        if (dst) dd.assign(dst + i, dst + k);
        size_t offIn = 0, offOut = 0;
        for (size_t m = i; m < k && hr == DXB_S_OK; ++m)
        {
            ds[m - i].pixels = static_cast<uint8_t*>(t_v.lane->dIn[slot]) + offIn;
            hr = cuda_hr(cudaMemcpyAsync(ds[m - i].pixels, src[m].pixels, src[m].slicePitch, cudaMemcpyHostToDevice, st), "H2D");
            offIn += (src[m].slicePitch + 255) & ~size_t(255);
            if (!dst) continue;
            dd[m - i].pixels = static_cast<uint8_t*>(t_v.lane->dOut[slot]) + offOut;
            if (dstIn && hr == DXB_S_OK) hr = cuda_hr(cudaMemcpyAsync(dd[m - i].pixels, dst[m].pixels, dst[m].slicePitch, cudaMemcpyHostToDevice, st), "H2D");
            offOut += (dst[m].slicePitch + 255) & ~size_t(255);
        }
        if (hr) break;
        hr = fn(ds.data(), dst ? dd.data() : nullptr, k - i, st); if (hr) break;
        for (size_t m = i; m < k && hr == DXB_S_OK && dst && !dstIn; ++m)
            hr = cuda_hr(cudaMemcpyAsync(dst[m].pixels, dd[m - i].pixels, dst[m].slicePitch, cudaMemcpyDeviceToHost, st), "D2H");
        i = k; slot = (slot + 1) % NSLOT;
    }
    for (int s = 0; s < NSLOT; ++s)
    {
        const int32_t h2 = cuda_hr(cudaStreamSynchronize(t_v.lane->streams[s]), "final sync");
        if (hr == DXB_S_OK) hr = h2;
    }
    return hr;
}

// ---- Convert ----------------------------------------------------------------------------------
int32_t plan_convert(const dxb200_image* src, size_t n, uint32_t dstFormat, uint32_t filter, const dxb200_image* dst, dxb_convert_params* P)
{
    if (!src || !dst || !n) return DXB_E_INVALIDARG;
    const uint32_t srcFormat = src[0].format;
    // Convert/ConvertEx argument checks (DirectXTexConvert.cpp:5113-5125): same format, BC formats -> E_INVALIDARG
    if (srcFormat == dstFormat) return DXB_E_INVALIDARG;
    if (is_compressed(srcFormat) || is_compressed(dstFormat)) return DXB_E_INVALIDARG;
    if (!is_supported_pixel_format(srcFormat) || !is_supported_pixel_format(dstFormat)) return DXB_E_NOT_SUPPORTED;
    // TEX_FILTER_DITHER = ordered 4x4 dithering; TEX_FILTER_DITHER_DIFFUSION = Floyd-Steinberg (serial per image, :4815-4858)
    if (filter & (DXB_FILTER_DITHER_MASK & ~(DXB_FILTER_DITHER | DXB_FILTER_DITHER_DIFFUSION))) return DXB_E_NOT_SUPPORTED;
    // the 16-bit packed destinations have dithered stores in the reference (:4302-4500) that this backend does not restate yet
    if ((filter & DXB_FILTER_DITHER_MASK) && (dstFormat == DXB_FMT_B5G6R5_UNORM || dstFormat == DXB_FMT_B5G5R5A1_UNORM || dstFormat == DXB_FMT_B4G4R4A4_UNORM))
        return DXB_E_NOT_SUPPORTED;
    for (size_t i = 0; i < n; ++i)
    {
        if (!src[i].pixels || !dst[i].pixels) return DXB_E_POINTER;
        if (src[i].format != srcFormat || dst[i].format != dstFormat) return DXB_E_INVALIDARG;
        if (src[i].width != dst[i].width || src[i].height != dst[i].height) return DXB_E_FAIL;
        if ((uint64_t)src[i].width * src[i].height > 0x7FFFFFFFull) return DXB_E_INVALIDARG;
    }
    P->srcFormat = srcFormat; P->dstFormat = dstFormat;
    P->inF = dxb_convert_flags(srcFormat); P->outF = dxb_convert_flags(dstFormat);
    P->flags = dxb_resolve_srgb_convert(filter, srcFormat, dstFormat);
    P->threshold = 0.5f;
    return DXB_S_OK;
}

int32_t launch_convert(dxb_convert_params P, const dxb200_image* src, const dxb200_image* dst, size_t n, cudaStream_t stream)
{
    std::vector<dxb_job> jobs(n);
    uint64_t total = 0;
    for (size_t i = 0; i < n; ++i)
    {
        dxb_job& j = jobs[i];
        j.src = src[i].pixels; j.dst = dst[i].pixels; j.srcPitch = src[i].rowPitch; j.dstPitch = dst[i].rowPitch;
        j.width = (uint32_t)src[i].width; j.height = (uint32_t)src[i].height; j.nbx = j.nby = 0; j.pad = 0;
        j.firstUnit = (uint32_t)total;
        total += (uint64_t)j.width * j.height;
        if (total > 0x7FFFFFFFull) return DXB_E_INVALIDARG;
    }
    P.totalUnits = (uint32_t)total; P.njobs = (uint32_t)n;
    DeviceJobs<dxb_job> dj;
    int32_t hr = dj.upload(jobs, stream);
    if (hr != DXB_S_OK) return hr;
    if (P.flags & DXB_FILTER_DITHER_DIFFUSION)
    {
        // two error rows of (width + 2) pixels per image
        uint32_t maxw = 0;
        for (const dxb_job& j : jobs) maxw = std::max(maxw, j.width);
        const uint32_t errStride = 2u * (maxw + 2u);
        void* dErr = nullptr;
        hr = cuda_hr(cudaMallocAsync(&dErr, (size_t)errStride * n * sizeof(float) * 4, stream), "cudaMallocAsync(errors)");
        if (hr == DXB_S_OK)
        {
            dxb_launch_convert_diffuse(stream, (n > 1) ? dj.d : nullptr, jobs.data(), P, dErr, errStride);
            hr = check_launch("k_convert_diffuse");
            cudaFreeAsync(dErr, stream);
        }
        dj.release();
        return hr;
    }
    const uint32_t need = (uint32_t)((total + 255) / 256);
    const uint32_t grid = std::max(1u, std::min<uint32_t>(need, (uint32_t)t_v.dev->gridRow * 8u));
    dxb_launch_convert(grid, stream, dj.d, jobs.data(), P);
    hr = check_launch("k_convert");
    dj.release();
    return hr;
}

// ---- PremultiplyAlpha ---------------------------------------------------------------------------
int32_t plan_pmalpha(const dxb200_image* src, size_t n, uint32_t flags, const dxb200_image* dst, dxb_convert_params* P)
{
    if (!src || !dst || !n) return DXB_E_INVALIDARG;
    const uint32_t fmt = src[0].format;
    if (is_compressed(fmt)) return DXB_E_NOT_SUPPORTED;                                 // :224-229
    if (!is_supported_pixel_format(fmt)) return DXB_E_NOT_SUPPORTED;
    if (!(dxb_convert_flags(fmt) & DXB_CONVF_A)) return DXB_E_NOT_SUPPORTED;            // !HasAlpha
    for (size_t i = 0; i < n; ++i)
    {
        if (!src[i].pixels || !dst[i].pixels) return DXB_E_POINTER;
        if (src[i].format != fmt || dst[i].format != fmt) return DXB_E_INVALIDARG;
        if (src[i].width != dst[i].width || src[i].height != dst[i].height || !src[i].width || !src[i].height) return DXB_E_INVALIDARG;
    }
    memset(P, 0, sizeof(*P));
    P->srcFormat = fmt; P->dstFormat = fmt; P->inF = P->outF = dxb_convert_flags(fmt);
    // TEX_PMALPHA_IGNORE_SRGB = 0x1, TEX_PMALPHA_REVERSE = 0x2; the SRGB bits equal TEX_FILTER_SRGB_IN/OUT (:21-26)
    const uint32_t lflags = (flags & 0x1u) ? 0u : dxb_resolve_srgb_linear(flags & DXB_FILTER_SRGB_MASK, fmt);
    P->flags = (lflags & (DXB_FILTER_SRGB_IN | DXB_FILTER_SRGB_OUT)) | ((flags & 0x2u) ? 1u : 0u);
    return DXB_S_OK;
}

int32_t launch_pmalpha(dxb_convert_params P, const dxb200_image* src, const dxb200_image* dst, size_t n, cudaStream_t stream)
{
    std::vector<dxb_job> jobs(n);
    uint64_t total = 0;
    for (size_t i = 0; i < n; ++i)
    {
        dxb_job& j = jobs[i];
        j.src = src[i].pixels; j.dst = dst[i].pixels; j.srcPitch = src[i].rowPitch; j.dstPitch = dst[i].rowPitch;
        j.width = (uint32_t)src[i].width; j.height = (uint32_t)src[i].height; j.nbx = j.nby = 0; j.pad = 0;
        j.firstUnit = (uint32_t)total;
        total += (uint64_t)j.width * j.height;
        if (total > 0x7FFFFFFFull) return DXB_E_INVALIDARG;
    }
    P.totalUnits = (uint32_t)total; P.njobs = (uint32_t)n;
    DeviceJobs<dxb_job> dj;
    int32_t hr = dj.upload(jobs, stream);
    if (hr != DXB_S_OK) return hr;
    const uint32_t need = (uint32_t)((total + 255) / 256);
    const uint32_t grid = std::max(1u, std::min<uint32_t>(need, (uint32_t)t_v.dev->gridRow * 8u));
    dxb_launch_pmalpha(grid, stream, dj.d, jobs.data(), P);
    hr = check_launch("k_pmalpha");
    dj.release();
    return hr;
}

// ---- GenerateMipMaps ----------------------------------------------------------------------------
bool ispow2(size_t x) { return ((x != 0) && !(x & (x - 1))); }

int32_t plan_mips(const dxb200_image* chain, size_t items, size_t levels, uint32_t filter, uint32_t* mode)
{
    if (!chain || !items || levels < 2) return DXB_E_INVALIDARG;
    const uint32_t fmt = chain[0].format;
    if (is_compressed(fmt)) return DXB_E_NOT_SUPPORTED;                         // GenerateMipMaps :2852-2856
    if (!is_supported_pixel_format(fmt)) return DXB_E_NOT_SUPPORTED;
    const size_t w = chain[0].width, h = chain[0].height;
    if (levels > count_mips(w, h)) return DXB_E_INVALIDARG;
    for (size_t it = 0; it < items; ++it)
    {
        size_t lw = w, lh = h;
        for (size_t l = 0; l < levels; ++l)
        {
            const dxb200_image& im = chain[it * levels + l];
            if (!im.pixels) return DXB_E_POINTER;
            if (im.format != fmt || im.width != lw || im.height != lh) return DXB_E_INVALIDARG;
            if (lh > 1) lh >>= 1;
            if (lw > 1) lw >>= 1;
        }
    }
    uint32_t m = filter & DXB_FILTER_MODE_MASK;
    if (!m) m = (ispow2(w) && ispow2(h)) ? DXB_FILTER_BOX : DXB_FILTER_LINEAR;   // :3169-3174
    switch (m)
    {
    case DXB_FILTER_BOX: if (!ispow2(w) || !ispow2(h)) return DXB_E_FAIL; break;     // :1005-1006
    case DXB_FILTER_POINT: case DXB_FILTER_LINEAR: case DXB_FILTER_CUBIC: case DXB_FILTER_TRIANGLE: break;
    default: return DXB_E_NOT_SUPPORTED;
    }
    if ((uint64_t)w * h * items > 0x7FFFFFFFull) return DXB_E_INVALIDARG;
    *mode = m;
    return DXB_S_OK;
}

// Resize = one filter pass from src[i] to dst[i] (PerformResizeUsingCustomFilters, DirectXTexResize.cpp:805-837)
int32_t plan_resize(const dxb200_image* src, size_t n, uint32_t filter, const dxb200_image* dst, uint32_t* mode)
{
    if (!src || !dst || !n) return DXB_E_INVALIDARG;
    const uint32_t fmt = src[0].format;
    if (is_compressed(fmt)) return DXB_E_NOT_SUPPORTED;                         // Resize :875-879
    if (!is_supported_pixel_format(fmt)) return DXB_E_NOT_SUPPORTED;
    const size_t sw = src[0].width, sh = src[0].height, dw = dst[0].width, dh = dst[0].height;
    if (!sw || !sh || !dw || !dh) return DXB_E_INVALIDARG;
    if (sw > 0xFFFFFFFFull || sh > 0xFFFFFFFFull || dw > 0xFFFFFFFFull || dh > 0xFFFFFFFFull) return DXB_E_INVALIDARG;
    for (size_t i = 0; i < n; ++i)
    {
        if (!src[i].pixels || !dst[i].pixels) return DXB_E_POINTER;
        if (src[i].format != fmt || dst[i].format != fmt) return DXB_E_INVALIDARG;
        if (src[i].width != sw || src[i].height != sh || dst[i].width != dw || dst[i].height != dh) return DXB_E_INVALIDARG;
    }
    uint32_t m = filter & DXB_FILTER_MODE_MASK;
    if (!m) m = ((dw << 1) == sw && (dh << 1) == sh) ? DXB_FILTER_BOX : DXB_FILTER_LINEAR;      // :812-817
    switch (m)
    {
    case DXB_FILTER_BOX: if ((dw << 1) != sw || (dh << 1) != sh) return DXB_E_FAIL; break;      // :318-319
    case DXB_FILTER_POINT: case DXB_FILTER_LINEAR: case DXB_FILTER_CUBIC: case DXB_FILTER_TRIANGLE: break;
    default: return DXB_E_NOT_SUPPORTED;
    }
    if ((uint64_t)dw * dh * n > 0x7FFFFFFFull) return DXB_E_INVALIDARG;
    *mode = m;
    return DXB_S_OK;
}

// chain[] holds DEVICE pointers; level 0 of each item is populated
int32_t launch_mips(const dxb200_image* chain, size_t items, size_t levels, uint32_t filter, uint32_t mode, cudaStream_t stream)
{
    const uint32_t fmt = chain[0].format;
    dxb_mip_params P; memset(&P, 0, sizeof(P));
    P.format = fmt; P.mode = mode; P.filter = filter;
    P.lflags = dxb_resolve_srgb_linear(filter & DXB_FILTER_SRGB_MASK, fmt);
    int32_t hr = DXB_S_OK;
    // job records of every level, built once and uploaded with ONE copy (a per-level upload left the GPU idle
    // between the small launches of the tail of the chain)
    std::vector<const dxb200_image*> stale(items, nullptr);
    std::vector<dxb_mip_job> all(items * (levels - 1));
    std::vector<uint64_t> totals(levels, 0);
    for (size_t l = 1; l < levels; ++l)
    {
        uint64_t total = 0;
        for (size_t it = 0; it < items; ++it)
        {
            const dxb200_image& s = chain[it * levels + l - 1]; const dxb200_image& d = chain[it * levels + l];
            dxb_mip_job& j = all[(l - 1) * items + it];
            j.src = s.pixels; j.dst = d.pixels; j.srcPitch = s.rowPitch; j.dstPitch = d.rowPitch;
            j.sw = (uint32_t)s.width; j.sh = (uint32_t)s.height; j.dw = (uint32_t)d.width; j.dh = (uint32_t)d.height;
            j.firstUnit = (uint32_t)total; total += (uint64_t)j.dw * j.dh;
            if (s.height == 2) stale[it] = &s;          // box filter quirk, see dxb_mip_box
            j.stale = nullptr; j.stalePitch = 0;
            if (mode == DXB_FILTER_BOX && s.height <= 1 && s.width > 1 && stale[it])
            {
                j.stale = stale[it]->pixels + stale[it]->rowPitch;      // row 1 of that level
                j.stalePitch = stale[it]->rowPitch;
            }
        }
        totals[l] = total;
    }
    dxb_mip_job* dAll = nullptr;
    // first level whose SOURCE is at most 64x64: from there on one CTA per item finishes the chain in one launch
    size_t tailStart = levels;
    for (size_t l = 1; l < levels; ++l)
        if (chain[l - 1].width <= 64 && chain[l - 1].height <= 64) { tailStart = l; break; }
    const bool wantTail = (mode == DXB_FILTER_BOX || mode == DXB_FILTER_LINEAR || mode == DXB_FILTER_CUBIC) && (levels - tailStart) >= 2 && items <= 0x7FFFFFFFull;
    const bool wantFused = (mode == DXB_FILTER_BOX || mode == DXB_FILTER_LINEAR) && levels >= 4;      // LINEAR at 2:1 reads the same 2x2 patches
    if (items > 1 || wantTail || wantFused)
    {
        DXB_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&dAll), all.size() * sizeof(dxb_mip_job), stream));
        DXB_CUDA(cudaMemcpyAsync(dAll, all.data(), all.size() * sizeof(dxb_mip_job), cudaMemcpyHostToDevice, stream));
    }
    for (size_t l = 1; l < levels && hr == DXB_S_OK; ++l)
    {
        // three BOX / LINEAR levels per launch while the source is larger than the tail kernel's 64x64 and divides by 8
        if (wantFused && l + 2 < levels && (chain[l - 1].width > 64 || chain[l - 1].height > 64))
        {
            P.njobs = (uint32_t)items;
            if (dxb_launch_mip_box3(stream, dAll + (l - 1) * items, all.data() + (l - 1) * items, (uint32_t)items, P))
            {
                hr = check_launch("k_mip_box3");
                l += 2;
                continue;
            }
        }
        if (wantTail && l >= tailStart)
        {
            P.njobs = (uint32_t)items;
            if (dxb_launch_mip_tail(stream, dAll + (l - 1) * items, (uint32_t)items, (uint32_t)(levels - l), P))
            {
                hr = check_launch("k_mip_tail");
                break;
            }
        }
        if (mode == DXB_FILTER_TRIANGLE)
        {
            // gather lists are per level and shared by all items
            const dxb200_image& s0 = chain[l - 1]; const dxb200_image& d0 = chain[l];
            TriLists tx, ty;
            build_triangle_axis(s0.width, d0.width, (filter & DXB_FILTER_WRAP_U) != 0, tx);
            build_triangle_axis(s0.height, d0.height, (filter & DXB_FILTER_WRAP_V) != 0, ty);
            const size_t nOff = tx.off.size() + ty.off.size(), nEnt = tx.src.size() + ty.src.size();
            uint32_t* dU = nullptr; float* dW = nullptr;
            DXB_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&dU), (nOff + nEnt) * sizeof(uint32_t), stream));
            DXB_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&dW), nEnt * sizeof(float), stream));
            std::vector<uint32_t> hu; hu.reserve(nOff + nEnt);
            hu.insert(hu.end(), tx.off.begin(), tx.off.end()); hu.insert(hu.end(), ty.off.begin(), ty.off.end());
            hu.insert(hu.end(), tx.src.begin(), tx.src.end()); hu.insert(hu.end(), ty.src.begin(), ty.src.end());
            std::vector<float> hw; hw.reserve(nEnt);
            hw.insert(hw.end(), tx.w.begin(), tx.w.end()); hw.insert(hw.end(), ty.w.begin(), ty.w.end());
            DXB_CUDA(cudaMemcpyAsync(dU, hu.data(), hu.size() * sizeof(uint32_t), cudaMemcpyHostToDevice, stream));
            DXB_CUDA(cudaMemcpyAsync(dW, hw.data(), hw.size() * sizeof(float), cudaMemcpyHostToDevice, stream));
            DXB_CUDA(cudaStreamSynchronize(stream));      // host vectors go out of scope below
            P.triX.off = dU; P.triY.off = dU + tx.off.size();
            P.triX.src = dU + nOff; P.triY.src = dU + nOff + tx.src.size();
            P.triX.w = dW; P.triY.w = dW + tx.w.size();
        }
        const uint64_t total = totals[l];
        P.totalUnits = (uint32_t)total; P.njobs = (uint32_t)items;
        const uint32_t need = (uint32_t)((total + 255) / 256);
        const uint32_t grid = std::max(1u, std::min<uint32_t>(need, (uint32_t)t_v.dev->gridRow * 8u));
        dxb_launch_mip(grid, stream, (dAll && items > 1) ? dAll + (l - 1) * items : nullptr, all.data() + (l - 1) * items, P);
        hr = check_launch("k_mip_level");
        if (mode == DXB_FILTER_TRIANGLE)
        {
            cudaFreeAsync(const_cast<uint32_t*>(P.triX.off), stream);
            cudaFreeAsync(const_cast<float*>(P.triX.w), stream);
        }
    }
    if (dAll) cudaFreeAsync(dAll, stream);
    return hr;
}

} // namespace

// =================================================================================================
extern "C" {

const char* dxb200_version(void) { return "dxtex_b200 0.1 (sm_100a)"; }
const char* dxb200_last_error(void) { return t_lastError.c_str(); }
uint64_t dxb200_launch_count(void) { return g_launches.load(); }
uint64_t dxb200_tma_launch_count(void) { return g_tma_launches.load(); }
int32_t dxb200_set_option(uint32_t option, int32_t value)
{
    if (option == DXB200_OPT_BC7_FEED) { dxb_bc7_set_feed(value); return DXB_S_OK; }
    return DXB_E_INVALIDARG;
}
int32_t dxb200_get_option(uint32_t option) { return (option == DXB200_OPT_BC7_FEED) ? dxb_bc7_get_feed() : -1; }

int32_t dxb200_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { (void)cudaGetLastError(); return 0; }
    return n;
}

int32_t dxb200_init_devices(int ndev, const int* devices)
{
    if (ndev <= 0 || !devices) return DXB_E_INVALIDARG;
    std::lock_guard<std::mutex> lk(g_mu);
    int prev = -1;
    if (cudaGetDevice(&prev) != cudaSuccess) { (void)cudaGetLastError(); prev = -1; }
    int32_t hr = DXB_S_OK;
    for (int i = 0; i < ndev && hr == DXB_S_OK; ++i) hr = init_device_locked(devices[i], nullptr);
    // the calling thread keeps the first listed device current (what dxb200_init(device) always did)
    if (hr == DXB_S_OK) hr = cuda_hr(cudaSetDevice(devices[0]), "cudaSetDevice");
    else if (prev >= 0) (void)cudaSetDevice(prev);
    return hr;
}

int32_t dxb200_init(int device) { return dxb200_init_devices(1, &device); }

int32_t dxb200_initialized_devices(int* devices, int maxDevices)
{
    std::lock_guard<std::mutex> lk(g_mu);
    for (size_t i = 0; i < g_devs.size() && devices && (int)i < maxDevices; ++i) devices[i] = g_devs[i]->ordinal;
    return (int32_t)g_devs.size();
}

void dxb200_shutdown(void)
{
    std::lock_guard<std::mutex> lk(g_mu);
    int prev = -1;
    if (cudaGetDevice(&prev) != cudaSuccess) { (void)cudaGetLastError(); prev = -1; }
    for (auto& d : g_devs)
    {
        if (cudaSetDevice(d->ordinal) != cudaSuccess) { (void)cudaGetLastError(); continue; }
        for (int l = 0; l < NLANE; ++l)
            for (int i = 0; i < NSLOT; ++i)
            {
                Lane& L = d->lanes[l];
                if (L.streams[i]) { cudaStreamSynchronize(L.streams[i]); cudaStreamDestroy(L.streams[i]); L.streams[i] = nullptr; }
                if (L.dIn[i]) { cudaFree(L.dIn[i]); L.dIn[i] = nullptr; L.dInCap[i] = 0; }
                if (L.dOut[i]) { cudaFree(L.dOut[i]); L.dOut[i] = nullptr; L.dOutCap[i] = 0; }
            }
    }
    g_devs.clear();
    if (prev >= 0) (void)cudaSetDevice(prev);
}

// Pinned host memory for full-rate, overlapped H2D / D2H.  The pages are placed on the NUMA node of the calling thread's
// current CUDA device (memory policy MPOL_PREFERRED around the allocation): a rank whose staging buffers sit on the other
// socket pays the inter-socket link on every copy (8 ranks x 51 GB/s measured 0.75 end-to-end efficiency in round 1).
void* dxb200_host_alloc(size_t bytes)
{
    std::vector<Device*> devs;
    if (device_list(&devs) != DXB_S_OK) return nullptr;
    int cur = -1, node = -1;
    if (cudaGetDevice(&cur) != cudaSuccess) { (void)cudaGetLastError(); cur = -1; }
    for (Device* d : devs) if (d->ordinal == cur) node = d->numaNode;
    if (node < 0 && cur >= 0) node = device_numa_node(cur);
    bool policy = false;
#if defined(SYS_set_mempolicy)
    if (node >= 0 && node < 64)
    {
        unsigned long mask = 1ul << node;
        policy = (syscall(SYS_set_mempolicy, 1 /* MPOL_PREFERRED */, &mask, sizeof(mask) * 8 + 1) == 0);
    }
#endif
    void* p = nullptr;
    const cudaError_t e = cudaHostAlloc(&p, bytes, cudaHostAllocPortable);
#if defined(SYS_set_mempolicy)
    if (policy) (void)syscall(SYS_set_mempolicy, 0 /* MPOL_DEFAULT */, nullptr, 0);
#endif
    if (e != cudaSuccess) { (void)cudaGetLastError(); return nullptr; }
    return p;
}
void dxb200_host_free(void* p) { if (p) cudaFreeHost(p); }

int32_t dxb200_compute_pitch(uint32_t format, size_t width, size_t height, size_t* rowPitch, size_t* slicePitch)
{
    if (!rowPitch || !slicePitch) return DXB_E_POINTER;
    return compute_pitch(format, width, height, rowPitch, slicePitch);
}

int32_t dxb200_calculate_mip_levels(size_t width, size_t height, size_t* levels)
{
    if (!levels) return DXB_E_POINTER;
    if (*levels > 1) { if (*levels > count_mips(width, height)) return DXB_E_INVALIDARG; }
    else if (*levels == 0) *levels = count_mips(width, height);
    else *levels = 1;
    return DXB_S_OK;
}

// ---- Compress -----------------------------------------------------------------------------------
int32_t dxb200_compress_device(const dxb200_image* src, size_t nimages, uint32_t dstFormat, uint32_t flags, float threshold,
                               float alphaWeight, const dxb200_image* dst, void* stream)
{
    (void)alphaWeight;      // only the reference's DirectCompute path has an alpha weight (DirectXTex.h:919); the CPU encoder we match has none
    CompressPlan plan;
    int32_t hr = plan_compress(src, nimages, dstFormat, flags, threshold, dst, &plan);
    if (hr != DXB_S_OK) return hr;
    DevScope scope;
    hr = scope.enter(src[0].pixels);
    if (hr != DXB_S_OK) return hr;
    return launch_compress(plan, src, dst, nimages, static_cast<cudaStream_t>(stream));
}

int32_t dxb200_compress_ex(const dxb200_image* src, size_t nimages, uint32_t dstFormat, uint32_t flags, float threshold,
                           float alphaWeight, const dxb200_image* dst, dxb200_status_fn status, void* user)
{
    (void)alphaWeight;
    CompressPlan plan;
    int32_t hr = plan_compress(src, nimages, dstFormat, flags, threshold, dst, &plan);
    if (hr != DXB_S_OK) return hr;
    BandSplit bands;
    split_bands(src, dst, nimages, 4, 1, false, true, bands);
    Progress prog; prog.fn = status; prog.user = user;
    for (size_t u : bands.units) prog.total += u;
    // bands (whole block rows) are independent: contiguous band ranges go to the initialised devices, weighted by their bytes
    hr = run_sharded(bands.src.size(), [&](size_t i) { return bands.src[i].slicePitch + bands.dst[i].slicePitch; },
        [&](size_t lo, size_t hi)
        {
            return run_staged(bands.src.data() + lo, bands.dst.data() + lo, hi - lo,
                [&](const dxb200_image* ds, const dxb200_image* dd, size_t cnt, cudaStream_t st) { return launch_compress(plan, ds, dd, cnt, st); },
                status ? &prog : nullptr, bands.units.data() + lo);
        });
    if (hr == DXB_S_OK && status && !status(prog.total, prog.total, user)) hr = DXB_E_ABORT;
    return hr;
}

int32_t dxb200_compress(const dxb200_image* src, size_t nimages, uint32_t dstFormat, uint32_t flags, float threshold,
                        float alphaWeight, const dxb200_image* dst)
{
    return dxb200_compress_ex(src, nimages, dstFormat, flags, threshold, alphaWeight, dst, nullptr, nullptr);
}

// ---- Decompress (DirectXTexCompress.cpp:852-979; DecompressBC :425-535) ---------------------------------
static int32_t plan_decompress(const dxb200_image* src, size_t n, uint32_t dstFormat, const dxb200_image* dst, dxb_compress_params* P)
{
    if (!src || !dst || !n) return DXB_E_INVALIDARG;
    const uint32_t srcFormat = src[0].format;
    if (!is_compressed(srcFormat) || is_compressed(dstFormat)) return DXB_E_INVALIDARG;
    if (!is_supported_pixel_format(dstFormat)) return DXB_E_NOT_SUPPORTED;
    for (size_t i = 0; i < n; ++i)
    {
        if (!src[i].pixels || !dst[i].pixels) return DXB_E_POINTER;
        if (src[i].format != srcFormat || dst[i].format != dstFormat) return DXB_E_INVALIDARG;
        if (src[i].width != dst[i].width || src[i].height != dst[i].height) return DXB_E_FAIL;
        if (!src[i].width || !src[i].height || src[i].width > 0xFFFFFFFFull || src[i].height > 0xFFFFFFFFull) return DXB_E_INVALIDARG;
    }
    memset(P, 0, sizeof(*P));
    P->srcFormat = srcFormat; P->dstFormat = dstFormat;
    P->inF = dxb_convert_flags(srcFormat); P->outF = dxb_convert_flags(dstFormat);
    P->cflags = dxb_resolve_srgb_convert(0, srcFormat, dstFormat);          // ConvertScanline(..., TEX_FILTER_DEFAULT) (:500)
    return DXB_S_OK;
}

static int32_t launch_decompress(dxb_compress_params P, const dxb200_image* src, const dxb200_image* dst, size_t n, cudaStream_t stream)
{
    std::vector<dxb_job> jobs(n);
    uint64_t total = 0;
    for (size_t i = 0; i < n; ++i)
    {
        dxb_job& j = jobs[i];
        j.src = src[i].pixels; j.dst = dst[i].pixels; j.srcPitch = src[i].rowPitch; j.dstPitch = dst[i].rowPitch;
        j.width = (uint32_t)src[i].width; j.height = (uint32_t)src[i].height;
        j.nbx = (j.width + 3) / 4; j.nby = (j.height + 3) / 4; j.pad = 0;
        j.firstUnit = (uint32_t)total; total += (uint64_t)j.nbx * j.nby;
        if (total > 0x7FFFFFFFull) return DXB_E_INVALIDARG;
    }
    P.totalUnits = (uint32_t)total; P.njobs = (uint32_t)n;
    DeviceJobs<dxb_job> dj;
    int32_t hr = dj.upload(jobs, stream);
    if (hr != DXB_S_OK) return hr;
    const uint32_t need = (uint32_t)((total + 127) / 128);
    const uint32_t grid = std::max(1u, std::min<uint32_t>(need, (uint32_t)t_v.dev->gridBC15 * 8u));
    dxb_launch_decompress(grid, stream, dj.d, jobs[0], P);
    hr = check_launch("k_decompress");
    dj.release();
    return hr;
}

int32_t dxb200_decompress_device(const dxb200_image* src, size_t nimages, uint32_t dstFormat, const dxb200_image* dst, void* stream)
{
    dxb_compress_params P;
    int32_t hr = plan_decompress(src, nimages, dstFormat, dst, &P);
    if (hr != DXB_S_OK) return hr;
    DevScope scope;
    hr = scope.enter(src[0].pixels);
    if (hr != DXB_S_OK) return hr;
    return launch_decompress(P, src, dst, nimages, static_cast<cudaStream_t>(stream));
}

int32_t dxb200_decompress(const dxb200_image* src, size_t nimages, uint32_t dstFormat, const dxb200_image* dst)
{
    dxb_compress_params P;
    int32_t hr = plan_decompress(src, nimages, dstFormat, dst, &P);
    if (hr != DXB_S_OK) return hr;
    BandSplit bands;
    split_bands(src, dst, nimages, 1, 4, true, false, bands);
    return run_sharded(bands.src.size(), [&](size_t i) { return bands.src[i].slicePitch + bands.dst[i].slicePitch; },
        [&](size_t lo, size_t hi)
        {
            return run_staged(bands.src.data() + lo, bands.dst.data() + lo, hi - lo,
                [&](const dxb200_image* ds, const dxb200_image* dd, size_t cnt, cudaStream_t st) { return launch_decompress(P, ds, dd, cnt, st); });
        });
}

// ---- Convert ------------------------------------------------------------------------------------
int32_t dxb200_convert_device(const dxb200_image* src, size_t nimages, uint32_t dstFormat, uint32_t filter, float threshold,
                              const dxb200_image* dst, void* stream)
{
    dxb_convert_params P;
    int32_t hr = plan_convert(src, nimages, dstFormat, filter, dst, &P);
    if (hr != DXB_S_OK) return hr;
    P.threshold = threshold;       // alpha threshold of the 1-bit alpha destination (B5G5R5A1)
    DevScope scope;
    hr = scope.enter(src[0].pixels);
    if (hr != DXB_S_OK) return hr;
    return launch_convert(P, src, dst, nimages, static_cast<cudaStream_t>(stream));
}

int32_t dxb200_convert_ex(const dxb200_image* src, size_t nimages, uint32_t dstFormat, uint32_t filter, float threshold, const dxb200_image* dst,
                          dxb200_status_fn status, void* user)
{
    dxb_convert_params P;
    int32_t hr = plan_convert(src, nimages, dstFormat, filter, dst, &P);
    if (hr != DXB_S_OK) return hr;
    P.threshold = threshold;
    BandSplit bands;
    // bands start on multiples of 4 rows so that the 4x4 ordered-dither matrix keeps its phase
    // (error diffusion carries state from row to row: whole images only)
    size_t rowsPerUnit = (P.flags & DXB_FILTER_DITHER) ? 4 : 1;
    if (P.flags & DXB_FILTER_DITHER_DIFFUSION) for (size_t i = 0; i < nimages; ++i) rowsPerUnit = std::max(rowsPerUnit, src[i].height);
    split_bands(src, dst, nimages, rowsPerUnit, rowsPerUnit, false, false, bands);
    Progress prog; prog.fn = status; prog.user = user;
    for (size_t u : bands.units) prog.total += u;
    hr = run_sharded(bands.src.size(), [&](size_t i) { return bands.src[i].slicePitch + bands.dst[i].slicePitch; },
        [&](size_t lo, size_t hi)
        {
            return run_staged(bands.src.data() + lo, bands.dst.data() + lo, hi - lo,
                [&](const dxb200_image* ds, const dxb200_image* dd, size_t cnt, cudaStream_t st) { return launch_convert(P, ds, dd, cnt, st); },
                status ? &prog : nullptr, bands.units.data() + lo);
        });
    if (hr == DXB_S_OK && status && !status(prog.total, prog.total, user)) hr = DXB_E_ABORT;
    return hr;
}

int32_t dxb200_convert(const dxb200_image* src, size_t nimages, uint32_t dstFormat, uint32_t filter, float threshold, const dxb200_image* dst)
{
    return dxb200_convert_ex(src, nimages, dstFormat, filter, threshold, dst, nullptr, nullptr);
}

// ---- GenerateMipMaps ----------------------------------------------------------------------------
int32_t dxb200_generate_mipmaps_device(const dxb200_image* chain, size_t items, size_t levels, uint32_t filter, void* stream)
{
    uint32_t mode = 0;
    int32_t hr = plan_mips(chain, items, levels, filter, &mode);
    if (hr != DXB_S_OK) return hr;
    DevScope scope;
    hr = scope.enter(chain[0].pixels);
    if (hr != DXB_S_OK) return hr;
    return launch_mips(chain, items, levels, filter, mode, static_cast<cudaStream_t>(stream));
}

// host chains of items [lo, hi): level 0 up, kernels, levels 1.. down; whole items per chunk, on the calling thread's lane
static int32_t mips_host_range(const dxb200_image* chain, size_t lo, size_t hi, size_t levels, uint32_t filter, uint32_t mode)
{
    const size_t CHUNK = size_t(1) << 30;
    int32_t hr = DXB_S_OK;
    size_t it = lo;
    cudaStream_t st = t_v.lane->streams[0];
    while (it < hi && hr == DXB_S_OK)
    {
        size_t bytes = 0, k = it;
        while (k < hi)
        {
            size_t b = 0;
            for (size_t l = 0; l < levels; ++l) b += (chain[k * levels + l].slicePitch + 255) & ~size_t(255);
            if (k > it && bytes + b > CHUNK) break;
            bytes += b; ++k;
        }
        hr = ensure_buffer(&t_v.lane->dIn[0], &t_v.lane->dInCap[0], bytes); if (hr) break;
        std::vector<dxb200_image> dev(chain + it * levels, chain + k * levels);
        size_t off = 0;
        for (size_t m = 0; m < dev.size() && hr == DXB_S_OK; ++m)
        {
            dev[m].pixels = static_cast<uint8_t*>(t_v.lane->dIn[0]) + off;
            off += (dev[m].slicePitch + 255) & ~size_t(255);
            if ((m % levels) == 0)
                hr = cuda_hr(cudaMemcpyAsync(dev[m].pixels, chain[it * levels + m].pixels, dev[m].slicePitch, cudaMemcpyHostToDevice, st), "H2D");
        }
        if (hr) break;
        hr = launch_mips(dev.data(), k - it, levels, filter, mode, st); if (hr) break;
        for (size_t m = 0; m < dev.size() && hr == DXB_S_OK; ++m)
            if ((m % levels) != 0)
                hr = cuda_hr(cudaMemcpyAsync(chain[it * levels + m].pixels, dev[m].pixels, dev[m].slicePitch, cudaMemcpyDeviceToHost, st), "D2H");
        if (hr) break;
        hr = cuda_hr(cudaStreamSynchronize(st), "mips sync");
        it = k;
    }
    return hr;
}

int32_t dxb200_generate_mipmaps(const dxb200_image* chain, size_t items, size_t levels, uint32_t filter)
{
    uint32_t mode = 0;
    int32_t hr = plan_mips(chain, items, levels, filter, &mode);
    if (hr != DXB_S_OK) return hr;
    // image-per-GPU sharding: contiguous item ranges per device; a single item's chain stays on one device (SURVEY 8(e))
    return run_sharded(items, [&](size_t i) { return chain[i * levels].slicePitch; },
        [&](size_t lo, size_t hi) { return mips_host_range(chain, lo, hi, levels, filter, mode); });
}

// ---- GenerateMipMaps + Compress in one call: the mip chain never leaves HBM --------------------------------------------
// texconv runs GenerateMipMaps and then Compress on the result (Texconv/texconv.cpp; SURVEY 3.5); with the two host-pointer calls
// the chain travels device -> host -> device in between.  Here level 0 of every item goes up once, the chain is built and
// compressed in device memory, and only the packed blocks come back: 4 B/texel up + 1.33 B/texel down (BC3 from RGBA8)
// instead of 4 + 5.33 + 5.33 + 1.33.  Per item: base[i] = level 0 (host), dst[i * levels + l] = the BC image of level l (host).
// Chunks of whole items are pipelined over the lane's NSLOT (stream, buffer) slots: H2D, mip kernels, compress kernel, D2H.
int32_t dxb200_mipmaps_compress(const dxb200_image* base, size_t items, size_t levels, uint32_t filter, uint32_t dstFormat,
                                uint32_t flags, float threshold, float alphaWeight, const dxb200_image* dst)
{
    (void)alphaWeight;
    if (!base || !dst || !items || !levels) return DXB_E_INVALIDARG;
    // the chain every item will have on the device (ScratchImage layout of the source format)
    std::vector<dxb200_image> chain(items * levels);
    for (size_t i = 0; i < items; ++i)
    {
        size_t w = base[i].width, h = base[i].height;
        if (!base[i].pixels) return DXB_E_POINTER;
        if (levels > count_mips(w, h)) return DXB_E_INVALIDARG;
        for (size_t l = 0; l < levels; ++l)
        {
            dxb200_image& c = chain[i * levels + l];
            c.width = w; c.height = h; c.format = base[i].format;
            const int32_t hp = compute_pitch(c.format, w, h, &c.rowPitch, &c.slicePitch);
            if (hp != DXB_S_OK) return hp;
            c.pixels = const_cast<uint8_t*>(base[i].pixels);          // placeholder for validation; replaced by device addresses per chunk
            if (h > 1) h >>= 1;
            if (w > 1) w >>= 1;
        }
        chain[i * levels].rowPitch = base[i].rowPitch; chain[i * levels].slicePitch = base[i].slicePitch;
    }
    uint32_t mode = 0;
    int32_t hr = plan_mips(chain.data(), items, levels, filter, &mode);
    if (hr != DXB_S_OK) return hr;
    CompressPlan plan;
    hr = plan_compress(chain.data(), items * levels, dstFormat, flags, threshold, dst, &plan);
    if (hr != DXB_S_OK) return hr;
    auto range = [&](size_t lo, size_t hi) -> int32_t
    {
        const size_t CHUNK = size_t(64) << 20;
        int32_t h2 = DXB_S_OK;
        size_t it = lo; int slot = 0;
        while (it < hi && h2 == DXB_S_OK)
        {
            size_t inBytes = 0, outBytes = 0, k = it;
            while (k < hi)
            {
                size_t a = 0, b = 0;
                for (size_t l = 0; l < levels; ++l)
                {
                    a += (chain[k * levels + l].slicePitch + 255) & ~size_t(255);
                    b += (dst[k * levels + l].slicePitch + 255) & ~size_t(255);
                }
                if (k > it && inBytes + a > CHUNK) break;
                inBytes += a; outBytes += b; ++k;
            }
            cudaStream_t st = t_v.lane->streams[slot];
            h2 = cuda_hr(cudaStreamSynchronize(st), "slot sync"); if (h2) break;
            h2 = ensure_buffer(&t_v.lane->dIn[slot], &t_v.lane->dInCap[slot], inBytes); if (h2) break;
            h2 = ensure_buffer(&t_v.lane->dOut[slot], &t_v.lane->dOutCap[slot], outBytes); if (h2) break;
            std::vector<dxb200_image> dc(chain.begin() + it * levels, chain.begin() + k * levels), dd(dst + it * levels, dst + k * levels);
            size_t offIn = 0, offOut = 0;
            for (size_t m = 0; m < dc.size() && h2 == DXB_S_OK; ++m)
            {
                dc[m].pixels = static_cast<uint8_t*>(t_v.lane->dIn[slot]) + offIn;  offIn += (dc[m].slicePitch + 255) & ~size_t(255);
                dd[m].pixels = static_cast<uint8_t*>(t_v.lane->dOut[slot]) + offOut; offOut += (dd[m].slicePitch + 255) & ~size_t(255);
                if ((m % levels) == 0)
                    h2 = cuda_hr(cudaMemcpyAsync(dc[m].pixels, base[it + m / levels].pixels, dc[m].slicePitch, cudaMemcpyHostToDevice, st), "H2D");
            }
            if (h2) break;
            h2 = launch_mips(dc.data(), k - it, levels, filter, mode, st); if (h2) break;
            h2 = launch_compress(plan, dc.data(), dd.data(), dc.size(), st); if (h2) break;
            for (size_t m = 0; m < dd.size() && h2 == DXB_S_OK; ++m)
                h2 = cuda_hr(cudaMemcpyAsync(dst[it * levels + m].pixels, dd[m].pixels, dd[m].slicePitch, cudaMemcpyDeviceToHost, st), "D2H");
            it = k; slot = (slot + 1) % NSLOT;
        }
        for (int sl = 0; sl < NSLOT; ++sl)
        {
            const int32_t h3 = cuda_hr(cudaStreamSynchronize(t_v.lane->streams[sl]), "final sync");
            if (h2 == DXB_S_OK) h2 = h3;
        }
        return h2;
    };
    return run_sharded(items, [&](size_t i) { return base[i].slicePitch; }, range);
}

int32_t dxb200_premultiply_alpha_device(const dxb200_image* src, size_t nimages, uint32_t flags, const dxb200_image* dst, void* stream)
{
    dxb_convert_params P;
    int32_t hr = plan_pmalpha(src, nimages, flags, dst, &P);
    if (hr != DXB_S_OK) return hr;
    DevScope scope;
    hr = scope.enter(src[0].pixels);
    if (hr != DXB_S_OK) return hr;
    return launch_pmalpha(P, src, dst, nimages, static_cast<cudaStream_t>(stream));
}

int32_t dxb200_premultiply_alpha(const dxb200_image* src, size_t nimages, uint32_t flags, const dxb200_image* dst)
{
    dxb_convert_params P;
    int32_t hr = plan_pmalpha(src, nimages, flags, dst, &P);
    if (hr != DXB_S_OK) return hr;
    BandSplit bands;
    split_bands(src, dst, nimages, 1, 1, false, false, bands);
    return run_sharded(bands.src.size(), [&](size_t i) { return bands.src[i].slicePitch + bands.dst[i].slicePitch; },
        [&](size_t lo, size_t hi)
        {
            return run_staged(bands.src.data() + lo, bands.dst.data() + lo, hi - lo,
                [&](const dxb200_image* ds, const dxb200_image* dd, size_t cnt, cudaStream_t st) { return launch_pmalpha(P, ds, dd, cnt, st); });
        });
}

// ---- ScaleMipMapsAlphaForCoverage ----------------------------------------------------------------
static int32_t plan_alpha_coverage(const dxb200_image* src, size_t n, const dxb200_image* dst)
{
    if (!src || !dst || !n) return DXB_E_INVALIDARG;
    const uint32_t fmt = src[0].format;
    if (is_compressed(fmt)) return DXB_E_NOT_SUPPORTED;                         // :3495-3497
    if (!is_supported_pixel_format(fmt)) return DXB_E_NOT_SUPPORTED;
    for (size_t i = 0; i < n; ++i)
    {
        if (!src[i].pixels || !dst[i].pixels) return DXB_E_POINTER;
        if (src[i].format != fmt || dst[i].format != fmt) return DXB_E_INVALIDARG;
        if (src[i].width != dst[i].width || src[i].height != dst[i].height || !src[i].width || !src[i].height) return DXB_E_INVALIDARG;
        if ((uint64_t)src[i].width * src[i].height > 0x7FFFFFFFull) return DXB_E_INVALIDARG;
    }
    return DXB_S_OK;
}

// device pointers; count = device scratch (8 bytes).  Mirrors CalculateAlphaCoverage / EstimateAlphaScaleForCoverage.
static int32_t alpha_coverage_device(const dxb200_image& img, float ref, float scale, unsigned long long* dCount, cudaStream_t st, float* coverage)
{
    *coverage = 0.0f;
    if (img.width < 2 || img.height < 2) return DXB_S_OK;                      // no 2x2 cell: the reference's loops do not run
    dxb_job j; memset(&j, 0, sizeof(j));
    j.src = img.pixels; j.srcPitch = img.rowPitch; j.width = (uint32_t)img.width; j.height = (uint32_t)img.height;
    DXB_CUDA(cudaMemsetAsync(dCount, 0, sizeof(unsigned long long), st));
    const uint64_t cells = (uint64_t)(img.width - 1) * (img.height - 1);
    const uint32_t grid = (uint32_t)std::max<uint64_t>(1, std::min<uint64_t>((cells + 255) / 256, (uint64_t)t_v.dev->gridRow * 8u));
    dxb_launch_alpha_coverage(grid, st, j, img.format, scale, ref, dCount);
    int32_t hr = check_launch("k_alpha_coverage");
    if (hr != DXB_S_OK) return hr;
    unsigned long long hCount = 0;
    DXB_CUDA(cudaMemcpyAsync(&hCount, dCount, sizeof(hCount), cudaMemcpyDeviceToHost, st));
    DXB_CUDA(cudaStreamSynchronize(st));
    const float cscale = static_cast<float>((img.width - 1) * (img.height - 1) * 8 * 8);          // :300-304
    if (cscale > 0.0f) *coverage = static_cast<float>(hCount) / cscale;
    return DXB_S_OK;
}

static int32_t scale_alpha_for_coverage_device(const dxb200_image* src, size_t n, float ref, const dxb200_image* dst, cudaStream_t st)
{
    unsigned long long* dCount = nullptr;
    DXB_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&dCount), sizeof(unsigned long long), st));
    float target = 0.0f;
    int32_t hr = alpha_coverage_device(src[0], ref, 1.0f, dCount, st, &target);
    // base level: plain copy (:3511-3530)
    if (hr == DXB_S_OK)
        hr = cuda_hr(cudaMemcpy2DAsync(dst[0].pixels, dst[0].rowPitch, src[0].pixels, src[0].rowPitch, std::min(src[0].rowPitch, dst[0].rowPitch),
                                       src[0].slicePitch / std::max<size_t>(src[0].rowPitch, 1), cudaMemcpyDeviceToDevice, st), "copy base level");
    for (size_t l = 1; l < n && hr == DXB_S_OK; ++l)
    {
        // EstimateAlphaScaleForCoverage (:310-355): bisection on [0, 4], at most 10 coverage evaluations
        float lo = 0.0f, hi = 4.0f, scale = 1.0f;
        for (int it = 0; it < 10 && hr == DXB_S_OK; ++it)
        {
            float cov = 0.0f;
            hr = alpha_coverage_device(src[l], ref, scale, dCount, st, &cov);
            if (hr != DXB_S_OK) break;
            if (cov < target) lo = scale;
            else if (cov > target) hi = scale;
            else break;
            scale = (lo + hi) * 0.5f;
        }
        if (hr != DXB_S_OK) break;
        dxb_job j; memset(&j, 0, sizeof(j));
        j.src = src[l].pixels; j.dst = dst[l].pixels; j.srcPitch = src[l].rowPitch; j.dstPitch = dst[l].rowPitch;
        j.width = (uint32_t)src[l].width; j.height = (uint32_t)src[l].height;
        const uint64_t px = (uint64_t)j.width * j.height;
        const uint32_t grid = (uint32_t)std::max<uint64_t>(1, std::min<uint64_t>((px + 255) / 256, (uint64_t)t_v.dev->gridRow * 8u));
        dxb_launch_scale_alpha(grid, st, j, src[l].format, scale);
        hr = check_launch("k_scale_alpha");
    }
    cudaFreeAsync(dCount, st);
    return hr;
}

int32_t dxb200_scale_mipmaps_alpha_for_coverage_device(const dxb200_image* src, size_t nlevels, float alphaReference, const dxb200_image* dst, void* stream)
{
    int32_t hr = plan_alpha_coverage(src, nlevels, dst);
    if (hr != DXB_S_OK) return hr;
    DevScope scope;
    hr = scope.enter(src[0].pixels);
    if (hr != DXB_S_OK) return hr;
    return scale_alpha_for_coverage_device(src, nlevels, alphaReference, dst, static_cast<cudaStream_t>(stream));
}

int32_t dxb200_scale_mipmaps_alpha_for_coverage(const dxb200_image* src, size_t nlevels, float alphaReference, const dxb200_image* dst)
{
    int32_t hr = plan_alpha_coverage(src, nlevels, dst);
    if (hr != DXB_S_OK) return hr;
    std::vector<Device*> devs;
    hr = device_list(&devs);
    if (hr != DXB_S_OK) return hr;
    HostScope scope;
    hr = scope.enter(devs[0]);
    if (hr != DXB_S_OK) return hr;
    cudaStream_t st = t_v.lane->streams[0];
    size_t bytes = 0;
    for (size_t l = 0; l < nlevels; ++l) bytes += 2 * ((src[l].slicePitch + 255) & ~size_t(255));
    hr = ensure_buffer(&t_v.lane->dIn[0], &t_v.lane->dInCap[0], bytes);
    if (hr != DXB_S_OK) return hr;
    std::vector<dxb200_image> ds(src, src + nlevels), dd(dst, dst + nlevels);
    size_t off = 0;
    for (size_t l = 0; l < nlevels && hr == DXB_S_OK; ++l)
    {
        ds[l].pixels = static_cast<uint8_t*>(t_v.lane->dIn[0]) + off; off += (src[l].slicePitch + 255) & ~size_t(255);
        dd[l].pixels = static_cast<uint8_t*>(t_v.lane->dIn[0]) + off; off += (src[l].slicePitch + 255) & ~size_t(255);
        dd[l].rowPitch = src[l].rowPitch; dd[l].slicePitch = src[l].slicePitch;          // device copy uses the source layout
        hr = cuda_hr(cudaMemcpyAsync(ds[l].pixels, src[l].pixels, src[l].slicePitch, cudaMemcpyHostToDevice, st), "H2D");
    }
    if (hr == DXB_S_OK) hr = scale_alpha_for_coverage_device(ds.data(), nlevels, alphaReference, dd.data(), st);
    for (size_t l = 0; l < nlevels && hr == DXB_S_OK; ++l)
        hr = cuda_hr(cudaMemcpy2DAsync(dst[l].pixels, dst[l].rowPitch, dd[l].pixels, dd[l].rowPitch, std::min(dst[l].rowPitch, dd[l].rowPitch),
                                       src[l].slicePitch / std::max<size_t>(src[l].rowPitch, 1), cudaMemcpyDeviceToHost, st), "D2H");
    if (hr == DXB_S_OK) hr = cuda_hr(cudaStreamSynchronize(st), "alpha coverage sync");
    return hr;
}

int32_t dxb200_resize_device(const dxb200_image* src, size_t nimages, uint32_t filter, const dxb200_image* dst, void* stream)
{
    uint32_t mode = 0;
    int32_t hr = plan_resize(src, nimages, filter, dst, &mode);
    if (hr != DXB_S_OK) return hr;
    DevScope scope;
    hr = scope.enter(src[0].pixels);
    if (hr != DXB_S_OK) return hr;
    // a resize is a two-"level" chain per item whose second level has an arbitrary size
    std::vector<dxb200_image> pairs(2 * nimages);
    for (size_t i = 0; i < nimages; ++i) { pairs[2 * i] = src[i]; pairs[2 * i + 1] = dst[i]; }
    return launch_mips(pairs.data(), nimages, 2, filter, mode, static_cast<cudaStream_t>(stream));
}

static int32_t resize_host_range(const dxb200_image* src, const dxb200_image* dst, size_t lo, size_t hi, uint32_t filter, uint32_t mode)
{
    const size_t CHUNK = size_t(1) << 30;
    cudaStream_t st = t_v.lane->streams[0];
    int32_t hr = DXB_S_OK;
    size_t it = lo;
    while (it < hi && hr == DXB_S_OK)
    {
        size_t bytes = 0, k = it;
        while (k < hi)
        {
            const size_t b = ((src[k].slicePitch + 255) & ~size_t(255)) + ((dst[k].slicePitch + 255) & ~size_t(255));
            if (k > it && bytes + b > CHUNK) break;
            bytes += b; ++k;
        }
        hr = ensure_buffer(&t_v.lane->dIn[0], &t_v.lane->dInCap[0], bytes); if (hr) break;
        std::vector<dxb200_image> pairs(2 * (k - it));
        size_t off = 0;
        for (size_t i = it; i < k && hr == DXB_S_OK; ++i)
        {
            dxb200_image& s = pairs[2 * (i - it)]; dxb200_image& d = pairs[2 * (i - it) + 1];
            s = src[i]; d = dst[i];
            s.pixels = static_cast<uint8_t*>(t_v.lane->dIn[0]) + off; off += (s.slicePitch + 255) & ~size_t(255);
            d.pixels = static_cast<uint8_t*>(t_v.lane->dIn[0]) + off; off += (d.slicePitch + 255) & ~size_t(255);
            hr = cuda_hr(cudaMemcpyAsync(s.pixels, src[i].pixels, s.slicePitch, cudaMemcpyHostToDevice, st), "H2D");
        }
        if (hr) break;
        hr = launch_mips(pairs.data(), k - it, 2, filter, mode, st); if (hr) break;
        for (size_t i = it; i < k && hr == DXB_S_OK; ++i)
            hr = cuda_hr(cudaMemcpyAsync(dst[i].pixels, pairs[2 * (i - it) + 1].pixels, dst[i].slicePitch, cudaMemcpyDeviceToHost, st), "D2H");
        if (hr) break;
        hr = cuda_hr(cudaStreamSynchronize(st), "resize sync");
        it = k;
    }
    return hr;
}

int32_t dxb200_resize(const dxb200_image* src, size_t nimages, uint32_t filter, const dxb200_image* dst)
{
    uint32_t mode = 0;
    int32_t hr = plan_resize(src, nimages, filter, dst, &mode);
    if (hr != DXB_S_OK) return hr;
    return run_sharded(nimages, [&](size_t i) { return src[i].slicePitch + dst[i].slicePitch; },
        [&](size_t lo, size_t hi) { return resize_host_range(src, dst, lo, hi, filter, mode); });
}

} // extern "C"

// ---- ComputeMSE (DirectXTexMisc.cpp:388-468) and the IsAlphaAllOpaque scan (DirectXTexImage.cpp:800-852) ------------------------
// dxb_analyze.cuh states the arithmetic and the fixed fp64 reduction tree; here: validation, chunk bookkeeping, staging.
#include "dxb_analyze.cuh"

namespace {

// IsValid (DirectXTex.inl:57-60); every valid format this backend does not implement (typeless, planar, palettized, video, ...)
// is HRESULT_E_NOT_SUPPORTED (:395-407: no CPU fallback)
int32_t check_analyze_format(uint32_t f)
{
    if (f < 1u || f > 191u) return DXB_E_INVALIDARG;
    return (is_compressed(f) || is_supported_pixel_format(f)) ? DXB_S_OK : DXB_E_NOT_SUPPORTED;
}

uint32_t tile_rows(const dxb200_image& im) { return (uint32_t)((im.height + 3) / 4); }
uint32_t chunks_per_row(const dxb200_image& im) { return (uint32_t)(((im.width + 3) / 4 + DXB_AN_TILES - 1) / DXB_AN_TILES); }

int32_t plan_mse(const dxb200_image* a, const dxb200_image* b, size_t n)
{
    if (!a || !b || !n) return DXB_E_INVALIDARG;
    uint64_t chunks = 0;
    for (size_t i = 0; i < n; ++i)
    {
        if (!a[i].pixels || !b[i].pixels) return DXB_E_POINTER;
        if (a[i].width != b[i].width || a[i].height != b[i].height) return DXB_E_INVALIDARG;
        const int32_t ha = check_analyze_format(a[i].format), hb = check_analyze_format(b[i].format);
        if (ha == DXB_E_INVALIDARG || hb == DXB_E_INVALIDARG) return DXB_E_INVALIDARG;
        if (ha != DXB_S_OK || hb != DXB_S_OK) return DXB_E_NOT_SUPPORTED;
        if (!a[i].width || !a[i].height || a[i].width > 0xFFFFFFFFull || a[i].height > 0xFFFFFFFFull) return DXB_E_INVALIDARG;
        chunks += (uint64_t)tile_rows(a[i]) * chunks_per_row(a[i]);
        if (chunks > 0x7FFFFFFFull) return DXB_E_INVALIDARG;
    }
    return DXB_S_OK;
}

// enqueue the chunk kernels for pairs whose pixels live on the device: pair i writes its partials (4 doubles per chunk) from
// partials + 4 * firstPartial[i] on.  Pairs are grouped by the kind of their sides (BC or not), one launch per kind.
int32_t launch_mse(const dxb200_image* a, const dxb200_image* b, size_t n, uint32_t flags, const uint32_t* firstPartial, double* partials, cudaStream_t stream)
{
    std::vector<dxb_pair_job> kinds[3];
    for (size_t i = 0; i < n; ++i)
    {
        dxb_pair_job j; memset(&j, 0, sizeof(j));
        const bool bcA = is_compressed(a[i].format), bcB = is_compressed(b[i].format);
        const bool swap = !bcA && bcB;                           // a lone BC side goes first
        const dxb200_image& x = swap ? b[i] : a[i];
        const dxb200_image& y = swap ? a[i] : b[i];
        uint32_t f = (flags & DXB_CMSE_MASK) | dxb_cmse_implied(a[i].format, false) | dxb_cmse_implied(b[i].format, true);
        if (swap) f = dxb_cmse_swap(f);
        j.a = x.pixels; j.b = y.pixels; j.pitchA = x.rowPitch; j.pitchB = y.rowPitch;
        j.fmtA = x.format; j.fmtB = y.format; j.flags = f;
        j.width = (uint32_t)x.width; j.height = (uint32_t)x.height;
        j.nbx = (j.width + 3) / 4; j.cpr = chunks_per_row(x);
        j.firstPartial = firstPartial[i];
        kinds[(bcA && bcB) ? 2 : (bcA || bcB) ? 1 : 0].push_back(j);
    }
    int32_t hr = DXB_S_OK;
    for (auto& jobs : kinds)
    {
        if (jobs.empty() || hr != DXB_S_OK) continue;
        uint64_t total = 0;
        for (auto& j : jobs) { j.firstUnit = (uint32_t)total; total += (uint64_t)((j.height + 3) / 4) * j.cpr; }
        DeviceJobs<dxb_pair_job> dj;
        hr = dj.upload(jobs, stream);
        if (hr != DXB_S_OK) return hr;
        const uint32_t grid = (uint32_t)std::max<uint64_t>(1, std::min<uint64_t>(total, (uint64_t)t_v.dev->gridRow));
        dxb_launch_compute_mse(grid, stream, dj.d, jobs[0], (uint32_t)jobs.size(), (uint32_t)total, partials);
        hr = check_launch("k_compute_mse");
        dj.release();
    }
    return hr;
}

int32_t plan_opaque(const dxb200_image* images, size_t n)
{
    if (!images || !n) return DXB_E_INVALIDARG;
    const uint32_t fmt = images[0].format;
    for (size_t i = 0; i < n; ++i)
    {
        if (!images[i].pixels) return DXB_E_POINTER;
        if (images[i].format != fmt) return DXB_E_INVALIDARG;
        if (!images[i].width || !images[i].height || images[i].width > 0xFFFFFFFFull || images[i].height > 0xFFFFFFFFull) return DXB_E_INVALIDARG;
    }
    uint64_t chunks = 0;
    for (size_t i = 0; i < n; ++i) chunks += (uint64_t)tile_rows(images[i]) * chunks_per_row(images[i]);
    if (chunks > 0x7FFFFFFFull) return DXB_E_INVALIDARG;
    return check_analyze_format(fmt);
}

// BC formats without an alpha scan (BC4 / BC5 / BC6H): "not opaque" for every image (IsAlphaAllOpaqueBC :569-572)
bool opaque_trivially_false(uint32_t fmt) { return is_compressed(fmt) && !dxb_opaque_bc_scanned(fmt); }

// enqueue the scan of device images; *opaque (device) must hold 1 before, is set to 0 by a tile with a pixel below the threshold
int32_t launch_opaque(const dxb200_image* images, size_t n, int32_t* opaque, cudaStream_t stream)
{
    std::vector<dxb_pair_job> jobs(n);
    uint64_t total = 0;
    for (size_t i = 0; i < n; ++i)
    {
        dxb_pair_job& j = jobs[i]; memset(&j, 0, sizeof(j));
        j.a = images[i].pixels; j.pitchA = images[i].rowPitch; j.fmtA = images[i].format;
        j.width = (uint32_t)images[i].width; j.height = (uint32_t)images[i].height;
        j.nbx = (j.width + 3) / 4; j.cpr = chunks_per_row(images[i]);
        j.firstUnit = (uint32_t)total; total += (uint64_t)tile_rows(images[i]) * j.cpr;
    }
    DeviceJobs<dxb_pair_job> dj;
    int32_t hr = dj.upload(jobs, stream);
    if (hr != DXB_S_OK) return hr;
    const uint32_t grid = (uint32_t)std::max<uint64_t>(1, std::min<uint64_t>(total, (uint64_t)t_v.dev->gridRow));
    dxb_launch_alpha_opaque(grid, stream, dj.d, jobs[0], (uint32_t)n, (uint32_t)total, opaque);
    hr = check_launch("k_alpha_opaque");
    dj.release();
    return hr;
}

} // namespace

extern "C" {

int32_t dxb200_compute_mse_device(const dxb200_image* a, const dxb200_image* b, size_t n, uint32_t flags, float* out, void* stream)
{
    int32_t hr = plan_mse(a, b, n);
    if (hr != DXB_S_OK) return hr;
    if (!out) return DXB_E_POINTER;
    DevScope scope;
    hr = scope.enter(a[0].pixels);
    if (hr != DXB_S_OK) return hr;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    std::vector<uint32_t> first(n);
    std::vector<dxb_mse_final> fin(n);
    uint32_t chunks = 0;
    for (size_t i = 0; i < n; ++i)
    {
        const uint32_t c = tile_rows(a[i]) * chunks_per_row(a[i]);
        first[i] = chunks;
        fin[i].pixels = (uint64_t)a[i].width * a[i].height; fin[i].firstPartial = chunks; fin[i].nchunks = c;
        chunks += c;
    }
    double* dPart = nullptr;
    dxb_mse_final* dFin = nullptr;
    DXB_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&dPart), (size_t)chunks * 4 * sizeof(double), st));
    hr = cuda_hr(cudaMallocAsync(reinterpret_cast<void**>(&dFin), n * sizeof(dxb_mse_final), st), "cudaMallocAsync");
    if (hr == DXB_S_OK) hr = cuda_hr(cudaMemcpyAsync(dFin, fin.data(), n * sizeof(dxb_mse_final), cudaMemcpyHostToDevice, st), "H2D");
    if (hr == DXB_S_OK) hr = launch_mse(a, b, n, flags, first.data(), dPart, st);
    if (hr == DXB_S_OK)
    {
        dxb_launch_mse_finish(st, dFin, (uint32_t)n, dPart, out);
        hr = check_launch("k_mse_finish");
    }
    cudaFreeAsync(dPart, st);
    if (dFin) cudaFreeAsync(dFin, st);
    return hr;
}

int32_t dxb200_compute_mse(const dxb200_image* a, const dxb200_image* b, size_t n, uint32_t flags, float* mse, float* mseV)
{
    int32_t hr = plan_mse(a, b, n);
    if (hr != DXB_S_OK) return hr;
    if (!mse) return DXB_E_POINTER;
    // bands of whole tile rows (4 pixel rows, 1 block row); their chunk partials land where a whole-image launch puts them
    std::vector<dxb200_image> ba, bb;
    std::vector<size_t> bandImage;
    for (size_t i = 0; i < n; ++i)
    {
        BandSplit s;
        split_bands(a + i, b + i, 1, is_compressed(a[i].format) ? 1 : 4, is_compressed(b[i].format) ? 1 : 4, is_compressed(a[i].format), is_compressed(b[i].format), s);
        ba.insert(ba.end(), s.src.begin(), s.src.end()); bb.insert(bb.end(), s.dst.begin(), s.dst.end());
        bandImage.insert(bandImage.end(), s.src.size(), i);
    }
    std::vector<uint32_t> first(ba.size() + 1, 0);
    for (size_t k = 0; k < ba.size(); ++k) first[k + 1] = first[k] + tile_rows(ba[k]) * chunks_per_row(ba[k]);
    std::vector<double> partials((size_t)first.back() * 4);
    hr = run_sharded(ba.size(), [&](size_t k) { return ba[k].slicePitch + bb[k].slicePitch; },
        [&](size_t lo, size_t hi) -> int32_t
        {
            const size_t count = (size_t)(first[hi] - first[lo]) * 4;
            double* dPart = nullptr;
            DXB_CUDA(cudaMalloc(reinterpret_cast<void**>(&dPart), std::max<size_t>(count, 1) * sizeof(double)));
            size_t next = lo;
            int32_t h2 = run_staged(ba.data() + lo, bb.data() + lo, hi - lo,
                [&](const dxb200_image* da, const dxb200_image* db, size_t cnt, cudaStream_t st)
                {
                    std::vector<uint32_t> fp(cnt);
                    for (size_t m = 0; m < cnt; ++m) fp[m] = first[next + m] - first[lo];
                    next += cnt;
                    return launch_mse(da, db, cnt, flags, fp.data(), dPart, st);
                }, nullptr, nullptr, true);
            if (h2 == DXB_S_OK) h2 = cuda_hr(cudaMemcpy(partials.data() + (size_t)first[lo] * 4, dPart, count * sizeof(double), cudaMemcpyDeviceToHost), "D2H partials");
            cudaFree(dPart);
            return h2;
        });
    if (hr != DXB_S_OK) return hr;
    // the image level of the tree, on the host (the same IEEE fp64 additions as k_mse_finish)
    size_t k = 0;
    for (size_t i = 0; i < n; ++i)
    {
        const uint32_t p0 = first[k];
        while (k < ba.size() && bandImage[k] == i) ++k;
        float o[5];
        dxb_cmse_finish(partials.data() + (size_t)p0 * 4, first[k] - p0, (uint64_t)a[i].width * a[i].height, o);
        mse[i] = o[0];
        if (mseV) memcpy(mseV + 4 * i, o + 1, 4 * sizeof(float));
    }
    return DXB_S_OK;
}

int32_t dxb200_is_alpha_all_opaque_device(const dxb200_image* images, size_t n, int32_t* opaque, void* stream)
{
    int32_t hr = plan_opaque(images, n);
    if (hr != DXB_S_OK) return hr;
    if (!opaque) return DXB_E_POINTER;
    DevScope scope;
    hr = scope.enter(images[0].pixels);
    if (hr != DXB_S_OK) return hr;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const bool none = opaque_trivially_false(images[0].format);
    dxb_launch_set_i32(st, opaque, none ? 0 : 1);
    hr = check_launch("k_set_i32");
    if (hr == DXB_S_OK && !none) hr = launch_opaque(images, n, opaque, st);
    return hr;
}

int32_t dxb200_is_alpha_all_opaque(const dxb200_image* images, size_t n, int32_t* opaque)
{
    int32_t hr = plan_opaque(images, n);
    if (hr != DXB_S_OK) return hr;
    if (!opaque) return DXB_E_POINTER;
    if (opaque_trivially_false(images[0].format)) { *opaque = 0; return DXB_S_OK; }
    const bool bc = is_compressed(images[0].format);
    BandSplit bands;
    split_bands(images, images, n, bc ? 1 : 4, bc ? 1 : 4, bc, bc, bands);
    std::atomic<int32_t> result{1};
    hr = run_sharded(bands.src.size(), [&](size_t k) { return bands.src[k].slicePitch; },
        [&](size_t lo, size_t hi) -> int32_t
        {
            int32_t* dFlag = nullptr;
            DXB_CUDA(cudaMalloc(reinterpret_cast<void**>(&dFlag), sizeof(int32_t)));
            int32_t h2 = DXB_S_OK, found = 1;
            dxb_launch_set_i32(t_v.lane->streams[0], dFlag, 1);
            h2 = check_launch("k_set_i32");
            if (h2 == DXB_S_OK) h2 = cuda_hr(cudaStreamSynchronize(t_v.lane->streams[0]), "flag init");
            if (h2 == DXB_S_OK)
                h2 = run_staged(bands.src.data() + lo, nullptr, hi - lo,
                    [&](const dxb200_image* ds, const dxb200_image*, size_t cnt, cudaStream_t st) { return launch_opaque(ds, cnt, dFlag, st); });
            if (h2 == DXB_S_OK) h2 = cuda_hr(cudaMemcpy(&found, dFlag, sizeof(int32_t), cudaMemcpyDeviceToHost), "D2H flag");
            if (h2 == DXB_S_OK && found == 0) result.store(0);
            cudaFree(dFlag);
            return h2;
        });
    if (hr != DXB_S_OK) return hr;
    *opaque = result.load();
    return DXB_S_OK;
}

} // extern "C"
