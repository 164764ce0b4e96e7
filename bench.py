#!/usr/bin/env python
"""bench.py — benchmarks of the B200 DirectXTex backend on the BASELINE.json configurations.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config c2|c3|c4|c5] [--impl reference] [--batch B] [--dump-outputs DIR]

Default (= the headline, BASELINE.json `metric`, configs[1]):  Mtexels/s BC7 encode, 4096x4096 RGBA32F -> BC7_UNORM,
TEX_COMPRESS_DEFAULT.  A step = one pass of the hot path over a batch of B (default 32) 4096^2 images per GPU, so that the
K = 20 steps the driver asks for keep the GPU busy for seconds (sustained clocks, dozens of clock samples), not 64 ms.
One process per GPU (torchrun), image-per-GPU sharding (weak scaling); at N > 1 the packed blocks are all-gathered over NCCL
on a side stream that overlaps the next step's kernel (double-buffered output).

Other legs (`--config`): c3 = 2048^2 RGBA16F -> 12-level CUBIC mip chain -> BC6H_UF16 of every level; c4 = 1024 x 1024^2 RGBA8
-> 11-level BOX chain -> BC3, the batch sharded over the GPUs (strong scaling), one all-gather of the packed blocks;
c5 = 8192^2 R8 -> BC4 and Convert R8 -> R32F -> R8 (the HBM-bound row kernel).

Prints ONE JSON line (rank 0):  `value` = device-resident throughput (inputs in HBM), `e2e` = the same metric through the
host-pointer C ABI with pinned host buffers (H2D + D2H inside the timed region), `roofline` = the dominant kernel against the
measured HBM peak, `cpu_baseline` = the UNMODIFIED reference (oracle/_ref) on the host cores on a bounded sample, `parity` =
the result of this very run checked against the reference (SURVEY 8(d): parity checks run with every measurement).
`--impl reference` times the reference's own CPU implementation on a bounded sample per step.  `cpu_baseline` and `parity` are
null where the reference build (oracle/Makefile) is absent.
`--dump-outputs DIR` writes what the last timed step computed (rank 0), as DIR/<name>.npy in float32: every output buffer of
the step, or a fixed seeded sample of its 16-byte rows where the outputs together exceed 60 MiB.  The inputs are seeded, so two
builds run with the same arguments can be compared output for output.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)


def peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return {"hbm_gbs": 6650.0}, "fallback (B200_PROFILING.md)"


def ncu_metric(path, key):
    """value of `key` from a committed ncu summary under profiles/ (None if absent)"""
    try:
        for line in open(os.path.join(ROOT, "profiles", path)):
            parts = line.split()
            if parts and parts[0] == key:
                v = float(parts[-1])
                if len(parts) >= 3 and parts[1].lower().endswith("byte"):          # ncu scales byte counts: normalise to Mbyte
                    v *= {"byte": 1e-6, "kbyte": 1e-3, "mbyte": 1.0, "gbyte": 1e3}.get(parts[1].lower(), 1.0)
                return v
    except Exception:
        pass
    return None


class ClockSampler:
    """samples nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)"""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = [float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 7 for i in range(4) if r[3 + i].lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def host_threads():
    return len(os.sched_getaffinity(0))


def load_ref(threads=None):
    """the oracle (test infrastructure): only the cpu_baseline / parity / --impl reference legs use it"""
    from tests import oracle_lib
    ref = oracle_lib.load_ref()
    # torchrun exports OMP_NUM_THREADS=1: the reference arm must use all the host threads it can
    os.environ.setdefault("OMP_PROC_BIND", "spread")
    ref.L.ref_omp_set_threads(threads or host_threads())
    return ref


# =====================================================================================================================
# Workloads.  Every workload provides:
#   setup(ctx)          device-resident inputs/outputs for this rank
#   step(ctx, i)        one pass of the hot path on device-resident data (enqueue only); returns the (start, end) CUDA events
#                       around the dominant kernel's C-ABI call
#   gather_bytes        bytes of packed blocks this rank contributes to the end-of-step all-gather (0 = none)
#   e2e_setup / e2e_step  the same pass through the host-pointer C ABI (pinned host memory)
#   reference_step(ref) one bounded sample of the reference's own CPU path; returns (units, seconds, description)
#   parity(ctx, ref)    dict
class Ctx:
    pass


def _img(capi, w, h, fmt, row, sl, ptr):
    return capi.Image(w, h, fmt, row, sl, ptr)


class C2:
    """BASELINE configs[1]: 4096x4096 RGBA32F -> BC7_UNORM, TEX_COMPRESS_DEFAULT"""
    name = "c2"
    metric = "Mtexels/s BC7 encode (4096^2 RGBA, default quality)"
    dtype = "f32"
    scaling = "weak"
    W = H = 4096
    SRC, DST = 2, 98
    kernel = "k_compress_bc7_tma"     # batches: the TMA-fed persistent kernel (DXB200_OPT_BC7_FEED = 4, automatic); a single image: k_compress_bc7
    bound_note = ("BC7 mode/partition search is issue-bound, not HBM-bound (SURVEY 8(d)); DRAM traffic = algorithmic bytes; "
                  "issue-slot utilisation and warp-instructions per block: profiles/r02_ncu_k_compress_bc7.txt")
    ncu_file = "r02_ncu_k_compress_bc7_tma.txt"
    small_sample = {"side": 64}          # the 1-thread rate of the reference is measured on this smaller sample

    def __init__(self, args, world):
        self.B = args.batch or 32
        self.world = world
        if self.B == 1:                    # a single image takes the direct kernel under the automatic feed
            self.kernel, self.ncu_file = "k_compress_bc7", "r02_ncu_k_compress_bc7.txt"

    def workload(self):
        return ("4096x4096 RGBA32F -> BC7_UNORM, TEX_COMPRESS_DEFAULT (BASELINE.json configs[1]); a step = a batch of %d such images per GPU "
                "(image-per-GPU sharding, weak scaling), packed blocks all-gathered over NCCL at N>1 (overlapped with the next step)" % self.B)

    def units_per_step(self):           # texels per rank per step
        return self.B * self.W * self.H

    def algo_bytes(self):               # SURVEY 8(d): 17 B/texel = 285,212,672 B per image
        return self.B * (self.W * self.H * 16 + (self.W // 4) * (self.H // 4) * 16)

    def setup(self, ctx):
        torch, capi, F, synth = ctx.torch, ctx.capi, ctx.F, ctx.synth
        self.img = synth.c2_rgba32f(self.W, self.H, seed=synth.SEED + ctx.rank)
        self.row_in, self.slice_in = F.compute_pitch(self.SRC, self.W, self.H)
        self.row_out, self.slice_out = F.compute_pitch(self.DST, self.W, self.H)
        base = torch.from_numpy(self.img.reshape(self.H, self.W * 4)).cuda()
        # batch entry b = the base image rolled by 4*b rows and 4*b pixels: distinct block content, generated on the device
        self.d_in = torch.empty((self.B, self.H, self.W * 4), dtype=torch.float32, device="cuda")
        for b in range(self.B):
            self.d_in[b] = torch.roll(base, shifts=(4 * b, 16 * b), dims=(0, 1))
        self.d_out = [torch.zeros(self.B * self.slice_out, dtype=torch.uint8, device="cuda") for _ in range(2)]
        self.src = capi.images([_img(capi, self.W, self.H, self.SRC, self.row_in, self.slice_in, self.d_in[b].data_ptr()) for b in range(self.B)])
        self.dst = [capi.images([_img(capi, self.W, self.H, self.DST, self.row_out, self.slice_out, o.data_ptr() + b * self.slice_out) for b in range(self.B)])
                    for o in self.d_out]
        self.gather_bytes = self.B * self.slice_out

    def step(self, ctx, i):
        e0, e1 = ctx.event(), ctx.event()
        e0.record()
        hr = ctx.capi.lib.dxb200_compress_device(self.src, self.B, self.DST, 0, 0.5, 1.0, self.dst[i & 1], ctx.stream_ptr)
        e1.record()
        if hr != 0:
            raise ctx.capi.DxTexError(hr, "dxb200_compress_device")
        return e0, e1, self.d_out[i & 1]

    def outputs(self, ctx):
        return {"bc7_blocks": self.d_out[ctx.last_step & 1]}

    def alternates(self, ctx):
        """the same batch through the other feed of the BC7 kernel (dxb200_set_option(DXB200_OPT_BC7_FEED, ..)): ms per step, output equal.
        The default (4 = automatic) feeds batches by TMA tensor-map tile loads (k_compress_bc7_tma) and single images by direct loads."""
        capi, torch = ctx.capi, ctx.torch
        feed = capi.lib.dxb200_get_option(capi.OPT_BC7_FEED)
        used_tma = feed in (1, 2, 3) or (feed == 4 and self.B > 1)
        other, name = (0, "k_compress_bc7 (direct loads)") if used_tma else (1, "k_compress_bc7_tma")
        want = self.d_out[ctx.last_step & 1].clone()
        t0 = capi.tma_launch_count()
        capi.lib.dxb200_set_option(capi.OPT_BC7_FEED, other)
        try:
            for _ in range(2):
                self.step(ctx, ctx.last_step)
            a, b = ctx.event(), ctx.event()
            a.record()
            for _ in range(3):
                self.step(ctx, ctx.last_step)
            b.record()
            torch.cuda.synchronize()
        finally:
            capi.lib.dxb200_set_option(capi.OPT_BC7_FEED, feed)
        same = bool(torch.equal(want, self.d_out[ctx.last_step & 1]))
        return {name: {"ms_per_step": a.elapsed_time(b) / 3.0, "tma_launches": capi.tma_launch_count() - t0, "output_equal": same,
                       "what": "the same batch with DXB200_OPT_BC7_FEED = %d instead of the default %d" % (other, feed)}}

    def e2e_setup(self, ctx):
        capi = ctx.capi
        self.Be = min(self.B, 8)
        self.pin_in = capi.lib.dxb200_host_alloc(self.Be * self.slice_in)
        self.pin_out = capi.lib.dxb200_host_alloc(self.Be * self.slice_out)
        assert self.pin_in and self.pin_out
        host = self.d_in[:self.Be].cpu().numpy()
        C.memmove(self.pin_in, host.ctypes.data, self.Be * self.slice_in)
        self.hsrc = capi.images([_img(capi, self.W, self.H, self.SRC, self.row_in, self.slice_in, self.pin_in + b * self.slice_in) for b in range(self.Be)])
        self.hdst = capi.images([_img(capi, self.W, self.H, self.DST, self.row_out, self.slice_out, self.pin_out + b * self.slice_out) for b in range(self.Be)])
        return {"units": self.Be * self.W * self.H, "h2d": self.Be * self.slice_in, "d2h": self.Be * self.slice_out,
                "api": "dxb200_compress (array of %d host images, pinned)" % self.Be}

    def e2e_step(self, ctx):
        hr = ctx.capi.lib.dxb200_compress(self.hsrc, self.Be, self.DST, 0, 0.5, 1.0, self.hdst)      # synchronous: returns after D2H
        if hr != 0:
            raise ctx.capi.DxTexError(hr, "dxb200_compress")

    def e2e_check(self, ctx):
        host = np.ctypeslib.as_array((C.c_uint8 * (self.Be * self.slice_out)).from_address(self.pin_out))
        dev = self.d_out[(ctx.last_step) & 1][: self.Be * self.slice_out].cpu().numpy()
        assert np.array_equal(host, dev), "e2e and device-resident outputs differ"
        ctx.capi.lib.dxb200_host_free(self.pin_in)
        ctx.capi.lib.dxb200_host_free(self.pin_out)

    # ---- reference side
    def _crop(self, side):
        y0 = (self.H - side) // 2
        return np.ascontiguousarray(self.img[y0:y0 + side, y0:y0 + side]), y0

    def reference_step(self, ref, side=256):
        if not hasattr(self, "img"):
            from directxtex_b200 import synth
            self.img = synth.c2_rgba32f(self.W, self.H)
        crop, _ = self._crop(side)
        sec = ref.compress_seconds(crop, side, side, self.SRC, self.DST, 0, 0.5, parallel=True)
        return side * side, sec, "centre %dx%d crop of the 4096x4096 C2 image, reference Compress(BC7_UNORM, DEFAULT|PARALLEL)" % (side, side)

    def parity(self, ctx, ref):
        """MSE of the GPU blocks of the centre 256^2 crop (first image of the batch) vs the reference encoder's on the same crop, both decoded
        by the reference decoder (ComputeMSE-style, 8-bit codes, RGBA)"""
        from tests import tolerance
        side = 256
        crop, y0 = self._crop(side)
        blocks = self.d_out[ctx.last_step & 1][: self.slice_out].cpu().numpy().reshape(self.H // 4, self.W // 4, 16)
        mine = np.ascontiguousarray(blocks[y0 // 4:(y0 + side) // 4, y0 // 4:(y0 + side) // 4]).reshape(-1)
        hr, theirs = ref.compress(crop, side, side, self.SRC, self.DST, 0)
        assert hr == 0
        a, b = tolerance.bc7_block_sse(ref, mine, crop), tolerance.bc7_block_sse(ref, theirs, crop)
        n = side * side * 4
        return {"what": "centre 256x256 crop of image 0: RGBA MSE (8-bit codes) of the GPU blocks vs the reference encoder's blocks, both through the reference decoder",
                "mse_gpu": a.sum() / n, "mse_ref": b.sum() / n, "ratio": float(a.sum() / max(b.sum(), 1e-9)),
                "blocks_worse_than_2x_plus_16": float((a > 2 * b + 16).mean()), "contract": "ratio <= 1.02, < 1% of blocks worse", "ok": bool(a.sum() <= 1.02 * b.sum())}


class C3:
    """BASELINE configs[2]: 2048x2048 RGBA16F -> full CUBIC mip chain -> BC6H_UF16 of every level"""
    name = "c3"
    metric = "Mtexels/s GenerateMipMaps(CUBIC) + BC6H_UF16 encode of the chain (2048^2 RGBA16F)"
    dtype = "f16"
    scaling = "weak"
    W = H = 2048
    FMT, DST = 10, 95
    kernel = "k_compress_bc6h"
    bound_note = "BC6H mode/shape search is issue-bound; the CUBIC mip kernels of the same step are reported under `kernels`"
    ncu_file = "r02_ncu_k_compress_bc6h.txt"
    small_sample = {"side": 64}

    def __init__(self, args, world):
        self.B = args.batch or 32
        self.world = world

    def workload(self):
        return ("2048x2048 RGBA16F -> 12-level mip chain (TEX_FILTER_CUBIC) -> BC6H_UF16 of every level (BASELINE.json configs[2]); "
                "a step = %d such textures per GPU" % self.B)

    def setup(self, ctx):
        torch, capi, F, synth = ctx.torch, ctx.capi, ctx.F, ctx.synth
        self.img = synth.c3_rgba16f(self.W, self.H, seed=synth.SEED + ctx.rank)
        self.layout, self.chain_bytes = F.mip_chain_layout(self.FMT, self.W, self.H, 0)
        self.olayout, self.out_bytes = capi.texture_layout(self.DST, self.W, self.H, 1, len(self.layout))
        self.levels = len(self.layout)
        self.chain_texels = sum(lw * lh for (_, lw, lh, _, _) in self.layout)
        base = torch.from_numpy(self.img.reshape(self.H, self.W * 4).view(np.int16)).cuda()
        self.d_chain = torch.zeros((self.B, self.chain_bytes), dtype=torch.uint8, device="cuda")
        for b in range(self.B):
            lvl0 = torch.roll(base, shifts=(4 * b, 16 * b), dims=(0, 1)).contiguous().view(torch.uint8).reshape(-1)
            self.d_chain[b, : lvl0.numel()] = lvl0
        self.d_out = [torch.zeros(self.B * self.out_bytes, dtype=torch.uint8, device="cuda") for _ in range(2)]
        self.chain = capi.images([_img(capi, lw, lh, self.FMT, row, sl, self.d_chain[b].data_ptr() + off)
                                  for b in range(self.B) for (off, lw, lh, row, sl) in self.layout])
        self.dst = [capi.images([_img(capi, lw, lh, self.DST, row, sl, o.data_ptr() + b * self.out_bytes + off)
                                 for b in range(self.B) for (off, lw, lh, row, sl) in self.olayout]) for o in self.d_out]
        self.gather_bytes = self.B * self.out_bytes

    def units_per_step(self):
        return self.B * self.chain_texels

    def algo_bytes(self):               # BC6H kernel: 8 B in + 1 B out per chain texel
        return self.B * (self.chain_bytes + self.out_bytes)

    def step(self, ctx, i):
        lib = ctx.capi.lib
        m0, m1, e0, e1 = ctx.event(), ctx.event(), ctx.event(), ctx.event()
        m0.record()
        hr = lib.dxb200_generate_mipmaps_device(self.chain, self.B, self.levels, ctx.F.TEX_FILTER_CUBIC, ctx.stream_ptr)
        m1.record()
        if hr != 0:
            raise ctx.capi.DxTexError(hr, "dxb200_generate_mipmaps_device")
        e0.record()
        hr = lib.dxb200_compress_device(self.chain, self.B * self.levels, self.DST, 0, 0.5, 1.0, self.dst[i & 1], ctx.stream_ptr)
        e1.record()
        if hr != 0:
            raise ctx.capi.DxTexError(hr, "dxb200_compress_device")
        ctx.extra_events.setdefault("mips_cubic", []).append((m0, m1))
        return e0, e1, self.d_out[i & 1]

    def outputs(self, ctx):
        return {"mip_chain_rgba16f": self.d_chain.view(ctx.torch.float16), "bc6h_blocks": self.d_out[ctx.last_step & 1]}

    def e2e_setup(self, ctx):
        capi = ctx.capi
        self.Be = min(self.B, 4)
        self.pin_chain = capi.lib.dxb200_host_alloc(self.Be * self.chain_bytes)
        self.pin_out = capi.lib.dxb200_host_alloc(self.Be * self.out_bytes)
        host = self.d_chain[: self.Be].cpu().numpy()
        C.memmove(self.pin_chain, host.ctypes.data, self.Be * self.chain_bytes)
        self.hchain = capi.images([_img(capi, lw, lh, self.FMT, row, sl, self.pin_chain + b * self.chain_bytes + off)
                                   for b in range(self.Be) for (off, lw, lh, row, sl) in self.layout])
        self.hdst = capi.images([_img(capi, lw, lh, self.DST, row, sl, self.pin_out + b * self.out_bytes + off)
                                 for b in range(self.Be) for (off, lw, lh, row, sl) in self.olayout])
        lvl0 = self.layout[0][4]
        return {"units": self.Be * self.chain_texels, "h2d": self.Be * (lvl0 + self.chain_bytes), "d2h": self.Be * (self.chain_bytes - lvl0 + self.out_bytes),
                "api": "dxb200_generate_mipmaps + dxb200_compress (host pointers, pinned; the chain returns to the host in between, as with the reference API)"}

    def e2e_step(self, ctx):
        lib = ctx.capi.lib
        hr = lib.dxb200_generate_mipmaps(self.hchain, self.Be, self.levels, ctx.F.TEX_FILTER_CUBIC)
        if hr == 0:
            hr = lib.dxb200_compress(self.hchain, self.Be * self.levels, self.DST, 0, 0.5, 1.0, self.hdst)
        if hr != 0:
            raise ctx.capi.DxTexError(hr, "c3 e2e")

    def e2e_check(self, ctx):
        host = np.ctypeslib.as_array((C.c_uint8 * (self.Be * self.out_bytes)).from_address(self.pin_out))
        dev = self.d_out[ctx.last_step & 1][: self.Be * self.out_bytes].cpu().numpy()
        assert np.array_equal(host, dev), "e2e and device-resident outputs differ"
        ctx.capi.lib.dxb200_host_free(self.pin_chain)
        ctx.capi.lib.dxb200_host_free(self.pin_out)

    def reference_step(self, ref, side=256):
        from directxtex_b200 import formats as F, synth
        if not hasattr(self, "img"):
            self.img = synth.c3_rgba16f(self.W, self.H)
        crop = np.ascontiguousarray(self.img[:side, :side])
        t0 = time.perf_counter()
        hr, chain = ref.generate_mipmaps(crop, side, side, self.FMT, F.TEX_FILTER_CUBIC)
        assert hr == 0
        layout, _ = F.mip_chain_layout(self.FMT, side, side, 0)
        for (off, lw, lh, row, sl) in layout:
            hr, _b = ref.compress(chain[off:off + sl], lw, lh, self.FMT, self.DST, 0)
            assert hr == 0
        sec = time.perf_counter() - t0
        return sum(lw * lh for (_, lw, lh, _, _) in layout), sec, "top-left %dx%d crop of the C3 image: reference GenerateMipMaps(CUBIC) + Compress(BC6H_UF16, PARALLEL) of every level" % (side, side)

    def parity(self, ctx, ref):
        """the whole 2048^2 CUBIC chain of texture 0 bit-exact vs the reference; BC6H of the 256^2 level and of a 256^2 crop of level 0 vs the
        reference encoder in its own metric"""
        from directxtex_b200 import formats as F
        from tests import tolerance
        chain = self.d_chain[0].cpu().numpy()
        lvl0 = chain[: self.layout[0][4]]
        hr, want = ref.generate_mipmaps(lvl0, self.W, self.H, self.FMT, F.TEX_FILTER_CUBIC)
        exact = bool(hr == 0 and np.array_equal(chain, want))
        out = self.d_out[ctx.last_step & 1][: self.out_bytes].cpu().numpy()
        res = {"what": "texture 0: 12-level CUBIC chain memcmp vs reference GenerateMipMaps; BC6H of mip level 3 (256^2) vs the reference encoder, "
                       "error = squared half-bit-pattern differences (the reference encoder's metric)", "chain_bit_exact": exact}
        (off, lw, lh, row, sl), (ooff, _, _, _, osl) = self.layout[3], self.olayout[3]
        level = chain[off:off + sl]
        f32 = level.view(np.float16).reshape(lh, lw, 4).astype(np.float32)
        hr, theirs = ref.compress(level, lw, lh, self.FMT, self.DST, 0)
        assert hr == 0
        a, _, amax = tolerance.bc6h_block_errors(ref, out[ooff:ooff + osl], f32, self.DST)
        b, _, bmax = tolerance.bc6h_block_errors(ref, theirs, f32, self.DST)
        res.update({"bc6h_err_gpu": a.sum() / (lw * lh * 3), "bc6h_err_ref": b.sum() / (lw * lh * 3), "ratio": float(a.sum() / max(b.sum(), 1e-9)),
                    "float_max_err_gpu": amax, "float_max_err_ref": bmax, "contract": "chain bit-exact; ratio <= 1.02", "ok": bool(exact and a.sum() <= 1.02 * b.sum())})
        return res


class C4:
    """BASELINE configs[3]: 1024 x 1024^2 RGBA8 -> 11-level BOX chain -> BC3, sharded across the GPUs"""
    name = "c4"
    metric = "Mtexels/s GenerateMipMaps(BOX) + BC3 encode of the chains (1024 x 1024^2 RGBA8)"
    dtype = "u8"
    scaling = "strong"
    W = H = 1024
    FMT, DST = 28, 77
    TOTAL = 1024
    kernel = "k_compress_bc15_t<77,28>"
    bound_note = "BC3: one thread per block, sequential fp32 Newton fits mandated by bit-exactness (issue bound); BOX mips HBM-bound"
    ncu_file = "r02_ncu_c4.txt"
    small_sample = {"count": 1}

    def __init__(self, args, world):
        self.world = world
        self.total = args.batch or self.TOTAL

    def workload(self):
        return ("batch of %d x 1024x1024 RGBA8 -> 11-level mip chain (default filter = BOX) -> BC3_UNORM of every level (BASELINE.json configs[3]); "
                "contiguous image ranges per GPU (%d per GPU at N=%d), one all-gather of the packed blocks per step" % (self.total, self.total // self.world, self.world))

    def setup(self, ctx):
        torch, capi, F, synth = ctx.torch, ctx.capi, ctx.F, ctx.synth
        from directxtex_b200 import dist as D
        self.lo, self.hi = D.shard_range(self.total, ctx.world, ctx.rank)
        self.B = self.hi - self.lo
        self.layout, self.chain_bytes = F.mip_chain_layout(self.FMT, self.W, self.H, 0)
        self.levels = len(self.layout)
        self.olayout, self.out_bytes = capi.texture_layout(self.DST, self.W, self.H, 1, self.levels)
        self.chain_texels = sum(lw * lh for (_, lw, lh, _, _) in self.layout)
        # 8 distinct seeded base images; image k = base[k % 8] rolled by 4 * (k // 8) rows and pixels (generated on the device)
        self.bases = [synth.c1_rgba8(self.W, self.H, seed=synth.SEED + s) for s in range(8)]
        dbase = [torch.from_numpy(b.reshape(self.H, self.W * 4)).cuda() for b in self.bases]
        self.d_chain = torch.zeros((self.B, self.chain_bytes), dtype=torch.uint8, device="cuda")
        for j in range(self.B):
            k = self.lo + j
            self.d_chain[j, : self.W * self.H * 4] = torch.roll(dbase[k % 8], shifts=(4 * (k // 8), 16 * (k // 8)), dims=(0, 1)).reshape(-1)
        self.d_out = [torch.zeros(self.B * self.out_bytes, dtype=torch.uint8, device="cuda") for _ in range(2)]
        self.chain = capi.images([_img(capi, lw, lh, self.FMT, row, sl, self.d_chain[j].data_ptr() + off)
                                  for j in range(self.B) for (off, lw, lh, row, sl) in self.layout])
        self.dst = [capi.images([_img(capi, lw, lh, self.DST, row, sl, o.data_ptr() + j * self.out_bytes + off)
                                 for j in range(self.B) for (off, lw, lh, row, sl) in self.olayout]) for o in self.d_out]
        self.gather_bytes = self.B * self.out_bytes

    def host_image(self, k):
        return np.roll(self.bases[k % 8].reshape(self.H, self.W * 4), (4 * (k // 8), 16 * (k // 8)), (0, 1)).reshape(self.H, self.W, 4)

    def units_per_step(self):
        return self.B * self.chain_texels

    def algo_bytes(self):               # BC3 kernel: 4 B in + 1 B out per chain texel
        return self.B * (self.chain_bytes + self.out_bytes)

    def step(self, ctx, i):
        lib = ctx.capi.lib
        m0, m1, e0, e1 = ctx.event(), ctx.event(), ctx.event(), ctx.event()
        m0.record()
        hr = lib.dxb200_generate_mipmaps_device(self.chain, self.B, self.levels, 0, ctx.stream_ptr)
        m1.record()
        if hr != 0:
            raise ctx.capi.DxTexError(hr, "dxb200_generate_mipmaps_device")
        e0.record()
        hr = lib.dxb200_compress_device(self.chain, self.B * self.levels, self.DST, 0, 0.5, 1.0, self.dst[i & 1], ctx.stream_ptr)
        e1.record()
        if hr != 0:
            raise ctx.capi.DxTexError(hr, "dxb200_compress_device")
        ctx.extra_events.setdefault("mips_box", []).append((m0, m1))
        return e0, e1, self.d_out[i & 1]

    def outputs(self, ctx):
        return {"mip_chain_rgba8": self.d_chain, "bc3_blocks": self.d_out[ctx.last_step & 1]}

    def e2e_setup(self, ctx):
        capi = ctx.capi
        self.Be = min(self.B, 128)
        lvl0 = self.W * self.H * 4
        self.pin_in = capi.lib.dxb200_host_alloc(self.Be * lvl0)
        self.pin_out = capi.lib.dxb200_host_alloc(self.Be * self.out_bytes)
        host = self.d_chain[: self.Be, :lvl0].contiguous().cpu().numpy()
        C.memmove(self.pin_in, host.ctypes.data, self.Be * lvl0)
        self.hbase = capi.images([_img(capi, self.W, self.H, self.FMT, self.W * 4, lvl0, self.pin_in + j * lvl0) for j in range(self.Be)])
        self.hdst = capi.images([_img(capi, lw, lh, self.DST, row, sl, self.pin_out + j * self.out_bytes + off)
                                 for j in range(self.Be) for (off, lw, lh, row, sl) in self.olayout])
        return {"units": self.Be * self.chain_texels, "h2d": self.Be * lvl0, "d2h": self.Be * self.out_bytes,
                "api": "dxb200_mipmaps_compress (host level-0 images in, packed BC3 chains out; the mip chain stays in HBM)"}

    def e2e_step(self, ctx):
        hr = ctx.capi.lib.dxb200_mipmaps_compress(self.hbase, self.Be, self.levels, 0, self.DST, 0, 0.5, 1.0, self.hdst)
        if hr != 0:
            raise ctx.capi.DxTexError(hr, "dxb200_mipmaps_compress")

    def e2e_check(self, ctx):
        host = np.ctypeslib.as_array((C.c_uint8 * (self.Be * self.out_bytes)).from_address(self.pin_out))
        dev = self.d_out[ctx.last_step & 1][: self.Be * self.out_bytes].cpu().numpy()
        assert np.array_equal(host, dev), "e2e and device-resident outputs differ"
        ctx.capi.lib.dxb200_host_free(self.pin_in)
        ctx.capi.lib.dxb200_host_free(self.pin_out)

    def _ref_chain_bc3(self, ref, img):
        from directxtex_b200 import formats as F
        hr, chain = ref.generate_mipmaps(img, self.W, self.H, self.FMT, 0)
        assert hr == 0
        layout, _ = F.mip_chain_layout(self.FMT, self.W, self.H, 0)
        outs = []
        for (off, lw, lh, row, sl) in layout:
            hr, b = ref.compress(chain[off:off + sl], lw, lh, self.FMT, self.DST, 0)
            assert hr == 0
            outs.append(b)
        return np.concatenate(outs)

    def reference_step(self, ref, count=4):
        from directxtex_b200 import synth
        if not hasattr(self, "bases"):
            self.bases = [synth.c1_rgba8(self.W, self.H, seed=synth.SEED + s) for s in range(8)]
            self.chain_texels = sum(max(1, self.W >> l) * max(1, self.H >> l) for l in range(11))
        t0 = time.perf_counter()
        for k in range(count):
            self._ref_chain_bc3(ref, self.bases[k % 8])
        sec = time.perf_counter() - t0
        return count * self.chain_texels, sec, "%d of the 1024^2 RGBA8 images: reference GenerateMipMaps(default = BOX) + Compress(BC3_UNORM, PARALLEL) of every level" % count

    def parity(self, ctx, ref):
        """sampled images of this rank's shard: the packed BC3 chain memcmp vs the reference (GenerateMipMaps + Compress per level)"""
        out = self.d_out[ctx.last_step & 1]
        picks = sorted({0, self.B // 3, self.B - 1})
        ok = True
        for j in picks:
            want = self._ref_chain_bc3(ref, self.host_image(self.lo + j))
            got = out[j * self.out_bytes:(j + 1) * self.out_bytes].cpu().numpy()
            ok = ok and bool(np.array_equal(got, want))
        return {"what": "images %s of rank 0's shard: packed BC3 mip chain (1,398,128 B each) memcmp vs reference GenerateMipMaps + Compress" % [self.lo + j for j in picks],
                "bit_exact": ok, "contract": "bit-exact", "ok": ok}


class C5:
    """BASELINE configs[4]: 8192x8192 R8 -> BC4_UNORM, and Convert R8 -> R32F -> R8 round trip"""
    name = "c5"
    metric = "Mtexels/s BC4 encode + Convert R8->R32F->R8 round trip (8192^2 R8)"
    dtype = "u8"
    scaling = "weak"
    W = H = 8192
    kernel = "k_convert_vec<61,41>"
    bound_note = "the R8 -> R32F row kernel is HBM-bound (5 B per texel); the BC4 kernel of the same step is reported under `kernels`"
    ncu_file = "r02_ncu_k_convert_vec.txt"
    small_sample = {"side": 1024}

    def __init__(self, args, world):
        self.B = args.batch or 24
        self.world = world

    def workload(self):
        return ("8192x8192 R8_UNORM -> BC4_UNORM, then Convert R8 -> R32_FLOAT -> R8 (BASELINE.json configs[4]); a step = %d such images per GPU" % self.B)

    def setup(self, ctx):
        torch, capi, F, synth = ctx.torch, ctx.capi, ctx.F, ctx.synth
        self.img = synth.c5_r8(self.W, self.H, seed=synth.SEED + ctx.rank)
        n = self.W * self.H
        base = torch.from_numpy(self.img).cuda()
        self.d_in = torch.empty((self.B, self.H, self.W), dtype=torch.uint8, device="cuda")
        for b in range(self.B):
            self.d_in[b] = torch.roll(base, shifts=(4 * b, 16 * b), dims=(0, 1))
        self.bc_row, self.bc_slice = F.compute_pitch(80, self.W, self.H)
        self.d_bc = [torch.zeros(self.B * self.bc_slice, dtype=torch.uint8, device="cuda") for _ in range(2)]
        self.d_f32 = torch.zeros((self.B, n), dtype=torch.float32, device="cuda")
        self.d_back = torch.zeros((self.B, n), dtype=torch.uint8, device="cuda")
        I = lambda fmt, row, sl, ptr: _img(capi, self.W, self.H, fmt, row, sl, ptr)
        self.src = capi.images([I(61, self.W, n, self.d_in[b].data_ptr()) for b in range(self.B)])
        self.bc = [capi.images([I(80, self.bc_row, self.bc_slice, o.data_ptr() + b * self.bc_slice) for b in range(self.B)]) for o in self.d_bc]
        self.f32 = capi.images([I(41, self.W * 4, n * 4, self.d_f32[b].data_ptr()) for b in range(self.B)])
        self.back = capi.images([I(61, self.W, n, self.d_back[b].data_ptr()) for b in range(self.B)])
        self.gather_bytes = self.B * self.bc_slice

    def units_per_step(self):
        return self.B * self.W * self.H

    def algo_bytes(self):               # R8 -> R32F: 1 B read + 4 B written per texel
        return self.B * self.W * self.H * 5

    def step(self, ctx, i):
        lib = ctx.capi.lib
        b0, b1, e0, e1, r0, r1 = (ctx.event() for _ in range(6))
        b0.record()
        hr = lib.dxb200_compress_device(self.src, self.B, 80, 0, 0.5, 1.0, self.bc[i & 1], ctx.stream_ptr)
        b1.record()
        e0.record()
        if hr == 0:
            hr = lib.dxb200_convert_device(self.src, self.B, 41, 0, 0.5, self.f32, ctx.stream_ptr)
        e1.record()
        r0.record()
        if hr == 0:
            hr = lib.dxb200_convert_device(self.f32, self.B, 61, 0, 0.5, self.back, ctx.stream_ptr)
        r1.record()
        if hr != 0:
            raise ctx.capi.DxTexError(hr, "c5 step")
        ctx.extra_events.setdefault("bc4", []).append((b0, b1))
        ctx.extra_events.setdefault("convert_r32f_to_r8", []).append((r0, r1))
        return e0, e1, self.d_bc[i & 1]

    def outputs(self, ctx):
        return {"bc4_blocks": self.d_bc[ctx.last_step & 1], "r32f": self.d_f32, "r8_roundtrip": self.d_back}

    def e2e_setup(self, ctx):
        capi = ctx.capi
        n = self.W * self.H
        self.Be = 1
        self.pin = [capi.lib.dxb200_host_alloc(s) for s in (n, self.bc_slice, n * 4, n)]
        C.memmove(self.pin[0], self.img.ctypes.data, n)
        I = lambda fmt, row, sl, ptr: _img(capi, self.W, self.H, fmt, row, sl, ptr)
        self.h = [capi.images([I(61, self.W, n, self.pin[0])]), capi.images([I(80, self.bc_row, self.bc_slice, self.pin[1])]),
                  capi.images([I(41, self.W * 4, n * 4, self.pin[2])]), capi.images([I(61, self.W, n, self.pin[3])])]
        return {"units": n, "h2d": n + n + 4 * n, "d2h": self.bc_slice + 4 * n + n, "api": "dxb200_compress + 2 x dxb200_convert (host pointers, pinned)"}

    def e2e_step(self, ctx):
        lib = ctx.capi.lib
        hr = lib.dxb200_compress(self.h[0], 1, 80, 0, 0.5, 1.0, self.h[1])
        if hr == 0:
            hr = lib.dxb200_convert(self.h[0], 1, 41, 0, 0.5, self.h[2])
        if hr == 0:
            hr = lib.dxb200_convert(self.h[2], 1, 61, 0, 0.5, self.h[3])
        if hr != 0:
            raise ctx.capi.DxTexError(hr, "c5 e2e")

    def e2e_check(self, ctx):
        n = self.W * self.H
        back = np.ctypeslib.as_array((C.c_uint8 * n).from_address(self.pin[3]))
        assert np.array_equal(back, self.img.reshape(-1)), "R8 -> R32F -> R8 is not the identity"
        bc = np.ctypeslib.as_array((C.c_uint8 * self.bc_slice).from_address(self.pin[1]))
        assert np.array_equal(bc, self.d_bc[ctx.last_step & 1][: self.bc_slice].cpu().numpy())
        for p in self.pin:
            ctx.capi.lib.dxb200_host_free(p)

    def reference_step(self, ref, side=2048):
        from directxtex_b200 import synth
        if not hasattr(self, "img"):
            self.img = synth.c5_r8(side, side)
        crop = np.ascontiguousarray(self.img[:side, :side])
        t0 = time.perf_counter()
        hr, _b = ref.compress(crop, side, side, 61, 80, 0)
        assert hr == 0
        hr, f = ref.convert(crop, side, side, 61, 41)
        assert hr == 0
        hr, _r = ref.convert(f, side, side, 41, 61)
        assert hr == 0
        sec = time.perf_counter() - t0
        return side * side, sec, "top-left %dx%d crop: reference Compress(BC4_UNORM, PARALLEL) + Convert R8->R32F + Convert R32F->R8" % (side, side)

    def parity(self, ctx, ref):
        got = self.d_bc[ctx.last_step & 1][: self.bc_slice].cpu().numpy().reshape(self.H // 4, self.W // 4 * 8)
        ok = True
        for by in (0, 777, 2047):
            rows = np.ascontiguousarray(self.img[by * 4:by * 4 + 4])
            hr, want = ref.compress(rows, self.W, 4, 61, 80, 0)
            ok = ok and hr == 0 and bool(np.array_equal(got[by], want))
        f = self.d_f32[0].cpu().numpy()
        conv = bool(np.array_equal(f, self.img.reshape(-1).astype(np.float32) / np.float32(255.0)))
        back = bool(np.array_equal(self.d_back[0].cpu().numpy(), self.img.reshape(-1)))
        return {"what": "image 0: BC4 block rows 0, 777, 2047 memcmp vs reference Compress; R8->R32F == b/255 exactly; R8->R32F->R8 identity",
                "bc4_bit_exact": ok, "convert_exact": conv, "roundtrip_identity": back, "contract": "bit-exact", "ok": bool(ok and conv and back)}


WORKLOADS = {"c2": C2, "c3": C3, "c4": C4, "c5": C5}


DUMP_BUDGET = 60 << 20      # bytes of float32 over all dumped outputs


def dump_outputs(outputs, path, torch):
    """writes each output as float32 (bytes as their values 0..255): whole, or -- when the outputs together exceed DUMP_BUDGET --
    the same seeded sample of 16-byte rows in every run; returns what was written"""
    os.makedirs(path, exist_ok=True)
    written = {}
    for name, t in sorted(outputs.items()):
        per_row = 16 // t.element_size()
        flat = t.reshape(-1)
        flat = flat[: flat.numel() // per_row * per_row].reshape(-1, per_row)
        n, cap = flat.shape[0], DUMP_BUDGET // len(outputs) // (per_row * 4)
        if n > cap:
            idx = np.sort(np.random.default_rng(0).choice(n, cap, replace=False))
            flat = flat[torch.from_numpy(idx).to(flat.device)]
        a = flat.float().cpu().numpy()
        np.save(os.path.join(path, name + ".npy"), a)
        written[name] = {"rows": int(a.shape[0]), "of_rows": int(n), "row_bytes": 16, "sample_seed": 0 if a.shape[0] < n else None}
    return written


# =====================================================================================================================
def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path (oracle/_ref = the unmodified sources), all host threads,
    one bounded sample of the workload per step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    wl = WORKLOADS[args.config](args, 1)
    ref = load_ref()
    for _ in range(args.warmup):
        wl.reference_step(ref)
    busy, units, desc = 0.0, 0, ""
    for _ in range(args.steps):
        u, sec, desc = wl.reference_step(ref)
        busy += sec
        units += u
    value = units / busy / 1e6
    cores = ref.threads()
    sample = desc + "; per step; OpenMP %d threads (OMP_PROC_BIND=spread); scalar DirectXMath shim (oracle/compat), not the SSE2 DirectXMath" % cores
    print(json.dumps({
        "impl": "reference", "metric": wl.metric, "value": value, "unit": "Mtexels/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": busy / args.steps * 1e3,
        "higher_is_better": True, "scaling": wl.scaling, "vs_baseline": None, "dtype": wl.dtype, "data": "synthetic",
        "config": {"workload": wl.workload(), "sample": sample},
        "cpu_baseline": {"value": value, "unit": "Mtexels/s", "cores": cores, "kind": "reference", "sample": sample},
        "e2e": {"value": value, "unit": "Mtexels/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--config", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--batch", type=int, default=0, help="images per GPU per step (c4: images in the whole batch); 0 = the config's default")
    ap.add_argument("--gather", default="nccl", choices=["nccl", "none"], help="end-of-step collection of the packed blocks at N>1")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed (rank 0) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.impl == "reference":
        return run_reference(args)
    args.warmup = max(args.warmup, 3)

    import torch
    import torch.distributed as dist
    from directxtex_b200 import capi, formats as F, synth

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    hr = capi.lib.dxb200_init(local)
    if hr != 0:
        raise capi.DxTexError(hr, "dxb200_init")

    ctx = Ctx()
    ctx.torch, ctx.capi, ctx.F, ctx.synth = torch, capi, F, synth
    ctx.rank, ctx.world, ctx.local = rank, world, local
    ctx.stream = torch.cuda.current_stream()
    ctx.stream_ptr = C.c_void_p(ctx.stream.cuda_stream)
    ctx.event = lambda: torch.cuda.Event(enable_timing=True)
    ctx.extra_events = {}
    wl = WORKLOADS[args.config](args, world)
    wl.setup(ctx)

    # ---- end-of-step all-gather of the packed blocks on a side stream, overlapping the next step's kernels
    side = torch.cuda.Stream() if world > 1 else None
    recv = [torch.empty(wl.gather_bytes * world, dtype=torch.uint8, device="cuda") for _ in range(2)] if (world > 1 and args.gather == "nccl") else None
    done = [None, None]

    def gather(i, out):
        if recv is None:
            return
        ready = torch.cuda.Event()
        ready.record(ctx.stream)
        with torch.cuda.stream(side):
            side.wait_event(ready)
            dist.all_gather_into_tensor(recv[i & 1], out[: wl.gather_bytes])
            ev = torch.cuda.Event()
            ev.record(side)
        done[i & 1] = ev

    def step(i):
        if done[i & 1] is not None:
            ctx.stream.wait_event(done[i & 1])          # the output buffer of step i-2 is free once its gather has finished
        e0, e1, out = wl.step(ctx, i)
        gather(i, out)
        return e0, e1

    def barrier():
        if world > 1:
            if side is not None:
                side.synchronize()
            dist.barrier()
        torch.cuda.synchronize()

    for i in range(args.warmup):
        step(i)
    barrier()
    ctx.extra_events = {}
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    launches0 = capi.launch_count()
    tma0 = capi.tma_launch_count()
    kern_ev = []
    e0, e1 = ctx.event(), ctx.event()
    barrier()
    e0.record()
    for i in range(args.steps):
        kern_ev.append(step(i))
    if side is not None:
        ctx.stream.wait_stream(side)
    e1.record()
    barrier()
    ctx.last_step = args.steps - 1
    launches = capi.launch_count() - launches0
    tma_timed = capi.tma_launch_count() - tma0
    clocks = sampler.stop() if rank == 0 else None
    dumped = dump_outputs(wl.outputs(ctx), args.dump_outputs, torch) if (args.dump_outputs and rank == 0) else None
    ms_total = e0.elapsed_time(e1)
    kern_ms = float(np.mean([a.elapsed_time(b) for a, b in kern_ev]))
    extra_ms = {k: float(np.mean([a.elapsed_time(b) for a, b in v])) for k, v in ctx.extra_events.items()}
    t = torch.tensor([ms_total, kern_ms], dtype=torch.float64, device="cuda")
    units = torch.tensor([float(wl.units_per_step())], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(units, op=dist.ReduceOp.SUM)
    ms_per_step = float(t[0]) / args.steps
    kern_ms = float(t[1])
    value = float(units[0]) / (ms_per_step * 1e-3) / 1e6

    alternates = wl.alternates(ctx) if (hasattr(wl, "alternates") and world == 1) else {}

    # ---- end to end through the host-pointer C ABI (pinned host memory, H2D + D2H inside the timed region)
    info = wl.e2e_setup(ctx)
    e2e_steps = max(3, min(args.steps, 5))
    for _ in range(2):
        wl.e2e_step(ctx)
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        wl.e2e_step(ctx)
    barrier()
    e2e_ms = (time.perf_counter() - t0) * 1e3 / e2e_steps
    te = torch.tensor([e2e_ms], dtype=torch.float64, device="cuda")
    ue = torch.tensor([float(info["units"])], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
        dist.all_reduce(ue, op=dist.ReduceOp.SUM)
    e2e_value = float(ue[0]) / (float(te[0]) * 1e-3) / 1e6
    wl.e2e_check(ctx)

    if rank == 0:
        pk, pk_kind = peaks()
        achieved = wl.algo_bytes() / (kern_ms * 1e-3) / 1e9
        from tests import oracle_lib
        cpu_baseline = parity = None
        if os.path.exists(oracle_lib.REF_SO):
            ref = load_ref()
            u, sec, desc = wl.reference_step(ref)
            threads = ref.threads()
            ref.L.ref_omp_set_threads(1)
            u1, sec1, _ = wl.reference_step(ref, **wl.small_sample)
            ref.L.ref_omp_set_threads(threads)
            parity = wl.parity(ctx, ref)
            cpu_baseline = {"value": u / sec / 1e6, "unit": "Mtexels/s", "cores": threads, "kind": "reference",
                            "sample": desc + ", %.2f s" % sec, "threads": threads, "proc_bind": os.environ.get("OMP_PROC_BIND"),
                            "one_thread_value": u1 / sec1 / 1e6, "per_core_scaling": (u / sec) / (u1 / sec1) / max(threads, 1),
                            "note": "the reference sources are compiled against a scalar DirectXMath stand-in (oracle/compat), not the SSE2 DirectXMath; "
                                    "bounded sample, not the full workload"}
        traffic = None
        rd, wr = ncu_metric(wl.ncu_file, "dram__bytes_read.sum"), ncu_metric(wl.ncu_file, "dram__bytes_write.sum")
        if rd is not None and wr is not None:
            traffic = (rd + wr) * 1e6
        inst = ncu_metric(wl.ncu_file, "smsp__inst_executed.sum")
        issue = ncu_metric(wl.ncu_file, "smsp__issue_active.avg.pct_of_peak_sustained_active")
        out = {
            "metric": wl.metric, "value": value, "unit": "Mtexels/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": wl.scaling, "vs_baseline": None, "dtype": wl.dtype, "data": "synthetic",
            "config": {"workload": wl.workload(), "name": wl.name,
                       "l2": "inputs per step are far larger than the 126 MB L2 (no flush needed)",
                       "parallelism": "image-per-GPU x%d" % world, "gather": (args.gather if world > 1 else "none"),
                       "timed_region_s": ms_total * 1e-3},
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": "Mtexels/s", "h2d_bytes_per_step": info["h2d"], "d2h_bytes_per_step": info["d2h"],
                    "ms_per_step": float(te[0]), "api": info["api"], "steps": e2e_steps},
            "gpu_launches": int(launches), "tma_launches": int(tma_timed),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": achieved / pk["hbm_gbs"],
                         "traffic": traffic, "traffic_source": ("dram__bytes_read.sum + dram__bytes_write.sum of one launch, profiles/" + wl.ncu_file) if traffic else None,
                         "peak_source": pk_kind, "kernel": wl.kernel, "kernel_ms": kern_ms, "algorithmic_bytes": wl.algo_bytes(),
                         "issue_slot_frac": (issue / 100.0) if issue else None,
                         "warp_inst_per_block": (inst / (4096 * 4096 / 16)) if (inst and args.config == "c2") else None,
                         "note": wl.bound_note},
            "kernels": dict({wl.kernel: kern_ms}, **extra_ms),
            "alternates": alternates,
            "cpu_baseline": cpu_baseline,
            "parity": parity,
        }
        if dumped is not None:
            out["dumped_outputs"] = {"dir": args.dump_outputs, "arrays": dumped}
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
