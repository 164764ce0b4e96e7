"""Measures ComputeMSE and the IsAlphaAllOpaque scan on device-resident images (CUDA events, median of >= 20 calls after warm-up),
beside a device-to-device copy of the same bytes in the same run, and prints whole-image quality figures of the GPU's C2 (BC7) and
C4 (BC3 mip chains) outputs.  Every input is larger than the B200's 126 MB L2.  Writes JSON lines to --out DIR/analysis.jsonl.

    python tools/analysis_bench.py --out DIR [--reps 30]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=30)
    args = ap.parse_args()
    import torch
    from directxtex_b200 import capi, synth
    os.makedirs(args.out, exist_ok=True)
    lines = []

    def emit(d):
        print(json.dumps(d), flush=True)
        lines.append(d)

    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:          # noqa: BLE001
        q = "unknown (%s)" % e
    emit({"gpu": q.splitlines()[0] if q else "unknown", "torch": torch.__version__})
    stream = torch.cuda.current_stream()
    sp = C.c_void_p(stream.cuda_stream)

    def timed(fn):
        for _ in range(3):
            fn()
        ts = []
        for _ in range(args.reps):
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            fn()
            e.record()
            torch.cuda.synchronize()
            ts.append(s.elapsed_time(e) * 1e-3)
        return float(np.median(ts))

    def copy_bw(nbytes):
        x = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
        y = torch.empty_like(x)
        t = timed(lambda: y.copy_(x))
        return 2 * nbytes / t            # read + write

    def dev(arr):
        return torch.from_numpy(np.ascontiguousarray(arr).view(np.uint8).reshape(-1).copy()).cuda()

    out = torch.zeros(5, dtype=torch.float32, device="cuda")

    def mse_case(name, a, fa, b, fb, w, h):
        da, db = dev(a), dev(b)
        ia, ib = [capi.make_image(da.data_ptr(), w, h, fa)], [capi.make_image(db.data_ptr(), w, h, fb)]
        assert capi.compute_mse_device(ia, ib, 0, out.data_ptr(), sp) == 0
        t = timed(lambda: capi.compute_mse_device(ia, ib, 0, out.data_ptr(), sp))
        nbytes = da.numel() + db.numel()
        cbw = copy_bw(nbytes // 2)
        emit({"op": "compute_mse", "case": name, "w": w, "h": h, "bytes": nbytes, "seconds": t, "GBps": nbytes / t / 1e9,
              "copy_GBps": cbw / 1e9, "fraction_of_copy": (nbytes / t) / cbw, "mse": float(out[0].item())})
        return da, db, t

    rng = np.random.default_rng(1)
    n8 = 8192
    a8 = rng.integers(0, 256, n8 * n8 * 4, dtype=np.uint8)
    b8 = a8 ^ rng.integers(0, 4, a8.size, dtype=np.uint8)
    mse_case("rgba8_8192", a8, 28, b8, 28, n8, n8)
    del a8, b8
    n = 4096
    af = synth.c2_rgba32f(n, n, seed=2)
    bf = (af + np.float32(0.01)).astype(np.float32)
    mse_case("rgba32f_4096", af, 2, bf, 2, n, n)
    del bf
    nr = 16384
    ar = rng.integers(0, 256, nr * nr, dtype=np.uint8)
    mse_case("r8_16384", ar, 61, ar ^ np.uint8(1), 61, nr, nr)
    del ar

    # BC7 (C2, 4096^2) against its RGBA32F source: fused kernel versus Decompress into a scratch image + an uncompressed compare
    blocks = capi.compress(af, n, n, 2, 98)
    dblk, dsrc, t_fused = mse_case("bc7_vs_rgba32f_4096_fused", blocks, 98, af, 2, n, n)
    scratch = torch.empty(n * n * 16, dtype=torch.uint8, device="cuda")
    ib, isrc, isc = [capi.make_image(dblk.data_ptr(), n, n, 98)], [capi.make_image(dsrc.data_ptr(), n, n, 2)], [capi.make_image(scratch.data_ptr(), n, n, 2)]

    def two_step():
        assert capi.lib.dxb200_decompress_device(capi.images(ib), 1, 2, capi.images(isc), sp) == 0
        assert capi.compute_mse_device(isc, isrc, 0, out.data_ptr(), sp) == 0
    t_two = timed(two_step)
    emit({"op": "compute_mse", "case": "bc7_vs_rgba32f_4096_decompress_then_compare", "seconds": t_two, "fused_seconds": t_fused,
          "fused_speedup": t_two / t_fused})

    # IsAlphaAllOpaque on the C4 batch's mip chains (opaque: a full scan)
    items, size = 64, 1024                     # 64 of the C4 batch's 1024^2 RGBA8 chains
    chains = []
    flag = torch.zeros(1, dtype=torch.int32, device="cuda")
    imgs, nbytes = [], 0
    for i in range(items):
        img = synth.c1_rgba8(size, size, seed=40 + i).reshape(-1)
        img[3::4] = 255
        chain, layout = capi.generate_mipmaps(img, size, size, 28)
        d = dev(chain)
        chains.append(d)
        imgs += [capi.Image(lw, lh, 28, row, sl, d.data_ptr() + off) for (off, lw, lh, row, sl) in layout]
        nbytes += chain.size
    assert capi.is_alpha_all_opaque_device(imgs, flag.data_ptr(), sp) == 0
    torch.cuda.synchronize()
    t = timed(lambda: capi.is_alpha_all_opaque_device(imgs, flag.data_ptr(), sp))
    cbw = copy_bw(nbytes)
    emit({"op": "is_alpha_all_opaque", "case": "c4_rgba8_chains_%dx%d^2" % (items, size), "bytes": nbytes, "seconds": t, "GBps": nbytes / t / 1e9,
          "copy_GBps": cbw / 1e9, "fraction_of_copy": (nbytes / t) / cbw, "opaque": int(flag.item())})
    del chains

    # whole-image quality of the GPU's outputs (no reference encoder involved)
    mse, mse_v = capi.compute_mse(blocks, 98, af, 2, n, n)
    emit({"quality": "C2 BC7 4096^2 vs RGBA32F source", "mse": float(mse), "mseV": [float(v) for v in mse_v]})
    img = synth.c1_rgba8(size, size, seed=40)
    bc3 = capi.compress(img, size, size, 28, 77)
    mse, mse_v = capi.compute_mse(bc3, 77, img, 28, size, size)
    emit({"quality": "C4 BC3 %d^2 level 0 vs RGBA8 source" % size, "mse": float(mse), "mseV": [float(v) for v in mse_v]})
    with open(os.path.join(args.out, "analysis.jsonl"), "w") as f:
        for d in lines:
            f.write(json.dumps(d) + "\n")


if __name__ == "__main__":
    main()
