"""gl_permutation_zs at standard_recursion_config geometry (135 wires, 80 routed, 4 constants + 80 sigmas, 2 challenges,
quotient_degree_factor 8), device output, at 2^16, 2^18 and 2^20 rows.

Reports per size: the wall time of the call (host clock around calls that end in a device synchronise; median of --reps
after --warmup), the recovery on its own (gl_fft_batch of the same 2R columns at the same n, device resident), the Z part
(call minus recovery) with the algorithmic bytes it moves and their rate, a per-kernel split from torch.profiler in a
separate pass, and the CPU oracle's glo_permutation_zs on the same instance with the host's core count.  The instance has
identity sigmas (k_j w^i, made with the library's forward transform) and random wires, so every grand product is 1.
Writes one JSON (default profiles/r3_permutation_zs_bench.json) with the GPU name and power limit read in the same run.

    python tools/permutation_zs_bench.py [--sizes 16,18,20] [--reps 7] [--warmup 2] [--out PATH] [--no-oracle]
"""
import argparse
import ctypes as C
import importlib
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

NUM_WIRES, R, NUM_CONSTANTS, NCH, DEG = 135, 80, 4, 2, 8
CHUNKS = -(-R // DEG)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "nvidia-smi unavailable: " + q.stderr.strip()


def timed(fn, sync, reps, warmup):
    for _ in range(warmup):
        fn()
    sync()
    ts = []
    for _ in range(reps):
        t = time.perf_counter()
        fn()
        sync()
        ts.append((time.perf_counter() - t) * 1e3)
    return statistics.median(ts), ts


def kernel_split(fn, sync):
    import torch
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        sync()
        torch.cuda.synchronize()
    out = {}
    for e in prof.key_averages():
        us = getattr(e, "device_time_total", None)
        if us is None:
            us = getattr(e, "cuda_time_total", 0)
        if us:
            out[e.key] = round(us / 1e3, 4)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="16,18,20")
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_permutation_zs_bench.json"))
    ap.add_argument("--no-oracle", action="store_true")
    args = ap.parse_args()
    glb = importlib.import_module("plonky2-lib_b200")
    N = glb._native
    P = glb.host.P
    ctx = glb.Context(0)
    k_is = np.array([pow(7, j, P) for j in range(R)], dtype=np.uint64)
    res = {"gpu": gpu_info(), "geometry": {"num_wires": NUM_WIRES, "num_routed_wires": R, "constants_sigmas": NUM_CONSTANTS + R,
                                           "num_challenges": NCH, "quotient_degree_factor": DEG}, "output": "GL_DEVICE",
           "timing": f"host clock around calls ending in a device synchronise, median of {args.reps} after {args.warmup} warm-up",
           "host_cores": os.cpu_count(), "omp_num_threads": os.environ.get("OMP_NUM_THREADS"), "sizes": []}
    for lg in [int(s) for s in args.sizes.split(",")]:
        n = 1 << lg
        rng = np.random.default_rng(lg)
        sig_coeffs = np.zeros((R, n), dtype=np.uint64)
        sig_coeffs[:, 1] = k_is                                   # sigma_j(x) = k_j x: the identity permutation
        sigmas = glb.fft(sig_coeffs, ctx=ctx)
        wires = rng.integers(0, P, (NUM_WIRES, n), dtype=np.uint64)
        cs_vals = np.concatenate([rng.integers(0, P, (NUM_CONSTANTS, n), dtype=np.uint64), sigmas])
        cs = glb.PolynomialBatch.from_values(cs_vals, 3, False, 4, ctx=ctx, want_coeffs=False)
        w = glb.PolynomialBatch.from_values(wires, 3, False, 4, ctx=ctx, want_coeffs=False)
        circuit = (lg, NUM_WIRES, R, NUM_CONSTANTS, 0, NCH, DEG, 0)
        betas = rng.integers(0, P, NCH, dtype=np.uint64)
        gammas = rng.integers(0, P, NCH, dtype=np.uint64)
        out = glb.DeviceBuffer((NCH * CHUNKS, n), ctx)
        grand = []

        def call():
            _, g = glb.host.permutation_zs(circuit, k_is, cs, w, betas, gammas, out=out, ctx=ctx)
            grand[:] = [int(x) for x in g]

        total_ms, total_all = timed(call, ctx.sync, args.reps, args.warmup)
        rec = glb.DeviceBuffer((2 * R, n), ctx)

        def recover():
            ctx.check(ctx._lib.gl_fft_batch(ctx._h, C.c_void_p(rec.ptr), lg, 2 * R, N.GL_DEVICE))

        rec_ms, rec_all = timed(recover, ctx.sync, args.reps, args.warmup)
        z_bytes = 2 * R * n * 8 + 2 * NCH * CHUNKS * n * 8
        z_ms = total_ms - rec_ms
        entry = {"log_n": lg, "call_ms": round(total_ms, 4), "call_ms_all": [round(t, 4) for t in total_all],
                 "recovery_fft_2R_ms": round(rec_ms, 4), "recovery_ms_all": [round(t, 4) for t in rec_all],
                 "z_part_ms": round(z_ms, 4), "z_part_bytes": z_bytes,
                 "z_part_GBps": round(z_bytes / (z_ms * 1e6), 1) if z_ms > 0 else None, "grand_products": grand}
        try:
            entry["kernels_ms_one_call_profiler"] = kernel_split(call, ctx.sync)
        except Exception as e:   # the profiler pass is an extra; its failure is reported, not hidden
            entry["kernels_ms_one_call_profiler"] = f"profiler failed: {e!r}"
        rec.free()
        out.free()
        cs.free()
        w.free()
        if not args.no_oracle:
            from oracle import pyoracle

            t = time.perf_counter()
            pyoracle.permutation_zs(circuit, k_is, wires, sigmas, betas, gammas)
            entry["oracle_cpu_ms"] = round((time.perf_counter() - t) * 1e3, 1)
        print(json.dumps(entry), flush=True)
        res["sizes"].append(entry)
        del wires, cs_vals, sigmas, sig_coeffs
    res["gpu_after"] = gpu_info()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", args.out)
    ctx.close()


if __name__ == "__main__":
    main()
