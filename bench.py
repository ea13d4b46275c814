#!/usr/bin/env python
"""bench.py -- LDE + Merkle commit throughput (BASELINE.json metric "LDE+Merkle commit cells/s").

Workload (BASELINE.json configs[1]): PolynomialBatch::from_values on 2^20 rows x 135 Goldilocks columns,
rate_bits = 3, cap_height = 4, Poseidon leaves.  A cell = one input trace element (n * c per commit).
A step = one commit.

  value   : inputs resident in HBM (GL_DEVICE), outputs left on the device, cap to the host.
  e2e     : the same call through the C ABI with HOST (pinned) buffers: values H2D, coefficients + cap D2H
            inside the timed region; e2e.pageable_per_polynomial = the drop-in's own buffers (one ordinary array per
            polynomial, gl_commit_from_values_cols).  At N > 1 every rank uploads its columns and downloads its
            coefficient columns, pipelined with the LDE rounds.
  proof_trace: informational, N = 1: the commits + prove_openings of one proof at config 1's row count.
  roofline: the dominant kernel (Poseidon leaf hashing) timed with the library's own CUDA events.
  cpu_baseline: the CPU oracle (a port of plonky2 v0.1.4 semantics, oracle/) on a bounded sample, rank 0, N=1.

N > 1 (torchrun, one rank per GPU): one commit sharded by LDE coset = top-level Merkle subtree
(SURVEY 8e).  Rank r inverse-transforms its share of the columns, the coefficients are NCCL all-gathered in a
few rounds that overlap the LDE of the previous round, every rank builds its leaf blocks + subtrees, and the
cap is NCCL all-gathered: total work fixed => "strong" scaling.

--impl reference: the reference's CPU implementation of the path is Rust in an un-vendored crate and
cannot be built here (no cargo); the reference arm times the oracle port on all host cores.
"""
from __future__ import annotations

import argparse
import importlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "lde_merkle_commit_cells_per_s"
UNIT = "cells/s"
LOG_N, COLS, RATE_BITS, CAP_HEIGHT = 20, 135, 3, 4
IMAD_PER_PERMUTATION = 6700  # SURVEY 8d: plonky2's own schedule, 32x32 multiply(-add)s per permutation


def workload_name(log_n, cols):
    return f"commit 2^{log_n} rows x {cols} Goldilocks cols, rate_bits={RATE_BITS}, cap_height={CAP_HEIGHT}, Poseidon leaves"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        hi = [x for x in sm if mx and x > 0.5 * mx] or sm
        return {"sm_mhz": float(np.median(hi)) if hi else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def cpu_baseline(log_n_sample: int, cols: int, repeat: int = 1):
    """The oracle port of the path on the host cores (bounded sample of the workload)."""
    from oracle import pyoracle as o

    use_all_host_threads(o)
    v = o.synthetic_values(cols, 1 << log_n_sample)
    o.commit_from_values(o.synthetic_values(4, 256), RATE_BITS, CAP_HEIGHT, want_leaves=False)  # warm tables
    best = None
    for _ in range(repeat):
        t = time.perf_counter()
        o.commit_from_values(v, RATE_BITS, CAP_HEIGHT, want_leaves=True)
        dt = time.perf_counter() - t
        best = dt if best is None else min(best, dt)
    cells = cols << log_n_sample
    return {
        "value": cells / best, "unit": UNIT, "cores": int(o.lib().glo_num_threads()), "kind": "port",
        "sample": f"one commit of 2^{log_n_sample} rows x {cols} cols (rate_bits={RATE_BITS}, cap_height={CAP_HEIGHT}) = "
                  f"1/{1 << (LOG_N - log_n_sample)} of the workload rows, {best:.2f} s; oracle/gl_oracle.c (OpenMP port of plonky2 v0.1.4 semantics)",
    }, best


def proof_trace(glb, ctx, torch, lg=16):
    """The other half of BASELINE.json's metric ("prove ms per circuit") as far as this path goes: the commit + opening
    trace of one data.prove(pw) at the row count SURVEY 8d estimates for config 1 (single ECDSA, 2^16 rows): wires,
    Z / partial products and quotient commits (135 + 20 + 16 polynomials, ordinary page-able host arrays in, coefficients
    out) + prove_openings over those and the build-time constants/sigmas oracle (84 polynomials).  Witness generation and
    compute_quotient_polys are host stages of the reference and are not part of this number.  Informational: never
    fails the bench."""
    try:
        fri = importlib.import_module("plonky2-lib_b200.fri")
        P = glb.host.P
        n = 1 << lg
        colsets = (84, 135, 20, 16)
        rng = np.random.default_rng(lg)
        vals = [rng.integers(0, P, size=(c, n), dtype=np.uint64) for c in colsets]
        const_sigmas = glb.PolynomialBatch.from_values(vals[0], RATE_BITS, False, CAP_HEIGHT, want_coeffs=False, ctx=ctx)
        zeta = (0x123456789ABCDEF % P, 0x0FEDCBA987654321 % P)
        g = pow(pow(7, (P - 1) >> 32, P), 1 << (32 - lg), P)
        inst = [(zeta, [(oi, pi) for oi, c in enumerate(colsets) for pi in range(c)]),
                ((zeta[0] * g % P, zeta[1] * g % P), [(2, pi) for pi in range(20)])]
        prm = fri.FriParams.for_degree(glb.FriConfig(), lg)

        def once():
            bs = [const_sigmas] + [glb.PolynomialBatch.from_values(v, RATE_BITS, False, CAP_HEIGHT, want_coeffs=True, ctx=ctx) for v in vals[1:]]
            ch = fri.Challenger(ctx)
            for b in bs:
                ch.observe_cap(b.merkle_tree.cap)
            proof = fri.prove_openings_device(bs, inst, ch, prm, ctx)      # gl_fri_prove: one C-ABI call, transcript on the device
            for b in bs[1:]:
                b.free()
            return proof

        once()
        best = None
        for _ in range(3):
            t = time.perf_counter()
            proof = once()
            dt = time.perf_counter() - t
            best = dt if best is None else min(best, dt)
        # the same trace with the witness already in HBM (what a device-side witness generator / N3 pipeline hands over)
        dvals = [torch.from_numpy(v.view(np.int64)).to(ctx_device(ctx)) for v in vals[1:]]

        def once_resident():
            bs = [const_sigmas] + [glb.PolynomialBatch.from_values(v, RATE_BITS, False, CAP_HEIGHT, want_coeffs=False, ctx=ctx) for v in dvals]
            ch = fri.Challenger(ctx)
            for b in bs:
                ch.observe_cap(b.merkle_tree.cap)
            fri.prove_openings_device(bs, inst, ch, prm, ctx, flat=True)
            for b in bs[1:]:
                b.free()

        once_resident()
        best_res = None
        for _ in range(3):
            t = time.perf_counter()
            once_resident()
            dt = time.perf_counter() - t
            best_res = dt if best_res is None else min(best_res, dt)
        const_sigmas.free()
        return {"config1_ecdsa_2^%d_rows_ms" % lg: best * 1e3, "config1_ecdsa_2^%d_rows_resident_inputs_ms" % lg: best_res * 1e3,
                "fri_layers": len(proof["commit_phase_merkle_caps"]),
                "query_rounds": len(proof["query_round_proofs"]),
                "what": "3 commits (135 + 20 + 16 polynomials, page-able host arrays, coefficients out) + prove_openings over 4 oracles (gl_fri_prove, one call); wall clock"}
    except Exception as e:  # noqa: BLE001
        return {"error": repr(e)}


def ctx_device(ctx):
    return "cuda:%d" % ctx.device


def use_all_host_threads(o):
    """torchrun exports OMP_NUM_THREADS=1 to every rank; the CPU arm is meant to use every host core it may run on."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    o.lib().glo_set_num_threads(max(1, n))


def config_for(log_n, cols, world):
    """The workload both arms run (the reference arm prints the same dict: same shape, same cells per step)."""
    return {
        "workload": workload_name(log_n, cols), "cells_per_step": cols << log_n,
        "l2": "inputs (1.13 GB) and LDE (9.06 GB) are larger than the 126 MB L2 (and than any host cache); no flush needed",
        "parallelism": ("N=1: one GPU runs the whole commit" if world == 1 else
                        f"N={world}: one commit sharded over {world} GPUs behind the C ABI (gl_group_*): IFFT by column blocks, NCCL "
                        "all-gather of the coefficients in rounds overlapped with the LDE and the streamed leaf absorb of earlier rounds, "
                        "LDE/Merkle by coset block = top-level subtree, NCCL all-gather of the cap") + "; the reference arm runs the same commit on the host cores",
    }


def golden_case(log_n, cols):
    """The full-size fixture the CPU oracle produced once for the benchmarked shapes (tests/golden/commit_fullsize.json)."""
    try:
        g = json.load(open(os.path.join(ROOT, "tests", "golden", "commit_fullsize.json")))
    except Exception:
        return None
    for case in g["cases"]:
        if (case["lg_n"], case["c"], case["rate_bits"], case["cap_height"]) == (log_n, cols, RATE_BITS, CAP_HEIGHT):
            return case
    return None


def check_parity(cap_host, log_n, cols):
    """Every N: the cap this run produced must be the oracle's, bit for bit.  A mismatch fails the run."""
    case = golden_case(log_n, cols)
    if case is None:
        return {"parity_checked": False, "parity_note": "no full-size golden fixture for this shape (tests/golden/commit_fullsize.json holds 2^18 and 2^20 x 135)"}
    got = [f"{int(x):016x}" for x in np.asarray(cap_host).reshape(-1)]
    if got != case["cap"]:
        raise SystemExit("bench.py: PARITY FAILURE: the Merkle cap differs from tests/golden/commit_fullsize.json (oracle) at 2^%d x %d" % (log_n, cols))
    return {"parity_checked": True, "parity_note": "cap (16 x 4 field elements) equals the CPU oracle's at this exact shape: tests/golden/commit_fullsize.json"}


def run_reference(args):
    """Reference arm: the reference's own CPU implementation is un-buildable here (Rust, un-vendored plonky2 fork, no
    cargo) so the oracle port stands in: upstream's CPU schedule (fast partial rounds, MDS on 32-bit halves, per-column
    FFTs, transpose, recursive subtree Merkle), OpenMP where upstream uses rayon, on every host core.

    SAME CONFIG as the GPU arm: every timed step is one commit of the full workload (2^20 rows x 135 columns).  A 2^16-row
    calibration commit projects the cost first; only if K full-size steps would not fit --ref-budget-s (slow or few
    cores) is the per-step sample cut to the largest 2^k rows that fits, and the line says so (config.sample).  Warm-up
    steps are small commits: they spin up the thread pool and build the twiddle / Poseidon tables, there is no JIT."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import pyoracle as o

    use_all_host_threads(o)
    cores = int(o.lib().glo_num_threads())
    for _ in range(max(args.warmup, 0)):
        o.commit_from_values(o.synthetic_values(args.cols, 1 << 10), RATE_BITS, CAP_HEIGHT, want_leaves=False)
    lg = args.ref_log_n
    if lg <= 0:
        cal = min(16, args.log_n)
        vc = o.synthetic_values(args.cols, 1 << cal)
        t = time.perf_counter()
        o.commit_from_values(vc, RATE_BITS, CAP_HEIGHT, want_leaves=True)
        t_cal = time.perf_counter() - t
        lg = args.log_n
        budget = args.ref_budget_s
        if budget <= 0:
            # the driver gives a 1-GPU lease's reference arm 1800 s and each arm of the 8-GPU scaling sequence 870 s
            # (BENCH_r01.json / SCALE_r01.json step limits): stay well inside whichever applies to this box
            try:
                ngpu = len(subprocess.run(["nvidia-smi", "-L"], capture_output=True, text=True, timeout=20).stdout.strip().splitlines())
            except Exception:
                ngpu = 0
            budget = 1150 if ngpu <= 1 else 700
        args.ref_budget_s = budget
        # measured: a 2^20-row commit costs ~1.15x what 16 commits of 2^16 rows do (caches, page faults)
        while lg > cal and args.steps * t_cal * (1 << (lg - cal)) * 1.15 > budget:
            lg -= 1
        del vc
    v = o.synthetic_values(args.cols, 1 << lg)
    cap = None
    t0 = time.perf_counter()
    for _ in range(args.steps):
        cap = o.commit_from_values(v, RATE_BITS, CAP_HEIGHT, want_leaves=True)["cap"]
    dt = time.perf_counter() - t0
    cells = args.cols << lg
    val = cells * args.steps / dt
    full = lg == args.log_n
    sample = (("each step = one commit of the FULL workload, 2^%d rows x %d cols" % (lg, args.cols)) if full else
              ("each step = one commit of 2^%d rows x %d cols (1/%d of the workload rows: %d full-size steps would not fit "
               "--ref-budget-s %d on this host)" % (lg, args.cols, 1 << (args.log_n - lg), args.steps, args.ref_budget_s)))
    sample += ("; oracle port of plonky2 v0.1.4's CPU schedule (fast partial rounds), %d OpenMP threads; the Rust reference "
               "cannot be built: no cargo, plonky2 fork not vendored" % cores)
    config = config_for(args.log_n, args.cols, args.gpus)
    if not full:
        config["sample"] = sample
    out = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        "config": config,
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "same_config": full,
    }
    if full:
        out.update(check_parity(cap, args.log_n, args.cols))
    emit(out)


def synthetic_values_device(torch, cols, n, device, col0=0):
    """values[col][row] = splitmix64(seed ^ ((col << 32) + row)) mod p, generated on the device (int64 wraps)."""
    def c64(x):
        return x - (1 << 64) if x >= (1 << 63) else x

    col = (torch.arange(col0, col0 + cols, dtype=torch.int64, device=device) << 32)[:, None]
    row = torch.arange(n, dtype=torch.int64, device=device)[None, :]
    z = (col + row) ^ c64(0x706C6F6E6B7932)
    z = z + c64(0x9E3779B97F4A7C15)

    def lsr(x, k):
        return (x >> k) & ((1 << (64 - k)) - 1)

    z = (z ^ lsr(z, 30)) * c64(0xBF58476D1CE4E5B9)
    z = (z ^ lsr(z, 27)) * c64(0x94D049BB133111EB)
    z = z ^ lsr(z, 31)
    # canonical: z >= p (unsigned)  <=>  z in [-2^32 + 1, -1] as signed
    ge = (z < 0) & (z >= -(1 << 32) + 1)
    return torch.where(ge, z + ((1 << 32) - 1), z).contiguous()


DUMP_SEED, DUMP_BYTES = 0x706C6F6E6B7932, 32 << 20


def u64_halves(a):
    """u64 -> float64 [..., 2] = (low 32 bits, high 32 bits): exact, which a u64 -> float cast of a field element is not."""
    a = np.asarray(a).view(np.uint64)
    return np.stack([a & np.uint64(0xFFFFFFFF), a >> np.uint64(32)], axis=-1).astype(np.float64)


def dump_outputs(out_dir, cap_host, coeffs_dev):
    """What the last timed step handed its caller, as .npy files: the whole cap and, when the step returns coefficients
    (1.13 GB at the default shape), every coefficient column at a fixed, seeded sample of rows, with those row indices."""
    import torch

    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "cap.npy"), u64_halves(cap_host))
    if coeffs_dev is None:
        return
    cols, n = coeffs_dev.shape
    k = max(1, min(n, DUMP_BYTES // (16 * cols)))
    rows = np.sort(np.random.default_rng(DUMP_SEED).choice(n, size=k, replace=False))
    sample = coeffs_dev.index_select(1, torch.from_numpy(rows).to(coeffs_dev.device)).cpu().numpy()
    np.save(os.path.join(out_dir, "coeffs_sample.npy"), u64_halves(sample))
    np.save(os.path.join(out_dir, "coeffs_sample_rows.npy"), rows.astype(np.float64))


_RESULT_FD = None


def _claim_stdout():
    """stdout carries exactly ONE line, the JSON result.  Native libraries (NCCL's version banner, CUDA) write to
    file descriptor 1 directly, so everything that is not the result goes to stderr: fd 1 is pointed at fd 2 for the
    whole run and the result line is written to the saved descriptor at the end."""
    global _RESULT_FD
    if _RESULT_FD is None:
        sys.stdout.flush()
        _RESULT_FD = os.dup(1)
        os.dup2(2, 1)


def emit(result: dict):
    line = (json.dumps(result) + "\n").encode()
    sys.stdout.flush()
    if _RESULT_FD is None:
        os.write(1, line)
    else:
        os.write(_RESULT_FD, line)


def main():
    _claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--log-n", type=int, default=LOG_N)
    ap.add_argument("--cols", type=int, default=COLS)
    ap.add_argument("--ref-log-n", type=int, default=0, help="rows (log2) of the reference arm's per-step commit; 0 = the full workload if K steps fit --ref-budget-s")
    ap.add_argument("--ref-budget-s", type=int, default=0, help="time budget of the reference arm's K timed steps; 0 = 1150 s on a 1-GPU box, 700 s on a multi-GPU box")
    ap.add_argument("--cpu-log-n", type=int, default=18, help="rows (log2) of the cpu_baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-proof-trace", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step to DIR/<name>.npy (float64; each u64 field element as its "
                         "low and high 32 bits along the last axis): the cap and a seeded sample of the coefficients")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; this path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")  # keep stdout to the one JSON line
        dist.init_process_group("nccl", device_id=dev)
    glb = importlib.import_module("plonky2-lib_b200")
    ctx = glb.Context(local)
    lib, N = ctx._lib, glb._native
    import ctypes as C

    log_n, cols = args.log_n, args.cols
    n = 1 << log_n
    cells = n * cols
    stream = torch.cuda.ExternalStream(ctx.stream, device=dev)

    values = synthetic_values_device(torch, cols, n, dev)
    torch.cuda.synchronize()
    cap_dev = torch.zeros((1 << CAP_HEIGHT, 4), dtype=torch.int64, device=dev)
    phases = []

    if world == 1:
        coeffs_dev = torch.empty_like(values)

        def step():
            h = C.c_void_p()
            ctx.check(lib.gl_commit_from_values(ctx._h, values.data_ptr(), log_n, cols, RATE_BITS, CAP_HEIGHT,
                                                coeffs_dev.data_ptr(), cap_dev.data_ptr(), C.byref(h), N.GL_DEVICE))
            phases.append(ctx.commit_phase_ms())
            lib.gl_commit_free(h)
            return cap_dev
    else:
        # One commit sharded over the ranks, entirely behind the C ABI (gl_group_*, csrc/gl_group.inc.cu): rank r
        # inverse-transforms its polynomials of every round, the rounds are all-gathered in place by the library's own
        # NCCL communicator while the previous round is extended, every rank builds its leaf blocks + subtrees, and the cap
        # is all-gathered.  torch.distributed is the launcher's control plane only (token broadcast, barrier, max of times).
        par = importlib.import_module("plonky2-lib_b200.parallel")
        par.check_shardable(world, RATE_BITS, CAP_HEIGHT)
        ctx.check(lib.gl_ctx_bind_host_numa(ctx._h)) if os.environ.get("BENCH_NUMA_BIND", "1") == "1" else None
        tok = torch.zeros(N.GL_GROUP_ID_BYTES, dtype=torch.uint8, device=dev)
        if rank == 0:
            tok.copy_(torch.frombuffer(bytearray(glb.Group.unique_id()), dtype=torch.uint8))
        dist.broadcast(tok, 0)
        group = glb.Group.from_token(ctx, rank, world, bytes(tok.cpu().numpy().tobytes()))
        vptr = (C.c_void_p * 1)(values.data_ptr())
        capptr = (C.c_void_p * 1)(cap_dev.data_ptr())
        hs = (C.c_void_p * 1)()

        # GL_COMMIT_STREAM_HASH: every complete group of 8 gathered polynomials is absorbed into the leaves' sponge states as
        # soon as its round is extended, so the compute stream has hashing to do while the next all-gather is on the wire
        # (same digests; the phase split below comes from one extra, untimed commit without the flag)
        gflags = N.GL_COMMIT_STREAM_HASH if os.environ.get("BENCH_GROUP_STREAM_HASH", "1") == "1" else 0

        def step(flags=gflags):
            group.check(lib.gl_group_commit_from_values(group._h, vptr, log_n, cols, RATE_BITS, CAP_HEIGHT, None, capptr, hs,
                                                        N.GL_DEVICE, flags))
            phases.append(group.commit_phase_ms())
            lib.gl_commit_free(hs[0])
            return cap_dev

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # torch ops and NCCL collectives of a step are issued on the library's stream
    torch.cuda.set_stream(stream)
    for _ in range(args.warmup):
        step()
    launches0 = ctx.kernel_launches
    phases.clear()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record(stream)
    for _ in range(args.steps):
        cap = step()
    e1.record(stream)
    barrier()
    wall = time.perf_counter() - t0
    dev_ms = e0.elapsed_time(e1)
    # the C ABI blocks at return, so device time == wall time up to launch latency; report the device clock
    t = torch.tensor([dev_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms = float(t.item())
    clocks = sampler.stop() if rank == 0 else None
    launches = ctx.kernel_launches - launches0
    if world > 1 and gflags:
        # phase split and the dominant kernel's time: one commit with the leaves hashed in one pass (k_leaf_hash_cols),
        # outside the timed region, timed by the library's CUDA events like every other step
        phases.clear()
        step(0)
        barrier()
    ms_per_step = dev_ms / args.steps
    value = cells * args.steps / (dev_ms * 1e-3)
    cap_host = cap.cpu().numpy().view(np.uint64)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, cap_host, coeffs_dev if world == 1 else None)

    # ---- e2e: HOST (pinned) buffers through the same C-ABI call -------------------------------------
    e2e = None
    if world == 1 and not args.no_e2e:
        hv = glb.pinned_empty((cols, n))
        hc = glb.pinned_empty((cols, n))
        hcap = np.zeros((1 << CAP_HEIGHT, 4), dtype=np.uint64)
        hv[:] = values.cpu().numpy().view(np.uint64)

        def estep():
            h = C.c_void_p()
            ctx.check(lib.gl_commit_from_values(ctx._h, hv.ctypes.data, log_n, cols, RATE_BITS, CAP_HEIGHT,
                                                hc.ctypes.data, hcap.ctypes.data, C.byref(h), N.GL_HOST))
            lib.gl_commit_free(h)

        for _ in range(2):
            estep()
        torch.cuda.synchronize()
        ksteps = max(2, min(args.steps, 5))
        e0.record(stream)
        for _ in range(ksteps):
            estep()
        e1.record(stream)
        torch.cuda.synchronize()
        ems = e0.elapsed_time(e1) / ksteps
        assert np.array_equal(hcap, cap_host), "e2e cap differs from the device-resident run"
        e2e = {"value": cells / (ems * 1e-3), "unit": UNIT, "h2d_bytes_per_step": int(cells * 8),
               "d2h_bytes_per_step": int(cells * 8 + hcap.nbytes), "ms_per_step": ems,
               "api": "gl_commit_from_values(space=GL_HOST), pinned host buffers"}
        # the drop-in's own buffers: one ordinary (page-able) array per polynomial, coefficients back the same way
        # (gl_commit_from_values_cols; staged through page-locked rings by helper threads, csrc/host_staging.cu)
        pcols = [np.array(hv[j]) for j in range(cols)]
        ocols = [np.zeros(n, dtype=np.uint64) for _ in range(cols)]
        ip = (C.c_void_p * cols)(*[a.ctypes.data for a in pcols])
        op = (C.c_void_p * cols)(*[a.ctypes.data for a in ocols])
        hcap2 = np.zeros_like(hcap)

        def pstep():
            h = C.c_void_p()
            ctx.check(lib.gl_commit_from_values_cols(ctx._h, ip, log_n, cols, RATE_BITS, CAP_HEIGHT, op,
                                                     hcap2.ctypes.data, C.byref(h)))
            lib.gl_commit_free(h)

        pstep()
        torch.cuda.synchronize()
        e0.record(stream)
        for _ in range(ksteps):
            pstep()
        e1.record(stream)
        torch.cuda.synchronize()
        pms = e0.elapsed_time(e1) / ksteps
        assert np.array_equal(hcap2, cap_host) and np.array_equal(ocols[cols - 1], hc[cols - 1]), "page-able e2e differs"
        e2e["pageable_per_polynomial"] = {"value": cells / (pms * 1e-3), "unit": UNIT, "ms_per_step": pms,
                                          "api": "gl_commit_from_values_cols, %d separate page-able arrays in and out" % cols}
        del hv, hc, pcols, ocols

    if world > 1 and not args.no_e2e:
        # ---- e2e at N GPUs: the same collective C-ABI call with HOST buffers.  Every rank holds the batch in page-locked
        # host memory (allocated after gl_ctx_bind_host_numa, i.e. on the GPU's NUMA node), uploads only the polynomials it
        # inverse-transforms, and brings exactly those coefficient vectors back while the LDE and the tree run; every rank
        # receives the whole cap on the host.  Summed over the ranks each input cell crosses PCIe once each way.
        hv = glb.pinned_empty((cols, n))
        hc = glb.pinned_empty((cols, n))
        hc[:] = 0
        hcap = np.zeros((1 << CAP_HEIGHT, 4), dtype=np.uint64)
        hv[:] = values.cpu().numpy().view(np.uint64)
        hvp, hcp, hcapp = (C.c_void_p * 1)(hv.ctypes.data), (C.c_void_p * 1)(hc.ctypes.data), (C.c_void_p * 1)(hcap.ctypes.data)
        # GL_COMMIT_STREAM_HASH: the leaves absorb each round as soon as it is extended, so hashing runs while the next
        # rounds are still on PCIe / NVLink (at 2 GPUs the step is bound by the arithmetic: plain hashing there)
        eflags = N.GL_COMMIT_STREAM_HASH if world >= int(os.environ.get("BENCH_STREAM_HASH_MIN_WORLD", "4")) else 0

        def estep():
            group.check(lib.gl_group_commit_from_values(group._h, hvp, log_n, cols, RATE_BITS, CAP_HEIGHT, hcp, hcapp, hs,
                                                        N.GL_HOST, eflags))
            lib.gl_commit_free(hs[0])

        for _ in range(2):
            estep()
        barrier()
        ksteps = max(2, min(args.steps, 5))
        e0.record(stream)
        for _ in range(ksteps):
            estep()
        e1.record(stream)
        barrier()
        t = torch.tensor([e0.elapsed_time(e1) / ksteps], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ems = float(t.item())
        assert np.array_equal(hcap, cap_host), "e2e cap differs from the device-resident run"
        # the coefficient vectors that came back: every polynomial on exactly one rank, and the fixture's sample columns
        mine = np.array([bool(hc[j].any()) for j in range(cols)])
        cnt = torch.tensor(mine.astype(np.int64), device=dev)
        dist.all_reduce(cnt)
        assert bool((cnt == 1).all()), "e2e: every coefficient vector must come back on exactly one rank"
        case = golden_case(log_n, cols)
        if case is not None:
            import hashlib
            for j, want in case["coeff_cols"].items():
                if mine[int(j)]:
                    assert hashlib.sha256(np.ascontiguousarray(hc[int(j)]).tobytes()).hexdigest() == want, "e2e coefficients differ from the oracle's"
        if rank == 0:
            e2e = {"value": cells / (ems * 1e-3), "unit": UNIT, "h2d_bytes_per_step": int(cells * 8),
                   "d2h_bytes_per_step": int(cells * 8 + world * cap_host.nbytes), "ms_per_step": ems,
                   "api": "gl_group_commit_from_values(space=GL_HOST%s): per rank its polynomials H2D from pinned memory, the coefficient "
                          "exchange by the ranks' own pull kernels over peer memory (NVLink), its coefficient vectors D2H, the whole cap D2H" % (", GL_COMMIT_STREAM_HASH" if eflags else "")}
        del hv, hc

    if rank != 0:
        if world > 1:
            group.close()
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel: k_leaf_hash_cols, timed by the library's CUDA events -------
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    leaf_ms = float(np.mean([p["leaf_hash"] for p in phases]))
    N_local = (n << RATE_BITS) // world
    leaf_bytes = N_local * cols * 8 + N_local * 32
    perms_leaf = N_local * ((cols + 7) // 8)
    achieved = leaf_bytes / (leaf_ms * 1e-3) / 1e9
    phase_mean = {k: float(np.mean([p[k] for p in phases])) for k in phases[0]}
    roofline = {
        "bound": "hbm", "kernel": "k_leaf_hash_cols (Poseidon hash_no_pad of every LDE row)",
        "achieved": achieved, "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak,
        "peak_source": "MEASURED_PEAKS.json hbm_gbs (measured)" if peaks else "fallback 6650 GB/s",
        "traffic": None, "kernel_ms": leaf_ms, "algorithmic_bytes_per_launch": leaf_bytes,
        "note": "integer-pipe bound kernel (17 Poseidon permutations per 1080-byte leaf): see roofline_int",
    }
    # integer roofline (SURVEY 8d): algorithmic work in 32x32->64 multiply-add equivalents against the MEASURED
    # mad.wide.u32 issue rate of this GPU (tools/pipe_peaks.cu -> profiles/r2_pipe_peaks.json)
    imad_peak, imad_src = 148 * 64 * 1.965e9, "nominal 148 SM x 64 lanes x 1965 MHz"
    try:
        pk = json.load(open(os.path.join(ROOT, "profiles", "r2_pipe_peaks.json")))
        imad_peak = float(pk["imad_wide"]["ops_per_s"])
        imad_src = "measured mad.wide.u32 rate, profiles/r2_pipe_peaks.json (tools/pipe_peaks.cu)"
    except Exception:
        pass
    perms_commit = N_local * ((cols + 7) // 8) + (N_local - (1 << CAP_HEIGHT) // world)
    ntt_bfly = (cols * n * log_n // 2 if world == 1 else 0) + cols * N_local * log_n // 2
    imad_commit = perms_commit * IMAD_PER_PERMUTATION + ntt_bfly * 4 + cols * N_local * 4
    roofline_int = {
        "bound": "imad", "kernel": "k_leaf_hash_cols",
        "achieved": perms_leaf * IMAD_PER_PERMUTATION / (leaf_ms * 1e-3) / 1e12,
        "unit": "T 32x32->64 multiply-add equivalents/s (6700 per permutation, 4 per butterfly: SURVEY 8d)",
        "permutations_per_s": perms_leaf / (leaf_ms * 1e-3),
        "peak": imad_peak / 1e12, "peak_source": imad_src,
        "whole_commit_achieved": imad_commit / (ms_per_step * 1e-3) / 1e12,
    }
    roofline_int["frac"] = roofline_int["achieved"] / roofline_int["peak"]
    roofline_int["whole_commit_frac"] = roofline_int["whole_commit_achieved"] / roofline_int["peak"]
    try:
        tr = json.load(open(os.path.join(ROOT, "profiles", "r2_leaf_hash_traffic.json")))
        if tr.get("cols") == cols:
            roofline["traffic"] = tr["dram_bytes_per_leaf"] * N_local
            roofline["traffic_source"] = tr.get("source")
    except Exception:
        pass

    out = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "u64", "data": "synthetic",
        "config": config_for(log_n, cols, world),
        "phases_ms": phase_mean, "wall_ms_per_step": wall / args.steps * 1e3,
        "roofline": roofline, "roofline_int": roofline_int, "clocks": clocks, "gpu_launches": int(launches),
        "cap0": [f"{int(x):016x}" for x in cap_host[0]],
    }
    out.update(check_parity(cap_host, log_n, cols))
    if e2e:
        out["e2e"] = e2e
    if world == 1 and not args.no_proof_trace:
        out["proof_trace"] = proof_trace(glb, ctx, torch)
    if world == 1 and not args.no_cpu_baseline:
        cb, _ = cpu_baseline(min(args.cpu_log_n, log_n), cols)
        out["cpu_baseline"] = cb
    emit(out)
    if world > 1:
        group.close()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
