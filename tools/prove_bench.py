"""gl_prove (the whole prover from the witness on, one call) at standard_recursion_config geometry: 135 wires, 80 routed,
4 constants (2 selectors) + 80 sigmas, 2 challenges, quotient_degree_factor 8; FRI rate 3, cap 4, 16 proof-of-work bits,
28 query rounds.  The circuit is the repo's gate set on a numpy-vectorised instance (tests/prove_circuit.py `large`): row 0
a PublicInputGate, the other rows NoopGate / ConstantGate, 2^16 copy-constraint swaps.

Reports per size, each the median of --reps after --warmup, timed with a host clock around calls that return synchronised:
  prove_device_ms    gl_prove with the witness in device memory (a torch CUDA tensor)
  prove_host_ms      gl_prove with the witness in page-able host memory (numpy)
  stepwise_ms        the same proof driven stage by stage from Python (PolynomialBatch commits, the product Challenger,
                     permutation_zs into device memory, compute_quotient_polys to host and back, fri.opening_set,
                     fri.prove_openings_device); its words are checked equal to gl_prove's
  verify_ms          plonk_verifier.verify_proof on the proof's bytes
Writes one JSON (default profiles/r4_prove_bench.json) with the GPU name and power limit read in the same run.

    python tools/prove_bench.py [--sizes 13,16,18,20] [--reps 5] [--warmup 1] [--out PATH]
"""
import argparse
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
sys.path.insert(0, os.path.join(ROOT, "tests"))

DIGEST = np.array([11, 22, 33, 44], dtype=np.uint64)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "nvidia-smi unavailable: " + q.stderr.strip()


def timed(fn, reps, warmup):
    for _ in range(warmup):
        fn()
    ts = []
    for _ in range(reps):
        t = time.perf_counter()
        fn()
        ts.append((time.perf_counter() - t) * 1e3)
    return statistics.median(ts), ts


def prove_stepwise(glb, fri, ctx, c, cs, fp, wires, pis):
    """plonky2's prove() stage by stage through the Python mirror; returns the words gl_prove writes."""
    import torch

    lg_n, _, R, _, _, nch, qdf, _ = c["circuit"]
    n = 1 << lg_n
    pih = glb.PoseidonHash.hash_no_pad(np.asarray(pis, dtype=np.uint64), ctx=ctx)
    w = glb.PolynomialBatch.from_values(wires, 3, False, 4, ctx=ctx, want_coeffs=False)
    ch = fri.Challenger(ctx)
    ch.observe_hash(DIGEST)
    ch.observe_hash(pih)
    ch.observe_cap(w.merkle_tree.cap)
    betas, gammas = ch.get_n_challenges(nch), ch.get_n_challenges(nch)
    zs = torch.empty((nch * -(-R // qdf), n), dtype=torch.int64, device=f"cuda:{ctx.device}")
    glb.host.permutation_zs(c["circuit"], c["k_is"], cs, w, betas, gammas, out=zs, ctx=ctx)
    zb = glb.PolynomialBatch.from_values(zs, 3, False, 4, ctx=ctx, want_coeffs=False)
    del zs
    ch.observe_cap(zb.merkle_tree.cap)
    alphas = ch.get_n_challenges(nch)
    q = glb.host.compute_quotient_polys(c["circuit"], c["gates"], c["k_is"], cs, w, zb, pih, betas, gammas, alphas, ctx=ctx)
    qb = glb.PolynomialBatch.from_coeffs(q, 3, False, 4, ctx=ctx)
    ch.observe_cap(qb.merkle_tree.cap)
    zeta = ch.get_extension_challenge()
    g = pow(pow(7, (fri.P - 1) >> 32, fri.P), 1 << (32 - lg_n), fri.P)
    oracles = [cs, w, zb, qb]
    batches = [(zeta, [(oi, pi) for oi, o in enumerate(oracles) for pi in range(o.num_columns)]),
               ((zeta[0] * g % fri.P, zeta[1] * g % fri.P), [(2, pi) for pi in range(nch)])]
    at_zeta, at_next = fri.opening_set(oracles, batches)
    cut = cs.num_columns + w.num_columns + nch
    opening_words = at_zeta[:cut] + at_next + at_zeta[cut:]
    ch.observe_extension_elements(np.array(at_zeta, dtype=np.uint64))
    ch.observe_extension_elements(np.array(at_next, dtype=np.uint64))
    flat = fri.prove_openings_device(oracles, batches, ch, fp, ctx, flat=True)
    out = np.concatenate([w.merkle_tree.cap.reshape(-1), zb.merkle_tree.cap.reshape(-1), qb.merkle_tree.cap.reshape(-1),
                          np.array(opening_words, dtype=np.uint64).reshape(-1), flat])
    for b in (w, zb, qb):
        b.free()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="13,16,18,20")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r4_prove_bench.json"))
    a = ap.parse_args()
    import torch

    glb = importlib.import_module("plonky2-lib_b200")
    importlib.import_module("plonky2-lib_b200.build").build()
    fri = importlib.import_module("plonky2-lib_b200.fri")
    wire = importlib.import_module("plonky2-lib_b200.wire")
    pv = importlib.import_module("plonky2-lib_b200.plonk_verifier")
    from prove_circuit import large

    ctx = glb.Context.default()
    res = {"gpu": gpu_info(), "geometry": "135 wires, 80 routed, 4 constants (2 selectors) + 80 sigmas, 2 challenges, qdf 8; "
           "rate 3, cap 4, 16 PoW bits, 28 queries; row 0 PublicInputGate, other rows NoopGate / ConstantGate",
           "timing": f"host clock around calls that return synchronised, median of {a.reps} after {a.warmup} warm-up",
           "sizes": {}}
    pis = [1, 2, 3, 4, 5]
    for lg_n in [int(s) for s in a.sizes.split(",")]:
        c = large(lg_n, pis, seed=lg_n)
        fp = fri.FriParams.for_degree(glb.FriConfig(), lg_n)
        cs = glb.PolynomialBatch.from_values(np.concatenate([c["constants"], c["sigmas"]]), 3, False, 4, ctx=ctx)
        wires_host = c["wires"]
        wires_dev = torch.from_numpy(wires_host.view(np.int64)).to(f"cuda:{ctx.device}")

        def prove(wires):
            return glb.host.prove(c["circuit"], c["gates"], c["k_is"], cs, DIGEST, fp, wires, pis, ctx=ctx)

        dev_ms, dev_all = timed(lambda: prove(wires_dev), a.reps, a.warmup)
        host_ms, host_all = timed(lambda: prove(wires_host), a.reps, a.warmup)
        p = prove(wires_dev)
        step = prove_stepwise(glb, fri, ctx, c, cs, fp, wires_dev, pis)
        assert np.array_equal(step, p["words"]), "stage-by-stage proof differs from gl_prove"
        step_ms, step_all = timed(lambda: prove_stepwise(glb, fri, ctx, c, cs, fp, wires_dev, pis), a.reps, a.warmup)
        data = wire.proof_with_public_inputs_to_bytes(p["caps"], p["openings"], p["opening_proof"], p["public_inputs"])
        common = pv.CommonData(c["circuit"], c["gates"], c["k_is"], fp, len(pis))
        vd = pv.VerifierData(cs.merkle_tree.cap, DIGEST)
        ver_ms, ver_all = timed(lambda: pv.verify_proof(data, common, vd, ctx=ctx), a.reps, a.warmup)
        res["sizes"][str(lg_n)] = {"rows": 1 << lg_n, "prove_device_ms": dev_ms, "prove_host_ms": host_ms, "stepwise_ms": step_ms,
                                   "verify_ms": ver_ms, "proof_bytes": len(data), "runs": {"prove_device": dev_all,
                                   "prove_host": host_all, "stepwise": step_all, "verify": ver_all}}
        print(lg_n, json.dumps({k: v for k, v in res["sizes"][str(lg_n)].items() if k != "runs"}), flush=True)
        cs.free()
        del wires_dev
        torch.cuda.empty_cache()
    res["gpu_after"] = gpu_info()
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", a.out)


if __name__ == "__main__":
    main()
