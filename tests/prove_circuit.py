"""Test infrastructure: whole-circuit instances for gl_prove at any size (numpy-vectorised, so 2^20 rows build in seconds),
shared by tests/test_gpu_prove.py and tools/prove_bench.py.  The gate set is tests/quotient_circuit.py's; row 0 is a
PublicInputGate whose wires 0..3 hold hash_no_pad(public_inputs), every other row a NoopGate or a ConstantGate."""
import numpy as np

from oracle import pyoracle as o
from quotient_circuit import GATES, UNUSED_SELECTOR

P = o.P


def identity_sigmas(k_is, lg_n) -> np.ndarray:
    """sigma_j(i) = k_j w^i: the values on the subgroup of the polynomials k_j X (the oracle's forward transform)."""
    n = 1 << lg_n
    out = np.empty((len(k_is), n), dtype=np.uint64)
    for j, k in enumerate(k_is):
        c = np.zeros(n, dtype=np.uint64)
        c[1 % n] = k
        out[j] = o.fft(c)
    return out


def large(lg_n, pis, seed, swaps=1 << 16):
    """standard_recursion_config geometry (135 wires, 80 routed, 2 selectors + 2 gate constants, 2 challenges, qdf 8).
    Identity sigmas with `swaps` random disjoint transpositions of routed positions outside the gates' wires (columns
    4 .. 79), whose two ends hold equal values: a witness that satisfies every constraint."""
    rng = np.random.default_rng(seed)
    n, R = 1 << lg_n, 80
    wires = rng.integers(0, P, (135, n), dtype=np.uint64)
    consts = np.zeros((4, n), dtype=np.uint64)
    is_const = rng.random(n) < 0.3
    is_const[0] = False
    consts[0] = np.where(is_const, 1, 0).astype(np.uint64)
    consts[0, 0] = 2
    consts[1] = UNUSED_SELECTOR
    vals = rng.integers(0, 1 << 32, (2, n), dtype=np.uint64)
    consts[2:4] = np.where(is_const, vals, 0)
    wires[0:2] = np.where(is_const, vals, wires[0:2])
    pih = o.hash_no_pad(np.asarray(pis, dtype=np.uint64))
    wires[0:4, 0] = pih
    k_is = np.array([pow(7, j, P) for j in range(R)], dtype=np.uint64)
    sigmas = identity_sigmas(k_is, lg_n)
    swaps = min(swaps, (R - 4) * n // 4)
    pos = 4 * n + rng.choice((R - 4) * n, 2 * swaps, replace=False)
    a, b = pos[:swaps], pos[swaps:]
    sf, wf = sigmas.reshape(-1), wires[:R].reshape(-1)
    sf[a], sf[b] = sf[b].copy(), sf[a].copy()
    wf[b] = wf[a]
    circuit = (lg_n, 135, R, 4, 2, 2, 8, len(GATES))
    gates = [(k, ops, s, g0, g1, 0) for (k, ops, s, g0, g1) in GATES]
    return {"circuit": circuit, "gates": gates, "k_is": k_is, "constants": consts, "sigmas": sigmas, "wires": wires, "pih": pih,
            "num_pis": len(pis)}
