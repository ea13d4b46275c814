"""The whole-proof verifier's vanishing evaluation (plonk_verifier.eval_vanishing_poly, exact extension-field integers)
against the CPU oracle's glo_vanishing_at_point, with the imaginary part set to zero: at subgroup points, where the openings
are rows of the instance's columns, and at random base-field points, where they are the polynomials' values there.  Satisfying
and corrupted instances of tests/quotient_circuit.py.  No device is needed."""
import importlib

import numpy as np
import pytest

from conftest import P
from quotient_circuit import build

pv = importlib.import_module("plonky2-lib_b200.plonk_verifier")


def _instance(corrupt, lg_n, oracle, seed):
    c = build(lg_n, seed=seed, corrupt=corrupt)
    rng = np.random.default_rng(seed)
    betas, gammas, alphas = (rng.integers(0, P, 2, dtype=np.uint64) for _ in range(3))
    if corrupt == "copy":      # the oracle refuses an open grand product: any columns do for comparing two evaluations
        zs = rng.integers(0, P, (20, 1 << lg_n), dtype=np.uint64)
    else:
        zs = oracle.permutation_zs(c["circuit"], c["k_is"], c["wires"], c["sigmas"], betas, gammas)
    return c, zs, betas, gammas, alphas


def _openings(lcs, lw, lz, nz, num_constants, nch=2):
    ext = lambda v: np.stack([np.asarray(v, dtype=np.uint64), np.zeros(len(v), dtype=np.uint64)], axis=1)  # noqa: E731
    return {"constants": ext(lcs[:num_constants]), "plonk_sigmas": ext(lcs[num_constants:]), "wires": ext(lw),
            "plonk_zs": ext(lz[:nch]), "plonk_zs_next": ext(nz[:nch]), "partial_products": ext(lz[nch:]),
            "quotient_polys": np.zeros((0, 2), dtype=np.uint64)}


def _compare(c, x, lcs, lw, lz, nz, betas, gammas, alphas, oracle):
    want = oracle.vanishing_at_point(c["circuit"], c["gates"], c["k_is"], x, lcs, lw, lz, nz, c["pih"], betas, gammas, alphas)
    got = pv.eval_vanishing_poly(c["circuit"], c["gates"], c["k_is"], (x, 0), _openings(lcs, lw, lz, nz, c["circuit"][3]), c["pih"],
                                 [int(b) for b in betas], [int(g) for g in gammas], [int(a) for a in alphas])
    assert got == [(int(v), 0) for v in want]
    return want


@pytest.mark.parametrize("corrupt", [None, "bit", "copy"])
def test_vanishing_at_subgroup_points_matches_oracle(oracle, corrupt):
    lg_n = 5
    c, zs, betas, gammas, alphas = _instance(corrupt, lg_n, oracle, seed=7)
    n = 1 << lg_n
    w = pow(pow(7, (P - 1) >> 32, P), 1 << (32 - lg_n), P)
    cs = np.concatenate([c["constants"], c["sigmas"]])
    nonzero = 0
    for i in range(1, n):
        want = _compare(c, pow(w, i, P), cs[:, i], c["wires"][:, i], zs[:, i], zs[:, (i + 1) % n], betas, gammas, alphas, oracle)
        nonzero += any(int(v) for v in want)
    if corrupt is None:
        assert nonzero == 0            # a satisfying witness: the vanishing polynomial is zero on the subgroup
    else:
        assert nonzero > 0


@pytest.mark.parametrize("corrupt", [None, "bit", "copy"])
def test_vanishing_at_random_points_matches_oracle(oracle, corrupt):
    lg_n = 4
    c, zs, betas, gammas, alphas = _instance(corrupt, lg_n, oracle, seed=11)
    g = pow(pow(7, (P - 1) >> 32, P), 1 << (32 - lg_n), P)
    cs = np.concatenate([c["constants"], c["sigmas"]])
    coeffs = [np.stack([oracle.ifft(col) for col in m]) for m in (cs, c["wires"], zs)]
    rng = np.random.default_rng(3)
    for _ in range(3):
        x = int(rng.integers(2, P, dtype=np.uint64))
        at = lambda m, pt: np.array([oracle.eval_base_poly_at_ext(col, (pt, 0))[0] for col in m], dtype=np.uint64)  # noqa: E731
        _compare(c, x, at(coeffs[0], x), at(coeffs[1], x), at(coeffs[2], x), at(coeffs[2], x * g % P), betas, gammas, alphas, oracle)

