"""CPU ORACLE for plonky2::plonk::prover::prove from the witness on (TEST INFRASTRUCTURE ONLY).

Upstream's order, built from the oracle's pieces: commit_from_values / commit_from_coeffs, fri_oracle.Challenger,
permutation_zs, quotient_polys, eval_base_poly_at_ext and fri_oracle.prove_openings.  Returns the structure
host.prove returns, so that wire.proof_with_public_inputs_to_bytes gives comparable bytes for both.
"""
from __future__ import annotations

import numpy as np

from . import fri_oracle as fo
from . import pyoracle as o

P = o.P
OPENING_SET_FIELDS = ("constants", "plonk_sigmas", "wires", "plonk_zs", "plonk_zs_next", "partial_products", "quotient_polys")


def prove(circuit, gates, k_is, constants, sigmas, circuit_digest, wires, public_inputs=(), rate_bits=3, cap_height=4, pow_bits=16,
          num_query_rounds=28, times_x=False) -> dict:
    """constants [num_constants][n], sigmas [num_routed_wires][n], wires [num_wires][n]: values on the subgroup."""
    lg_n, _, _, _, _, nch, qdf, _ = [int(v) for v in circuit]
    pis = np.asarray(public_inputs, dtype=np.uint64).reshape(-1)
    pih = o.hash_no_pad(pis)
    cs = o.commit_from_values(np.concatenate([constants, sigmas]), rate_bits, cap_height)
    w = o.commit_from_values(wires, rate_bits, cap_height)
    ch = fo.Challenger()
    ch.observe_hash(circuit_digest)
    ch.observe_hash(pih)
    ch.observe_cap(w["cap"])
    betas = [ch.get_challenge() for _ in range(nch)]
    gammas = [ch.get_challenge() for _ in range(nch)]
    z = o.commit_from_values(o.permutation_zs(circuit, k_is, wires, sigmas, betas, gammas), rate_bits, cap_height)
    ch.observe_cap(z["cap"])
    alphas = [ch.get_challenge() for _ in range(nch)]
    quotient = o.quotient_polys(circuit, gates, k_is, cs["leaves"], w["leaves"], z["leaves"], rate_bits, pih, betas, gammas, alphas)
    q = o.commit_from_coeffs(quotient, rate_bits, cap_height)
    ch.observe_cap(q["cap"])
    zeta = tuple(ch.get_extension_challenge())
    assert fo.ext_pow(zeta, 1 << lg_n) != (1, 0), "Opening point is in the subgroup."
    g = int(o.lib().glo_primitive_root_of_unity(lg_n))
    zeta_next = fo.ext_mul(zeta, (g, 0))
    oracles = [cs, w, z, q]
    polys = [c["coeffs"] for c in oracles]
    batches = [(zeta, [(oi, pi) for oi, c in enumerate(polys) for pi in range(c.shape[0])]), (zeta_next, [(2, pi) for pi in range(nch)])]
    at_zeta, at_next = fo.opening_set(polys, batches)
    nc, R, nw = constants.shape[0], sigmas.shape[0], wires.shape[0]
    zc = z["coeffs"].shape[0]
    cuts = np.cumsum([nc, R, nw, nch, zc - nch])
    parts = np.split(np.array(at_zeta, dtype=np.uint64).reshape(-1, 2), cuts)
    openings = dict(zip(OPENING_SET_FIELDS, (parts[0], parts[1], parts[2], parts[3], np.array(at_next, dtype=np.uint64).reshape(-1, 2),
                                             parts[4], parts[5])))
    for f in ("constants", "plonk_sigmas", "wires", "plonk_zs", "partial_products", "quotient_polys"):
        ch.observe_extension_elements(openings[f])
    ch.observe_extension_elements(openings["plonk_zs_next"])
    trees = [fo.MerkleTree(c["leaves"], cap_height) for c in oracles]
    fri = fo.prove_openings(polys, trees, batches, ch, lg_n, rate_bits, cap_height, pow_bits, num_query_rounds, times_x)
    return {"caps": (w["cap"], z["cap"], q["cap"]), "openings": openings, "opening_proof": fri, "public_inputs": pis,
            "constants_sigmas_cap": cs["cap"]}
