"""plonky2::plonk::verifier on top of the C ABI: `data.verify(proof)` (42 call sites in the reference, e.g.
src/ecdsa/gadgets/ecdsa.rs:352, src/hash/keccak256.rs:249, src/smt/gadgets/process/mod.rs:84) for circuits built from the gates
gl_quotient_polys evaluates.

`verify_proof` is upstream's `verify` = `validate_proof_with_pis_shape` + `get_challenges` + `verify_with_challenges`: parse the
ProofWithPublicInputs bytes with every length taken from the circuit, replay the transcript, evaluate the vanishing polynomial
at zeta from the openings (exact extension-field integers, as upstream does it in Rust), check it against the quotient
chunks, then verify the opening proof (fri_verifier).  A failed check raises PlonkVerifyError.
"""
from __future__ import annotations

import dataclasses
from typing import List, Optional, Sequence

import numpy as np

from . import wire
from .fri import Challenger, FriParams
from .fri_verifier import (Ext, FriVerifyError, _e, _eadd, _einv, _emul, _epow, _esub, _root_of_unity, fri_challenges,
                           validate_fri_proof_shape, verify_fri_proof)
from .host import (GATE_CONSTANT, GATE_PUBLIC_INPUT, GATE_U32_INTERLEAVE, GATE_UNINTERLEAVE_TO_B32, GATE_UNINTERLEAVE_TO_U32,
                   Context, PoseidonHash, _ctx, opening_set_lengths)

P = 0xFFFFFFFF00000001
UNUSED_SELECTOR = 0xFFFFFFFF


class PlonkVerifyError(ValueError):
    """an `ensure!` of plonky2::plonk::verifier (or of the FRI verifier under it) failed, or the bytes are not a proof"""


@dataclasses.dataclass
class CommonData:
    """The part of CommonCircuitData the verifier reads.  circuit / gates / k_is as host.compute_quotient_polys takes them."""
    circuit: tuple
    gates: Sequence
    k_is: Sequence[int]
    fri_params: FriParams
    num_public_inputs: int


@dataclasses.dataclass
class VerifierData:
    """VerifierOnlyCircuitData: the cap of the constants / sigmas commit and the circuit digest."""
    constants_sigmas_cap: np.ndarray
    circuit_digest: Sequence[int]


def _base(x: int) -> Ext:
    return int(x) % P, 0


def _reduce(terms: Sequence[Ext], alpha: Ext) -> Ext:
    """plonk_common::reduce_with_powers: sum_j terms[j] alpha^j (Horner from the back)."""
    acc: Ext = (0, 0)
    for t in reversed(list(terms)):
        acc = _eadd(_emul(acc, alpha), t)
    return acc


def _bit_constraints(bits: Sequence[Ext]) -> List[Ext]:
    return [_emul(b, _esub(b, (1, 0))) for b in bits]


def _gate_constraints(kind: int, num_ops: int, w: Sequence[Ext], consts: Sequence[Ext], pih: Sequence[int]) -> List[Ext]:
    """Gate::eval_unfiltered of the six gates the device evaluates (csrc/quotient_kernels.cu); consts: the local constants
    after the selectors."""
    out: List[Ext] = []
    if kind == GATE_CONSTANT:                     # local_constants[i] - local_wires[i]
        out = [_esub(consts[i], w[i]) for i in range(num_ops)]
    elif kind == GATE_PUBLIC_INPUT:               # local_wires[i] - public_inputs_hash[i]
        out = [_esub(w[i], _base(pih[i])) for i in range(4)]
    elif kind == GATE_U32_INTERLEAVE:             # src/u32/gates/interleave_u32.rs:89-126, bits big-endian
        for i in range(num_ops):
            bits = w[2 * num_ops + 32 * i:2 * num_ops + 32 * (i + 1)]
            out.append(_esub(_reduce(bits[::-1], (2, 0)), w[2 * i]))
            out.append(_esub(_reduce(bits[::-1], (4, 0)), w[2 * i + 1]))
            out += _bit_constraints(bits)
    elif kind in (GATE_UNINTERLEAVE_TO_U32, GATE_UNINTERLEAVE_TO_B32):   # uninterleave_to_u32.rs:98-145, _b32.rs:101-149
        for i in range(num_ops):
            bits = w[3 * num_ops + 64 * i:3 * num_ops + 64 * (i + 1)]
            out.append(_esub(_reduce(bits[::-1], (2, 0)), w[3 * i]))
            ev: Ext = (0, 0)
            od: Ext = (0, 0)
            for j in range(32):
                coeff = (1 << (31 - j)) if kind == GATE_UNINTERLEAVE_TO_U32 else (1 << (2 * (31 - j)))
                ev = _eadd(ev, _emul((coeff, 0), bits[2 * j]))
                od = _eadd(od, _emul((coeff, 0), bits[2 * j + 1]))
            out.append(_esub(ev, w[3 * i + 1]))
            out.append(_esub(od, w[3 * i + 2]))
            out += _bit_constraints(bits)
    return out                                     # NoopGate: no constraint


def _compute_filter(gate_index: int, group_start: int, group_end: int, s: Ext, many_selectors: bool) -> Ext:
    """gate.rs compute_filter: prod_{i in group, i != gate_index} (i - s), times (UNUSED_SELECTOR - s) with several selectors."""
    f: Ext = (1, 0)
    for i in range(group_start, group_end):
        if i != gate_index:
            f = _emul(f, _esub(_base(i), s))
    if many_selectors:
        f = _emul(f, _esub(_base(UNUSED_SELECTOR), s))
    return f


def eval_vanishing_poly(circuit, gates, k_is, x: Ext, openings: dict, pih, betas, gammas, alphas) -> List[Ext]:
    """vanishing_poly.rs eval_vanishing_poly at the extension point x: the terms vanishing_z_1 ++ partial products ++ gate
    constraints (every gate filtered and added into shared slots), reduced with each alpha (reduce_with_powers_multi).
    openings: OpeningSet field -> [k][2] values at x (plonk_zs_next at g x)."""
    degree_bits, num_wires, R, num_constants, num_selectors, nch, qdf, num_gates = [int(v) for v in circuit]
    o = {f: [_e(v) for v in np.asarray(openings[f]).reshape(-1, 2)] for f in wire.OPENING_SET_FIELDS}
    consts, sigmas, w = o["constants"], o["plonk_sigmas"], o["wires"]
    zs, zs_next, pp = o["plonk_zs"], o["plonk_zs_next"], o["partial_products"]
    n = 1 << degree_bits
    chunks = -(-R // qdf)
    num_prods = chunks - 1
    # eval_l_0(n, x) = (x^n - 1) / (n (x - 1))
    l0 = _emul(_esub(_epow(x, n), (1, 0)), _einv(_emul(_base(n), _esub(x, (1, 0)))))
    terms = [_emul(l0, _esub(zs[c], (1, 0))) for c in range(nch)]
    for c in range(nch):                            # check_partial_products
        beta, gamma = _base(betas[c]), _base(gammas[c])
        for q in range(chunks):
            num: Ext = (1, 0)
            den: Ext = (1, 0)
            for j in range(q * qdf, min(R, (q + 1) * qdf)):
                num = _emul(num, _eadd(_eadd(w[j], _emul(beta, _emul(_base(k_is[j]), x))), gamma))
                den = _emul(den, _eadd(_eadd(w[j], _emul(beta, sigmas[j])), gamma))
            prev = zs[c] if q == 0 else pp[c * num_prods + q - 1]
            nxt = zs_next[c] if q == chunks - 1 else pp[c * num_prods + q]
            terms.append(_esub(_emul(prev, num), _emul(nxt, den)))
    slots: List[Ext] = []
    for gi, g in enumerate(list(gates)[:num_gates]):   # evaluate_gate_constraints
        kind, num_ops, sel, g0, g1 = [int(v) for v in tuple(g)[:5]]
        gc = _gate_constraints(kind, num_ops, w, consts[num_selectors:], pih)
        if not gc:
            continue
        f = _compute_filter(gi, g0, g1, consts[sel], num_selectors > 1)
        slots += [(0, 0)] * (len(gc) - len(slots))
        for j, v in enumerate(gc):
            slots[j] = _eadd(slots[j], _emul(f, v))
    terms += slots
    return [_reduce(terms, _base(a)) for a in alphas[:nch]]


def fri_instance(circuit, zeta: Ext, constants_sigmas_width: int):
    """get_fri_instance(zeta): every polynomial of [constants_sigmas, wires, zs_partial_products, quotient] at zeta, the Z
    polynomials at g * zeta."""
    lens = opening_set_lengths(circuit)
    nch = lens["plonk_zs"]
    widths = [constants_sigmas_width, lens["wires"], nch + lens["partial_products"], lens["quotient_polys"]]
    at_zeta = [(oi, pi) for oi, c in enumerate(widths) for pi in range(c)]
    g = _root_of_unity(int(circuit[0]))
    return [(zeta, at_zeta), (_emul(zeta, (g, 0)), [(2, pi) for pi in range(nch)])], widths


def verify_proof(proof_bytes: bytes, common: CommonData, verifier_data: VerifierData, ctx: Optional[Context] = None) -> bool:
    """plonky2::plonk::verifier::verify: True, or PlonkVerifyError naming the check that failed."""
    ctx = _ctx(ctx)
    circuit, params = tuple(int(v) for v in common.circuit), common.fri_params
    degree_bits, nch, qdf = circuit[0], circuit[5], circuit[6]
    cfg = params.config
    if params.degree_bits != degree_bits:
        raise PlonkVerifyError("the FRI parameters are for another degree")
    lens = opening_set_lengths(circuit)
    _, widths = fri_instance(circuit, (0, 0), circuit[3] + circuit[2])
    # 1-2. parse with every length from the circuit, then the exact shape
    try:
        caps, openings, fp, public_inputs = wire.proof_with_public_inputs_from_bytes(
            proof_bytes, lens, widths, degree_bits, cfg.rate_bits, cfg.cap_height, params.reduction_arity_bits, cfg.num_query_rounds)
    except wire.WireError as e:
        raise PlonkVerifyError(f"malformed proof: {e}")
    if len(public_inputs) != common.num_public_inputs:
        raise PlonkVerifyError("wrong number of public inputs")
    cs_cap = np.asarray(verifier_data.constants_sigmas_cap, dtype=np.uint64)
    initial_caps = [cs_cap, caps[0], caps[1], caps[2]]
    # 3. the transcript (get_challenges)
    pih = PoseidonHash.hash_no_pad(np.asarray(public_inputs, dtype=np.uint64), ctx=ctx)
    ch = Challenger(ctx)
    ch.observe_hash(np.asarray(verifier_data.circuit_digest, dtype=np.uint64))
    ch.observe_hash(pih)
    ch.observe_cap(caps[0])
    betas, gammas = ch.get_n_challenges(nch), ch.get_n_challenges(nch)
    ch.observe_cap(caps[1])
    alphas = ch.get_n_challenges(nch)
    ch.observe_cap(caps[2])
    zeta = tuple(ch.get_extension_challenge())
    instance, _ = fri_instance(circuit, zeta, widths[0])
    batch_zeta = np.concatenate([openings[f] for f in ("constants", "plonk_sigmas", "wires", "plonk_zs", "partial_products",
                                                       "quotient_polys")])
    ch.observe_extension_elements(batch_zeta)
    ch.observe_extension_elements(openings["plonk_zs_next"])
    try:
        validate_fri_proof_shape(fp, instance, initial_caps, params, oracle_columns=widths)
        fri_ch = fri_challenges(ch, fp, degree_bits, params)
    except FriVerifyError as e:
        raise PlonkVerifyError(str(e))
    # 4-5. vanishing(zeta) == Z_H(zeta) * sum_i t_i(zeta) zeta^(i n), per challenge
    vanishing = eval_vanishing_poly(circuit, common.gates, common.k_is, zeta, openings, pih, betas, gammas, alphas)
    zeta_n = _epow(zeta, 1 << degree_bits)
    z_h = _esub(zeta_n, (1, 0))
    quotient = [_e(v) for v in openings["quotient_polys"]]
    for c in range(nch):
        if vanishing[c] != _emul(z_h, _reduce(quotient[c * qdf:(c + 1) * qdf], zeta_n)):
            raise PlonkVerifyError("Mismatch between evaluation and opening of quotient polynomial")
    # 6. the opening proof
    batches = [[_e(v) for v in batch_zeta], [_e(v) for v in openings["plonk_zs_next"]]]
    try:
        verify_fri_proof(instance, batches, fri_ch, initial_caps, fp, params, ctx)
    except FriVerifyError as e:
        raise PlonkVerifyError(str(e))
    return True
