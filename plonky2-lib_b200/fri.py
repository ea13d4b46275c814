"""plonky2::fri::prover on top of the C ABI (SURVEY.md 8f N1): `fri_proof` = commit phase + proof of work + query
phase, with the data-parallel work on the device and the serial Fiat-Shamir transcript (`Challenger`,
plonky2::iop::challenger) on the host.

Every layer tree stays resident (`gl_fri_layer_commit`); the 28 query rounds of a proof are answered with one
`gl_commit_open` per tree.  The Challenger's permutations run on the device (single states, or one
`gl_poseidon_duplex_chain` launch for a run of full input buffers; there is no CPU Poseidon in the product).  Upstream's `fri_proof_of_work` takes any satisfying witness found
by rayon `find_any`; here it is the smallest one (`gl_pow_grind`), which makes proofs deterministic.
"""
from __future__ import annotations

import dataclasses
from typing import List, Optional, Sequence

import numpy as np

from . import _native as N
from .host import Context, DeviceBuffer, FriConfig, GlPanic, PoseidonHash, _ctx, _h

P = 0xFFFFFFFF00000001
SPONGE_RATE, SPONGE_WIDTH = 8, 12


class Challenger:
    """plonky2::iop::challenger::Challenger<F, PoseidonHash>: overwrite-mode duplex sponge."""

    def __init__(self, ctx: Optional[Context] = None):
        self._ctx = _ctx(ctx)
        self.sponge_state = np.zeros(SPONGE_WIDTH, dtype=np.uint64)
        self.input_buffer: List[int] = []
        self.output_buffer: List[int] = []

    def observe_element(self, e: int):
        self.output_buffer = []           # any buffered outputs are now invalid
        self.input_buffer.append(int(e) % P)
        if len(self.input_buffer) == SPONGE_RATE:
            self._duplexing()

    def observe_elements(self, es):
        """Same transcript as element-by-element observation; runs of full input buffers become one
        gl_poseidon_duplex_chain call (one launch and one host round trip instead of one per permutation)."""
        es = np.asarray(es, dtype=np.uint64).reshape(-1) % np.uint64(P)
        if es.size == 0:
            return
        pending = np.concatenate([np.array(self.input_buffer, dtype=np.uint64), es])
        m = pending.size // SPONGE_RATE
        if m < 2:
            for e in es.tolist():
                self.observe_element(e)
            return
        chunks = np.ascontiguousarray(pending[: m * SPONGE_RATE])
        ctx = self._ctx
        ctx.check(ctx._lib.gl_poseidon_duplex_chain(ctx._h, self.sponge_state.ctypes.data, chunks.ctypes.data, m))
        rest = pending[m * SPONGE_RATE:]
        self.input_buffer = [int(x) for x in rest]
        # upstream: a duplexing refills output_buffer, the next observe_element clears it
        self.output_buffer = [] if rest.size else [int(x) for x in self.sponge_state[:SPONGE_RATE]]

    def observe_hash(self, h):
        self.observe_elements(h)

    def observe_cap(self, cap):
        self.observe_elements(cap)

    def observe_extension_elements(self, es):
        self.observe_elements(es)         # [a0, a1] per element, in order

    def get_challenge(self) -> int:
        if self.input_buffer or not self.output_buffer:
            self._duplexing()
        return self.output_buffer.pop()

    def get_n_challenges(self, n: int) -> List[int]:
        return [self.get_challenge() for _ in range(n)]

    def get_extension_challenge(self) -> List[int]:
        return self.get_n_challenges(2)

    def _duplexing(self):
        assert len(self.input_buffer) <= SPONGE_RATE
        for i, v in enumerate(self.input_buffer):
            self.sponge_state[i] = v
        self.input_buffer = []
        self.sponge_state = PoseidonHash.permute(self.sponge_state, ctx=self._ctx)
        self.output_buffer = [int(x) for x in self.sponge_state[:SPONGE_RATE]]


@dataclasses.dataclass
class FriParams:
    config: FriConfig
    degree_bits: int
    hiding: bool = False
    reduction_arity_bits: Sequence[int] = ()
    final_poly_times_x: bool = False      # GL_COMPAT_FRI_FINAL_POLY_TIMES_X: the pre-"remove multiplication by X" form

    @staticmethod
    def for_degree(config: FriConfig, degree_bits: int) -> "FriParams":
        ab = config.reduction_strategy.reduction_arity_bits(degree_bits, config.rate_bits, config.cap_height)
        return FriParams(config, degree_bits, False, tuple(ab))

    def lde_bits(self) -> int:
        return self.degree_bits + self.config.rate_bits


class FriLayerTree:
    """One resident layer tree of fri_committed_trees (MerkleTree over bit-reversed, arity-chunked values)."""

    def __init__(self, values_ext, length: int, arity_bits: int, cap_height: int, ctx: Context):
        """values_ext: DeviceBuffer holding `length` extension elements (natural order of their coset)."""
        import ctypes as C

        self._ctx, self.arity_bits, self.cap_height = ctx, arity_bits, cap_height
        self.num_leaves = length >> arity_bits
        cap_dev = DeviceBuffer((1 << cap_height, 4), ctx)
        h = C.c_void_p()
        ctx.check(ctx._lib.gl_fri_layer_commit(ctx._h, values_ext.ptr, length, arity_bits, cap_height,
                                               cap_dev.ptr, C.byref(h), N.GL_DEVICE))
        self.cap = cap_dev.to_host()
        cap_dev.free()
        self._h = h

    def open(self, leaf_indices):
        """(flattened evals [k][2 * arity], sibling paths [k][L][4])."""
        idx = _h(np.asarray(leaf_indices))
        k = idx.shape[0]
        L = (self.num_leaves.bit_length() - 1) - self.cap_height
        rows = np.empty((k, 2 << self.arity_bits), dtype=np.uint64)
        paths = np.empty((k, L, 4), dtype=np.uint64)
        self._ctx.check(self._ctx._lib.gl_commit_open(self._h, idx.ctypes.data, k, rows.ctypes.data, paths.ctypes.data, N.GL_HOST))
        return rows, paths

    def free(self):
        if getattr(self, "_h", None) and self._ctx._h:
            self._ctx._lib.gl_commit_free(self._h)
        self._h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def _to_device(x, ctx: Context) -> DeviceBuffer:
    if isinstance(x, DeviceBuffer):
        return x
    a = _h(x)
    return DeviceBuffer(a.shape, ctx).from_host(a)


def fri_committed_trees(coeffs_ext, values_ext, challenger: Challenger, fri_params: FriParams, ctx: Optional[Context] = None):
    """plonky2::fri::prover::fri_committed_trees -> (layer trees, final polynomial coefficients [len][2]).
    coeffs_ext / values_ext: [len][2] host arrays or DeviceBuffers; everything between the layers stays in HBM,
    only the caps (to the Challenger) and the final coefficients come back."""
    import ctypes as C

    ctx = _ctx(ctx)
    coeffs, values = _to_device(coeffs_ext, ctx), _to_device(values_ext, ctx)
    length = coeffs.shape[0]
    trees = []
    shift = 7  # F::MULTIPLICATIVE_GROUP_GENERATOR
    for arity_bits in fri_params.reduction_arity_bits:
        tree = FriLayerTree(values, length, arity_bits, fri_params.config.cap_height, ctx)
        challenger.observe_cap(tree.cap)
        trees.append(tree)
        beta = challenger.get_extension_challenge()
        shift = pow(shift, 1 << arity_bits, P)
        out_len = length >> arity_bits
        folded, nxt = DeviceBuffer((out_len, 2), ctx), DeviceBuffer((out_len, 2), ctx)
        b = (C.c_uint64 * 2)(int(beta[0]), int(beta[1]))
        ctx.check(ctx._lib.gl_fri_fold(ctx._h, coeffs.ptr, length, arity_bits, b, shift, folded.ptr, nxt.ptr, N.GL_DEVICE))
        if coeffs is not coeffs_ext:
            coeffs.free()
        if values is not values_ext:
            values.free()
        coeffs, values, length = folded, nxt, out_len
    # the coefficients being removed here are always zero
    final_len = length >> fri_params.config.rate_bits
    final = coeffs.to_host(final_len * 2).reshape(final_len, 2)
    if coeffs is not coeffs_ext:
        coeffs.free()
    if values is not values_ext:
        values.free()
    challenger.observe_extension_elements(final)
    return trees, final


def fri_proof_of_work(challenger: Challenger, config: FriConfig, ctx: Optional[Context] = None) -> int:
    import ctypes as C

    ctx = _ctx(ctx)
    min_leading_zeros = config.proof_of_work_bits + (64 - P.bit_length())
    state = challenger.sponge_state.copy()
    pos = len(challenger.input_buffer)
    for i, v in enumerate(challenger.input_buffer):
        state[i] = v
    s = (C.c_uint64 * 12)(*[int(x) for x in state])
    w = C.c_uint64()
    ctx.check(ctx._lib.gl_pow_grind(ctx._h, s, pos, min_leading_zeros, C.byref(w)))
    # recompute the response with the normal Challenger code, as upstream does
    challenger.observe_element(w.value)
    response = challenger.get_challenge()
    if min_leading_zeros and response >> (64 - min_leading_zeros):
        raise GlPanic(N.GL_E_STATE, "fri_proof_of_work: response does not have the required leading zeros")
    return w.value


def fri_prover_query_rounds(initial_batches, trees: Sequence[FriLayerTree], challenger: Challenger, n: int,
                            fri_params: FriParams):
    """28 x fri_prover_query_round; the challenger is only read here, so all x_index are drawn first and each
    tree answers every round with one gather."""
    rounds = fri_params.config.num_query_rounds
    xs = [challenger.get_challenge() % n for _ in range(rounds)]
    initial = [b.open(xs) for b in initial_batches]
    steps = []
    idx = list(xs)
    for tree in trees:
        idx = [x >> tree.arity_bits for x in idx]
        steps.append(tree.open(idx))
    out = []
    for q in range(rounds):
        out.append({
            "x_index": xs[q],
            "initial_trees_proof": [(rows[q], paths[q]) for rows, paths in initial],
            "steps": [{"evals": rows[q].reshape(-1, 2), "merkle_proof": paths[q]} for rows, paths in steps],
        })
    return out


def fri_proof(initial_batches, lde_polynomial_coeffs, lde_polynomial_values, challenger: Challenger,
              fri_params: FriParams, ctx: Optional[Context] = None) -> dict:
    """plonky2::fri::prover::fri_proof.  initial_batches: the resident PolynomialBatch oracles (their
    merkle_tree answers the initial openings)."""
    ctx = _ctx(ctx)
    n = int(lde_polynomial_values.shape[0])
    if int(lde_polynomial_coeffs.shape[0]) != n:
        raise GlPanic(N.GL_E_ARG, "assert_eq!(lde_polynomial_coeffs.len(), n)")
    trees, final_coeffs = fri_committed_trees(lde_polynomial_coeffs, lde_polynomial_values, challenger, fri_params, ctx)
    pow_witness = fri_proof_of_work(challenger, fri_params.config, ctx)
    query_round_proofs = fri_prover_query_rounds(initial_batches, trees, challenger, n, fri_params)
    proof = {
        "commit_phase_merkle_caps": [t.cap for t in trees],
        "query_round_proofs": query_round_proofs,
        "final_poly": final_coeffs,
        "pow_witness": pow_witness,
    }
    for t in trees:
        t.free()
    return proof


def fri_final_poly(oracles, batches, alpha, rate_bits: int, ctx: Optional[Context] = None, resident: bool = False):
    """reduce_polys_base / divide_by_linear / shift_poly over the resident commits, then lde + extension coset_fft:
    returns (lde_final_poly coefficients [N][2], lde_final_values [N][2]) as host arrays, or as DeviceBuffers
    when `resident` (what prove_openings uses: the polynomial never leaves HBM).
    batches: [(point (a0, a1), [(oracle_index, polynomial_index), ...]), ...]  (FriInstanceInfo.batches)."""
    import ctypes as C

    ctx = _ctx(ctx)
    nb = len(batches)
    total = sum(len(p) for _, p in batches)
    cb = (N.FriBatch * nb)()
    cp = (N.FriPoly * total)()
    at = 0
    for i, (point, polys) in enumerate(batches):
        cb[i].point[0], cb[i].point[1] = int(point[0]) % P, int(point[1]) % P
        cb[i].first_poly, cb[i].num_polys = at, len(polys)
        for oi, pi in polys:
            cp[at].oracle_index, cp[at].polynomial_index = oi, pi
            at += 1
    handles = (C.c_void_p * len(oracles))(*[o._h for o in oracles])
    n = 1 << oracles[0].degree_log
    lde = n << rate_bits
    al = (C.c_uint64 * 2)(int(alpha[0]) % P, int(alpha[1]) % P)
    if resident:
        coeffs, values = DeviceBuffer((lde, 2), ctx), DeviceBuffer((lde, 2), ctx)
        ctx.check(ctx._lib.gl_fri_final_poly(ctx._h, handles, len(oracles), cb, nb, cp, al, rate_bits, coeffs.ptr, values.ptr,
                                             N.GL_DEVICE))
        return coeffs, values
    coeffs = np.empty((lde, 2), dtype=np.uint64)
    values = np.empty((lde, 2), dtype=np.uint64)
    ctx.check(ctx._lib.gl_fri_final_poly(ctx._h, handles, len(oracles), cb, nb, cp, al, rate_bits,
                                         coeffs.ctypes.data, values.ctypes.data, N.GL_HOST))
    return coeffs, values


def _instance_arrays(batches):
    nb = len(batches)
    total = sum(len(p) for _, p in batches)
    cb = (N.FriBatch * nb)()
    cp = (N.FriPoly * total)()
    at = 0
    for i, (point, polys) in enumerate(batches):
        cb[i].point[0], cb[i].point[1] = int(point[0]) % P, int(point[1]) % P
        cb[i].first_poly, cb[i].num_polys = at, len(polys)
        for oi, pi in polys:
            cp[at].oracle_index, cp[at].polynomial_index = oi, pi
            at += 1
    return cb, nb, cp


def parse_flat_proof(flat: np.ndarray, oracle_columns: Sequence[int], fri_params: FriParams) -> dict:
    """The word stream gl_fri_prove writes (include/gl_b200.h) -> FriProof as the dict fri_proof returns."""
    cfg = fri_params.config
    lgN, h = fri_params.degree_bits + cfg.rate_bits, cfg.cap_height
    at = 0

    def take(k, shape=None):
        nonlocal at
        a = flat[at:at + k]
        at += k
        return a.reshape(shape) if shape else a

    caps = [take(4 << h, (1 << h, 4)).copy() for _ in fri_params.reduction_arity_bits]
    lg = lgN - sum(fri_params.reduction_arity_bits)
    final = take(2 << (lg - cfg.rate_bits), (-1, 2)).copy()
    pow_witness = int(take(1)[0])
    rounds = []
    for _ in range(cfg.num_query_rounds):
        x = int(take(1)[0])
        init = [(take(c).copy(), take(4 * (lgN - h), (lgN - h, 4)).copy()) for c in oracle_columns]
        steps, cur = [], lgN
        for ab in fri_params.reduction_arity_bits:
            ev = take(2 << ab, (-1, 2)).copy()
            L = cur - ab - h
            steps.append({"evals": ev, "merkle_proof": take(4 * L, (L, 4)).copy()})
            cur -= ab
        rounds.append({"x_index": x, "initial_trees_proof": init, "steps": steps})
    assert at == flat.shape[0]
    return {"commit_phase_merkle_caps": caps, "query_round_proofs": rounds, "final_poly": final, "pow_witness": pow_witness}


def c_params(fri_params: FriParams) -> N.FriParams:
    """gl_fri_params of FriParams (FriConfig, reduction_arity_bits, the GL_COMPAT_FRI_FINAL_POLY_TIMES_X form)."""
    cfg = fri_params.config
    prm = N.FriParams()
    prm.rate_bits, prm.cap_height, prm.proof_of_work_bits, prm.num_query_rounds = cfg.rate_bits, cfg.cap_height, cfg.proof_of_work_bits, cfg.num_query_rounds
    prm.num_reduction_layers = len(fri_params.reduction_arity_bits)
    for i, ab in enumerate(fri_params.reduction_arity_bits):
        prm.reduction_arity_bits[i] = ab
    prm.flags = N.GL_COMPAT_FRI_FINAL_POLY_TIMES_X if fri_params.final_poly_times_x else 0
    return prm


def prove_openings_device(oracles, batches, challenger: Challenger, fri_params: FriParams, ctx: Optional[Context] = None,
                          flat: bool = False):
    """PolynomialBatch::prove_openings through ONE C-ABI call (gl_fri_prove): the transcript runs on the device from the
    Challenger's current state and comes back advanced past the proof; three host synchronisations in total."""
    import ctypes as C

    ctx = _ctx(ctx)
    prm = c_params(fri_params)
    ch = N.Challenger()
    for i in range(12):
        ch.sponge_state[i] = int(challenger.sponge_state[i])
    for i, v in enumerate(challenger.input_buffer):
        ch.input_buffer[i] = int(v)
    for i, v in enumerate(challenger.output_buffer):
        ch.output_buffer[i] = int(v)
    ch.input_len, ch.output_len = len(challenger.input_buffer), len(challenger.output_buffer)
    cb, nb, cp = _instance_arrays(batches)
    handles = (C.c_void_p * len(oracles))(*[o._h for o in oracles])
    cols = (C.c_uint32 * len(oracles))(*[getattr(o, 'leaf_len', o.num_columns) for o in oracles])
    words = C.c_uint64(0)
    ctx.check(ctx._lib.gl_fri_proof_words(C.byref(prm), cols, len(oracles), fri_params.degree_bits, C.byref(words)))
    out = np.empty(words.value, dtype=np.uint64)
    ctx.check(ctx._lib.gl_fri_prove(ctx._h, handles, len(oracles), cb, nb, cp, C.byref(prm), C.byref(ch), out.ctypes.data,
                                    out.shape[0], C.byref(words)))
    challenger.sponge_state = np.array(list(ch.sponge_state), dtype=np.uint64)
    challenger.input_buffer = [int(ch.input_buffer[i]) for i in range(ch.input_len)]
    challenger.output_buffer = [int(ch.output_buffer[i]) for i in range(ch.output_len)]
    return out if flat else parse_flat_proof(out, [getattr(o, 'leaf_len', o.num_columns) for o in oracles], fri_params)


def opening_set(oracles, batches) -> list:
    """OpeningSet::new / FriOpenings: for every batch (point, [(oracle_index, polynomial_index), ...]) the values of its
    polynomials at its point, evaluated on the device from the resident coefficients (gl_commit_eval: one call per oracle
    and point)."""
    out = []
    for point, polys in batches:
        cache = {}
        vals = []
        for oi, pi in polys:
            if oi not in cache:
                cache[oi] = oracles[oi].eval_at(point)
            vals.append((int(cache[oi][pi][0]), int(cache[oi][pi][1])))
        out.append(vals)
    return out


def prove_openings(oracles, batches, challenger: Challenger, fri_params: FriParams, ctx: Optional[Context] = None) -> dict:
    """plonky2::fri::oracle::PolynomialBatch::prove_openings(instance, oracles, challenger, fri_params).

    The oracles may be sharded over a gl_group (host.ShardedPolynomialBatch): every rank holds all coefficients, so the
    FRI polynomial, the layer commits and the transcript run on the group's first local rank (every process of a
    multi-process group computes the same transcript), and the 28 x (row + path) initial-tree openings of the query phase
    are served by the ranks that own the leaves and exchanged over NCCL (gl_group_commit_open, SURVEY 8e)."""
    if ctx is None and oracles and hasattr(oracles[0], "group"):
        ctx = oracles[0].group.ctxs[0]
        if challenger._ctx is not ctx:
            challenger._ctx = ctx
    ctx = _ctx(ctx)
    alpha = challenger.get_extension_challenge()
    ctx.check(ctx._lib.gl_ctx_set_compat(ctx._h, N.GL_COMPAT_FRI_FINAL_POLY_TIMES_X if fri_params.final_poly_times_x else 0))
    try:
        lde_coeffs, lde_values = fri_final_poly(oracles, batches, alpha, fri_params.config.rate_bits, ctx, resident=True)
    finally:
        ctx.check(ctx._lib.gl_ctx_set_compat(ctx._h, 0))
    try:
        return fri_proof(oracles, lde_coeffs, lde_values, challenger, fri_params, ctx)
    finally:
        lde_coeffs.free()
        lde_values.free()
