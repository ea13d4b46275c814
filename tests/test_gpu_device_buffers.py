"""Every C-ABI entry point with a `space` argument, in both spaces and at the pointer alignments a caller can produce.

GL_HOST buffers are staged into pool blocks; GL_DEVICE pointers go to the kernels as they are, and those read and write
16-byte pairs (Poseidon states, digests, NTT outputs) or go through TMA descriptors.  One table, one row per entry point:
each row runs its call with
  (a) host numpy arrays, (b) host views at an 8-byte offset, (c) whole device tensors, (d) device views at a 16-byte
      offset (`buf[2:]`, inputs and outputs),
and every result must be bit-identical to the oracle (or, where the oracle has no restatement, to the host form).  Around
that: const inputs are byte-identical after the call, nothing but an output's own bytes changes (sentinel words on both
sides of every offset view), a device view at an 8-byte offset (`buf[1:]`) is refused with GL_E_ARG naming the argument
and leaves the buffer alone, and the same ctx then still computes the right answer.

The CPU test at the end keeps the table and the library's alignment guard complete: every header function with an
`int space` parameter has a row, and its body checks every device buffer argument the row passes."""
import ctypes as C
import dataclasses
import importlib
import os
import re
from typing import Callable, Dict, Optional

import numpy as np
import pytest

from conftest import P, adversarial_columns

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GL_HOST, GL_DEVICE, GL_E_ARG = 0, 1, 1

# The device buffer arguments of every entry point with a `space` parameter, by their names in include/gl_b200.h.
# gl_group_commit_open takes host buffers only and refuses GL_DEVICE outright.
DEVICE_ARGS = {
    "gl_poseidon_permute_batch": ("states",),
    "gl_poseidon_two_to_one_batch": ("l", "r", "out"),
    "gl_poseidon_hash_no_pad_batch": ("in", "out"),
    "gl_smt_leaf_hash_batch": ("keys", "values", "out"),
    "gl_smt_verify_process_batch": ("proofs", "sib_pool", "sib_off", "status"),
    "gl_smt_build": ("keys", "values", "root_out", "nodes_out", "leaf_hashes_out"),
    "gl_smt_set_proofs": ("keys", "values", "proofs_out", "sib_pool_out", "sib_off_out"),
    "gl_smt_find_batch": ("keys", "values", "queries", "proofs_out", "sib_pool_out", "sib_off_out"),
    "gl_merkle_build": ("leaves", "digests_out", "cap_out"),
    "gl_merkle_verify_batch": ("leaves", "leaf_indices", "paths", "cap", "ok"),
    "gl_fft_batch": ("data",),
    "gl_ifft_batch": ("data",),
    "gl_coset_fft_batch": ("data",),
    "gl_coset_ifft_batch": ("data",),
    "gl_commit_from_values": ("values", "coeffs_out", "cap_out"),
    "gl_commit_from_coeffs": ("coeffs", "cap_out"),
    "gl_commit_from_values_ex": ("values", "coeffs_out", "cap_out"),
    "gl_commit_from_coeffs_ex": ("coeffs", "cap_out"),
    "gl_commit_add_coeffs": ("coeffs",),
    "gl_commit_finish": ("cap_out",),
    "gl_commit_coeffs": ("coeffs_out",),
    "gl_commit_eval": ("values_out",),
    "gl_commit_download": ("leaves_out", "digests_out"),
    "gl_commit_open": ("leaf_indices", "rows_out", "paths_out"),
    "gl_commit_get_lde_values": ("indices", "rows_out"),
    "gl_group_commit_from_values": ("values", "coeffs_out", "cap_out"),
    "gl_group_commit_from_coeffs": ("coeffs", "cap_out"),
    "gl_group_commit_open": (),
    "gl_fri_layer_tree": ("values_ext", "digests_out", "cap_out"),
    "gl_fri_layer_commit": ("values_ext", "cap_out"),
    "gl_fri_fold": ("coeffs_ext", "folded_coeffs_out", "next_values_out"),
    "gl_fri_final_poly": ("lde_coeffs_out", "lde_values_out"),
    "gl_quotient_polys": ("chunks_out",),
    "gl_permutation_zs": ("zs_partial_products_out",),
    "gl_prove": ("wires",),
}

SENT = np.uint64(0xA5A5F00DDEADBEEF)   # sentinel word around every offset view and in every output before the call
PAD = 2                                 # sentinel words after an offset view
FORMS = ("host", "host8", "dev", "dev16")
LEAD = {"host": 0, "dev": 0, "host8": 1, "dev16": 2, "dev8": 1}   # words before the view


# ---- the runner ---------------------------------------------------------------------------------------------------------
@dataclasses.dataclass
class Case:
    """One call of a row.  ins: const inputs (name -> u64 words); inout: inputs the call overwrites with its result;
    outs: name -> output bytes; call(space, ptrs, views) runs it (raising GlPanic on an error code) and returns extra
    host-side results; want: name -> expected result (anything numpy views as bytes), the rest is compared with the host
    form; post: name -> normalisation of a result's bytes before comparing (unordered outputs)."""
    ins: Dict[str, np.ndarray]
    outs: Dict[str, int]
    call: Callable
    want: Dict[str, object] = dataclasses.field(default_factory=dict)
    inout: tuple = ()
    post: Dict[str, Callable] = dataclasses.field(default_factory=dict)
    check: Optional[Callable] = None
    done: Optional[Callable] = None


def _bytes(x) -> np.ndarray:
    return np.ascontiguousarray(x).view(np.uint8).reshape(-1)


def _alloc(form, words, init, device):
    lead = LEAD[form]
    total = words + (lead + PAD if lead else 0)
    base = np.full(max(total, 1), SENT, dtype=np.uint64)
    if init is not None:
        base[lead:lead + words] = init
    if form.startswith("dev"):
        import torch

        t = torch.from_numpy(base.view(np.int64).copy()).to(device)
        view = t[lead:lead + words]
        ptr = view.data_ptr() if words else t.data_ptr() + 8 * lead
        return t, view, ptr, base
    view = base[lead:lead + words]
    ptr = base.ctypes.data + 8 * lead      # also for an empty view, whose own address numpy does not keep
    return base, view, ptr, base.copy()


def _np(base) -> np.ndarray:
    return base if isinstance(base, np.ndarray) else base.cpu().numpy().view(np.uint64)


def _run(ctx, case: Case, form: str, bad: Optional[str] = None):
    """The call with every buffer in `form` (the argument `bad` as an 8-byte-offset device view); returns name -> bytes."""
    device = f"cuda:{ctx.device}"
    bufs = {}
    for name, data in case.ins.items():
        bufs[name] = _alloc("dev8" if name == bad else form, data.size, data, device)
    for name, nb in case.outs.items():
        bufs[name] = _alloc("dev8" if name == bad else form, -(-nb // 8), None, device)
    for name, (_, _, ptr, _) in bufs.items():
        f = "dev8" if name == bad else form
        if f in ("host8", "dev8"):
            assert ptr % 16 == 8, (name, f)
        elif f == "dev16":
            assert ptr % 16 == 0 and ptr % 256 != 0, (name, f)
    space = GL_DEVICE if form.startswith("dev") else GL_HOST
    ptrs = {k: b[2] for k, b in bufs.items()}
    views = {k: b[1] for k, b in bufs.items()}
    try:
        extra = case.call(space, ptrs, views) or {}
    finally:
        if bad is not None:   # refused before any copy or launch: the offending buffer is exactly as it was
            base, _, _, before = bufs[bad]
            assert np.array_equal(_np(base), before), f"{bad} was written to"
    out = {}
    for name, (base, _, _, before) in bufs.items():
        lead = LEAD["dev8" if name == bad else form]
        after = _bytes(_np(base))
        ref = _bytes(before)
        nb = case.outs.get(name, case.ins[name].nbytes if name in case.ins else 0)
        lo, hi = 8 * lead, 8 * lead + nb
        if name in case.outs or name in case.inout:
            out[name] = after[lo:hi].copy()
            assert np.array_equal(after[:lo], ref[:lo]) and np.array_equal(after[hi:], ref[hi:]), \
                f"{form}: bytes outside {name} changed"
        else:
            assert np.array_equal(after, ref), f"{form}: const input {name} changed"
    for k, v in extra.items():
        out[k] = _bytes(v)
    for k, f in case.post.items():
        out[k] = f(out[k])
    return out


def _same(got, want, what):
    assert got.shape == want.shape and np.array_equal(got, want), what


def _exercise(ctx, glb, case: Case, entries):
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    args = set(case.ins) | set(case.outs)
    assert args == {a for e in entries for a in DEVICE_ARGS[e]}, "the row passes other buffers than DEVICE_ARGS lists"
    try:
        res = {f: _run(ctx, case, f) for f in FORMS}
        ref = dict(res["host"])
        for k, w in case.want.items():
            w = _bytes(w)
            if k in case.post:
                w = case.post[k](w)
            _same(ref[k], w, f"host result {k} differs from the oracle")
        if case.check:
            case.check(res["host"])
        for f in FORMS[1:]:
            assert set(res[f]) == set(ref)
            for k in ref:
                _same(res[f][k], ref[k], f"{f}: {k} differs")
        for name in sorted(args):
            nb = case.ins[name].nbytes if name in case.ins else case.outs[name]
            if nb < 16:
                continue
            with pytest.raises(glb.GlPanic) as e:
                _run(ctx, case, "dev", bad=name)
            assert e.value.code == GL_E_ARG and re.search(rf": {re.escape(name)}\b", str(e.value)), str(e.value)
        again = _run(ctx, case, "dev16")
        for k in ref:
            _same(again[k], ref[k], f"after the refusals: {k} differs")
    finally:
        if case.done:
            case.done()


# ---- inputs --------------------------------------------------------------------------------------------------------------
NONCANON = np.array([2**64 - 1, P, P + 1, P + 2, P + 0x7FFF, 2**64 - 2, P - 1, 0, 1, 2**32 - 1, 2**32], dtype=np.uint64)


def _words(rng, n):
    """Seeded field words with the non-canonical encodings (2^64 - 1, p, p + i) at both ends."""
    x = rng.integers(0, P, n, dtype=np.uint64) if n else np.zeros(0, dtype=np.uint64)
    k = min(n, NONCANON.size)
    x[:k] = NONCANON[:k]
    if n > 2 * k:
        x[n - k:] = NONCANON[:k][::-1]
    return x


def _columns(rng, c, n):
    """[c][n]: adversarial_columns first, the rest seeded words with non-canonical ones."""
    a = np.stack([_words(rng, n) for _ in range(c)])
    adv = adversarial_columns(n)
    k = min(c - 1, adv.shape[0])
    a[1:1 + k] = adv[:k]
    a[0, : min(n, NONCANON.size)] = NONCANON[: min(n, NONCANON.size)]
    return np.ascontiguousarray(a)


def _rev(x, bits):
    return int(format(x, f"0{bits}b")[::-1], 2) if bits else 0


def _sorted_rows(width):
    def f(b):
        rows = b.view(np.uint64).reshape(-1, width)
        return _bytes(rows[np.lexsort(rows.T[::-1])])
    return f


# ---- rows ----------------------------------------------------------------------------------------------------------------
def row_permute(ctx, glb, o, m):
    s = _words(np.random.default_rng(m), 12 * m)
    return Case({"states": s}, {}, inout=("states",), want={"states": o.permute_batch(s.reshape(m, 12))},
                call=lambda sp, p, v: ctx.check(ctx._lib.gl_poseidon_permute_batch(ctx._h, p["states"], m, sp)))


def row_two_to_one(ctx, glb, o, m):
    rng = np.random.default_rng(m + 1)
    l, r = _words(rng, 4 * m), _words(rng, 4 * m)[::-1].copy()
    return Case({"l": l, "r": r}, {"out": 32 * m}, want={"out": o.two_to_one_batch(l.reshape(m, 4), r.reshape(m, 4))},
                call=lambda sp, p, v: ctx.check(ctx._lib.gl_poseidon_two_to_one_batch(ctx._h, p["l"], p["r"], p["out"], m, sp)))


def row_hash_no_pad(ctx, glb, o, m, ln):
    x = _words(np.random.default_rng(m * 16 + ln), m * ln)
    return Case({"in": x}, {"out": 32 * m}, want={"out": o.hash_no_pad_batch(x.reshape(m, ln))},
                call=lambda sp, p, v: ctx.check(ctx._lib.gl_poseidon_hash_no_pad_batch(ctx._h, p["in"], ln, m, p["out"], sp)))


def row_smt_leaf_hash(ctx, glb, o, m):
    rng = np.random.default_rng(m + 2)
    k, val = _words(rng, 4 * m), _words(rng, 4 * m)
    want = np.stack([o.smt_leaf_hash(k[4 * i:4 * i + 4], val[4 * i:4 * i + 4]) for i in range(m)])
    return Case({"keys": k, "values": val}, {"out": 32 * m}, want={"out": want},
                call=lambda sp, p, v: ctx.check(ctx._lib.gl_smt_leaf_hash_batch(ctx._h, p["keys"], p["values"], p["out"], m, sp)))


def _smt_keys(rng, m, repeats=False):
    k = rng.integers(0, P, (m, 4), dtype=np.uint64)
    v = rng.integers(1, P, (m, 4), dtype=np.uint64)
    if repeats:                      # updates, removals (zero values) and removals of absent keys
        k[m // 2: m // 2 + m // 8] = k[: m // 8]
        v[m // 3: m // 3 + m // 10] = 0
    return np.ascontiguousarray(k.reshape(-1)), np.ascontiguousarray(v.reshape(-1))


def _smt_oracle_root(o, k, v):
    t = o.Smt()
    for i in range(k.size // 4):
        t.set(k[4 * i:4 * i + 4], v[4 * i:4 * i + 4])
    return t.root()


def row_smt_verify(ctx, glb, o):
    m = 64
    k, v = _smt_keys(np.random.default_rng(3), m, repeats=True)
    hdr, pool, off = glb.host.smt_set_proofs(k, v, ctx=ctx)
    hdr = hdr.copy()
    hdr["new_root"][5, 0] ^= np.uint64(1)          # one proof that must fail
    proofs = np.ascontiguousarray(hdr).view(np.uint64).copy()

    def check(res):
        st = res["status"].view(np.int32)
        assert st[5] != 0 and not np.delete(st, 5).any()

    return Case({"proofs": proofs, "sib_pool": pool.reshape(-1).copy(), "sib_off": off.copy()}, {"status": 4 * m}, check=check,
                call=lambda sp, p, vw: ctx.check(ctx._lib.gl_smt_verify_process_batch(ctx._h, p["proofs"], p["sib_pool"], p["sib_off"],
                                                                                     m, p["status"], sp)))


def row_smt_build(ctx, glb, o, m):
    k, v = _smt_keys(np.random.default_rng(m), m)
    cap = 4 * m + 64
    cnt = C.c_uint64(0)

    def call(sp, p, vw):
        ctx.check(ctx._lib.gl_smt_build(ctx._h, p["keys"], p["values"], m, p["root_out"], p["nodes_out"], cap, C.byref(cnt),
                                        p["leaf_hashes_out"], sp))
        return {"num_nodes": np.array([cnt.value], dtype=np.uint64)}

    leaf = np.stack([o.smt_leaf_hash(k[4 * i:4 * i + 4], v[4 * i:4 * i + 4]) for i in range(m)])
    return Case({"keys": k, "values": v}, {"root_out": 32, "nodes_out": 96 * cap, "leaf_hashes_out": 32 * m}, call=call,
                want={"root_out": _smt_oracle_root(o, k, v), "leaf_hashes_out": leaf}, post={"nodes_out": _sorted_rows(12)})


def row_smt_set_proofs(ctx, glb, o):
    m = 300
    k, v = _smt_keys(np.random.default_rng(5), m, repeats=True)
    cap = 64 * m
    tot = C.c_uint64(0)

    def call(sp, p, vw):
        ctx.check(ctx._lib.gl_smt_set_proofs(ctx._h, p["keys"], p["values"], m, p["proofs_out"], p["sib_pool_out"], cap,
                                             p["sib_off_out"], C.byref(tot), sp))
        return {"num_siblings": np.array([tot.value], dtype=np.uint64)}

    root = _smt_oracle_root(o, k, v)

    def check(res):
        hdr = res["proofs_out"].view(glb.host.SMT_HDR_DTYPE)
        assert np.array_equal(hdr["new_root"][-1], root)
        assert 0 < res["num_siblings"].view(np.uint64)[0] <= cap

    return Case({"keys": k, "values": v}, {"proofs_out": 200 * m, "sib_pool_out": 32 * cap, "sib_off_out": 8 * (m + 1)},
                call=call, check=check)


def row_smt_find(ctx, glb, o):
    m, nq = 300, 77
    rng = np.random.default_rng(6)
    k, v = _smt_keys(rng, m, repeats=True)
    q = rng.integers(0, P, (nq, 4), dtype=np.uint64)
    q[::3] = k.reshape(m, 4)[: len(q[::3]) * 7: 7]             # every third query is a key that was set
    q = np.ascontiguousarray(q.reshape(-1))
    cap = 64 * nq
    tot = C.c_uint64(0)

    def call(sp, p, vw):
        ctx.check(ctx._lib.gl_smt_find_batch(ctx._h, p["keys"], p["values"], m, p["queries"], nq, p["proofs_out"],
                                             p["sib_pool_out"], cap, p["sib_off_out"], C.byref(tot), sp))
        return {"num_siblings": np.array([tot.value], dtype=np.uint64)}

    t = o.Smt()
    for i in range(m):
        t.set(k[4 * i:4 * i + 4], v[4 * i:4 * i + 4])
    found = np.array([t.find(q[4 * i:4 * i + 4])["found"] for i in range(nq)])

    def check(res):
        hdr = res["proofs_out"].view(glb.host.SMT_INCLUSION_DTYPE)
        assert np.array_equal(hdr["found"] != 0, found) and found.any() and not found.all()

    return Case({"keys": k, "values": v, "queries": q},
                {"proofs_out": 168 * nq, "sib_pool_out": 32 * cap, "sib_off_out": 8 * (nq + 1)}, call=call, check=check)


def row_merkle_build(ctx, glb, o, leaf_len):
    nl, h = 512, 2
    leaves = _words(np.random.default_rng(leaf_len), nl * leaf_len)
    dg, cp = o.merkle_tree(leaves.reshape(nl, leaf_len), h)
    return Case({"leaves": leaves}, {"digests_out": dg.nbytes, "cap_out": cp.nbytes}, want={"digests_out": dg, "cap_out": cp},
                call=lambda sp, p, v: ctx.check(ctx._lib.gl_merkle_build(ctx._h, p["leaves"], nl, leaf_len, h, p["digests_out"],
                                                                         p["cap_out"], sp)))


def row_merkle_verify(ctx, glb, o):
    nl, ll, h, k = 256, 6, 2, 5
    leaves = _words(np.random.default_rng(9), nl * ll).reshape(nl, ll)
    dg, cp = o.merkle_tree(leaves, h)
    idx = np.array([0, 77, 128, 255, 3], dtype=np.uint64)
    paths = np.stack([o.merkle_prove(dg, nl, h, int(i)) for i in idx])
    rows = leaves[idx].copy()
    rows[2, 1] ^= np.uint64(4)                                # one proof that must fail
    L = paths.shape[1]
    return Case({"leaves": rows.reshape(-1), "leaf_indices": idx, "paths": paths.reshape(-1), "cap": cp.reshape(-1)},
                {"ok": 4 * k}, want={"ok": np.array([1, 1, 0, 1, 1], dtype=np.int32)},
                call=lambda sp, p, v: ctx.check(ctx._lib.gl_merkle_verify_batch(ctx._h, p["leaves"], ll, p["leaf_indices"], p["paths"],
                                                                                L, p["cap"], h, k, p["ok"], sp)))


FFT_SHIFT = 7


def row_fft(ctx, glb, o, entry, lg):
    n = 1 << lg
    c = 2 if lg >= 20 else (5 if n >= 8 else 3)
    a = _columns(np.random.default_rng(lg * 8 + len(entry)), c, n)
    f = {"gl_fft_batch": o.fft, "gl_ifft_batch": o.ifft, "gl_coset_fft_batch": lambda x: o.coset_fft(x, FFT_SHIFT),
         "gl_coset_ifft_batch": lambda x: o.coset_ifft(x, FFT_SHIFT)}[entry]
    want = np.stack([f(col) for col in a])
    fn = getattr(ctx._lib, entry)
    if "coset" in entry:
        call = lambda sp, p, v: ctx.check(fn(ctx._h, p["data"], lg, c, FFT_SHIFT, sp))
    else:
        call = lambda sp, p, v: ctx.check(fn(ctx._h, p["data"], lg, c, sp))
    return Case({"data": a.reshape(-1)}, {}, inout=("data",), want={"data": want}, call=call)


def _commit_geometry(lg):
    return (2 if lg >= 20 else 3), (1 if lg >= 20 else 2), min(2, lg + (1 if lg >= 20 else 2))   # c, rate_bits, cap_height


def row_commit(ctx, glb, o, entry, lg):
    n = 1 << lg
    c, rb, h = _commit_geometry(lg)
    a = _columns(np.random.default_rng(100 + lg), c, n)
    values = entry.startswith("gl_commit_from_values")
    blinding = entry.endswith("_ex")
    w = (o.commit_from_values if values else o.commit_from_coeffs)(a, rb, h, want_leaves=False)
    lib = ctx._lib
    arg = "values" if values else "coeffs"
    outs = {"cap_out": 32 << h}
    want = {} if blinding else {"cap_out": w["cap"]}
    if values:
        outs["coeffs_out"] = a.nbytes
        want["coeffs_out"] = w["coeffs"]

    def call(sp, p, v):
        hd = C.c_void_p()
        if blinding:
            ctx.set_salt_seed(0xB17D)
        if entry == "gl_commit_from_values":
            rc = lib.gl_commit_from_values(ctx._h, p[arg], lg, c, rb, h, p["coeffs_out"], p["cap_out"], C.byref(hd), sp)
        elif entry == "gl_commit_from_coeffs":
            rc = lib.gl_commit_from_coeffs(ctx._h, p[arg], lg, c, rb, h, p["cap_out"], C.byref(hd), sp)
        elif entry == "gl_commit_from_values_ex":
            rc = lib.gl_commit_from_values_ex(ctx._h, p[arg], None, lg, c, rb, 1, h, p["coeffs_out"], None, p["cap_out"],
                                              C.byref(hd), sp)
        else:
            rc = lib.gl_commit_from_coeffs_ex(ctx._h, p[arg], None, lg, c, rb, 1, h, p["cap_out"], C.byref(hd), sp)
        if hd.value:
            lib.gl_commit_free(hd)
        ctx.check(rc)

    return Case({arg: a.reshape(-1)}, outs, want=want, call=call)


def row_commit_stream(ctx, glb, o):
    """gl_commit_begin_ex / add_coeffs / finish with the blocks handed over as device views at column offsets."""
    lg, c, rb, h = 4, 13, 2, 2
    n = 1 << lg
    a = _columns(np.random.default_rng(13), c, n)
    w = o.commit_from_coeffs(a, rb, h, want_leaves=False)
    lib = ctx._lib

    def call(sp, p, v):
        hd = C.c_void_p()
        ctx.check(lib.gl_commit_begin_ex(ctx._h, lg, c, rb, h, 1, C.byref(hd)))   # GL_COMMIT_STREAM_HASH
        try:
            for col0, nc in ((0, 5), (5, 4), (9, 4)):
                ctx.check(lib.gl_commit_add_coeffs(hd, col0, nc, p["coeffs"] + 8 * col0 * n, sp))
            ctx.check(lib.gl_commit_finish(hd, p["cap_out"], sp))
        finally:
            lib.gl_commit_free(hd)

    return Case({"coeffs": a.reshape(-1)}, {"cap_out": 32 << h}, want={"cap_out": w["cap"]}, call=call)


def _resident(ctx, glb, o, seed):
    lg, c, rb, h = 6, 5, 2, 2
    a = _columns(np.random.default_rng(seed), c, 1 << lg)
    b = glb.PolynomialBatch.from_values(a, rb, False, h, ctx=ctx)
    return b, o.commit_from_values(a, rb, h), (lg, c, rb, h)


def row_commit_reads(ctx, glb, o):
    """gl_commit_coeffs, gl_commit_eval and gl_commit_download of one resident commit."""
    b, w, (lg, c, rb, h) = _resident(ctx, glb, o, 21)
    pt = (C.c_uint64 * 2)(0x1234567890ABCDEF, P + 5)
    ev = np.array([o.eval_base_poly_at_ext(w["coeffs"][j], (0x1234567890ABCDEF, 5)) for j in range(c)], dtype=np.uint64)
    lib = ctx._lib

    def call(sp, p, v):
        ctx.check(lib.gl_commit_coeffs(b._h, p["coeffs_out"], sp))
        ctx.check(lib.gl_commit_eval(b._h, pt, p["values_out"], sp))
        ctx.check(lib.gl_commit_download(b._h, p["leaves_out"], p["digests_out"], sp))

    return Case({}, {"coeffs_out": w["coeffs"].nbytes, "values_out": 16 * c, "leaves_out": w["leaves"].nbytes,
                     "digests_out": w["digests"].nbytes}, call=call, done=b.free,
                want={"coeffs_out": w["coeffs"], "values_out": ev, "leaves_out": w["leaves"], "digests_out": w["digests"]})


def row_commit_open(ctx, glb, o):
    b, w, (lg, c, rb, h) = _resident(ctx, glb, o, 22)
    N = 1 << (lg + rb)
    idx = np.array([N - 1, 0, 77], dtype=np.uint64)
    paths = np.stack([o.merkle_prove(w["digests"], N, h, int(i)) for i in idx])
    return Case({"leaf_indices": idx}, {"rows_out": 8 * c * idx.size, "paths_out": paths.nbytes}, done=b.free,
                want={"rows_out": w["leaves"][idx], "paths_out": paths},
                call=lambda sp, p, v: ctx.check(ctx._lib.gl_commit_open(b._h, p["leaf_indices"], idx.size, p["rows_out"],
                                                                        p["paths_out"], sp)))


def row_commit_lde_values(ctx, glb, o):
    b, w, (lg, c, rb, h) = _resident(ctx, glb, o, 23)
    lgN, step = lg + rb, 2
    idx = np.array([0, 5, 17], dtype=np.uint64)
    rows = w["leaves"][[_rev(int(i) * step, lgN) for i in idx]]
    return Case({"indices": idx}, {"rows_out": rows.nbytes}, done=b.free, want={"rows_out": rows},
                call=lambda sp, p, v: ctx.check(ctx._lib.gl_commit_get_lde_values(b._h, p["indices"], idx.size, step, p["rows_out"],
                                                                                  sp)))


def row_fri_layer_tree(ctx, glb, o):
    ln, ab, h = 512, 3, 2
    x = _words(np.random.default_rng(31), 2 * ln)
    _, dg, cp = o.fri_layer_tree(x.reshape(ln, 2), ab, h)
    return Case({"values_ext": x}, {"digests_out": dg.nbytes, "cap_out": cp.nbytes}, want={"digests_out": dg, "cap_out": cp},
                call=lambda sp, p, v: ctx.check(ctx._lib.gl_fri_layer_tree(ctx._h, p["values_ext"], ln, ab, h, p["digests_out"],
                                                                           p["cap_out"], sp)))


def row_fri_layer_commit(ctx, glb, o):
    ln, ab, h = 512, 2, 3
    x = _words(np.random.default_rng(32), 2 * ln)
    _, _, cp = o.fri_layer_tree(x.reshape(ln, 2), ab, h)

    def call(sp, p, v):
        hd = C.c_void_p()
        rc = ctx._lib.gl_fri_layer_commit(ctx._h, p["values_ext"], ln, ab, h, p["cap_out"], C.byref(hd), sp)
        if hd.value:
            ctx._lib.gl_commit_free(hd)
        ctx.check(rc)

    return Case({"values_ext": x}, {"cap_out": cp.nbytes}, want={"cap_out": cp}, call=call)


def row_fri_fold(ctx, glb, o):
    ln, ab, shift = 512, 2, 7
    x = _words(np.random.default_rng(33), 2 * ln)
    beta = np.array([0xDEADBEEF12345, P - 3], dtype=np.uint64)
    folded = o.fri_fold(x.reshape(ln, 2), ab, beta)
    nxt = o.ext_coset_fft(folded, shift)
    b = (C.c_uint64 * 2)(*[int(t) for t in beta])
    return Case({"coeffs_ext": x}, {"folded_coeffs_out": folded.nbytes, "next_values_out": nxt.nbytes},
                want={"folded_coeffs_out": folded, "next_values_out": nxt},
                call=lambda sp, p, v: ctx.check(ctx._lib.gl_fri_fold(ctx._h, p["coeffs_ext"], ln, ab, b, shift, p["folded_coeffs_out"],
                                                                     p["next_values_out"], sp)))


def row_fri_final_poly(ctx, glb, o):
    lg, rb = 5, 2
    rng = np.random.default_rng(34)
    bs = [glb.PolynomialBatch.from_values(_columns(rng, c, 1 << lg), rb, False, 2, ctx=ctx) for c in (3, 4)]
    handles = (C.c_void_p * 2)(*[b._h.value for b in bs])
    cb = (glb._native.FriBatch * 2)()
    cp = (glb._native.FriPoly * 4)(*[glb._native.FriPoly(i, j) for i, j in ((0, 0), (0, 2), (1, 3), (1, 0))])
    cb[0].point[0], cb[0].point[1], cb[0].first_poly, cb[0].num_polys = 0x1111, 0x2222, 0, 3
    cb[1].point[0], cb[1].point[1], cb[1].first_poly, cb[1].num_polys = 0x3333, 0x4444, 3, 1
    al = (C.c_uint64 * 2)(0xABCDEF, 0x123)
    N = (1 << lg) << rb

    def check(res):   # the values are the coset_fft(7) of the coefficients over the extension
        cf = res["lde_coeffs_out"].view(np.uint64).reshape(N, 2)
        assert cf.any() and np.array_equal(res["lde_values_out"].view(np.uint64).reshape(N, 2), o.ext_coset_fft(cf, 7))

    def done():
        for b in bs:
            b.free()

    return Case({}, {"lde_coeffs_out": 16 * N, "lde_values_out": 16 * N}, check=check, done=done,
                call=lambda sp, p, v: ctx.check(ctx._lib.gl_fri_final_poly(ctx._h, handles, 2, cb, 2, cp, al, rb, p["lde_coeffs_out"],
                                                                           p["lde_values_out"], sp)))


def _circuit_ctypes(glb, c):
    N = glb._native
    cd = N.Circuit(*[int(x) for x in c["circuit"]])
    gates = (N.Gate * len(c["gates"]))(*[N.Gate(*[int(x) for x in tuple(g)[:5]], 0) for g in c["gates"]])
    return cd, gates


def row_quotient(ctx, glb, o):
    from quotient_circuit import build

    lg = 5
    c = build(lg, seed=lg)
    rng = np.random.default_rng(1234 + lg)
    betas, gammas, alphas = (rng.integers(0, P, 2, dtype=np.uint64) for _ in range(3))
    zs = o.permutation_zs(c["circuit"], c["k_is"], c["wires"], c["sigmas"], betas, gammas)
    vals = [np.concatenate([c["constants"], c["sigmas"]]), c["wires"], zs]
    bs = [glb.PolynomialBatch.from_values(v, 3, False, 4, ctx=ctx) for v in vals]
    leaves = [o.commit_from_values(v, 3, 4)["leaves"] for v in vals]
    want = o.quotient_polys(c["circuit"], c["gates"], c["k_is"], *leaves, 3, c["pih"], betas, gammas, alphas)
    cd, gates = _circuit_ctypes(glb, c)
    host = [np.ascontiguousarray(x, dtype=np.uint64) for x in (c["k_is"], c["pih"], betas, gammas, alphas)]

    def done():
        for b in bs:
            b.free()

    return Case({}, {"chunks_out": want.nbytes}, want={"chunks_out": want}, done=done,
                call=lambda sp, p, v: ctx.check(ctx._lib.gl_quotient_polys(ctx._h, C.byref(cd), gates, host[0].ctypes.data, bs[0]._h,
                                                                           bs[1]._h, bs[2]._h, host[1].ctypes.data, host[2].ctypes.data,
                                                                           host[3].ctypes.data, host[4].ctypes.data, p["chunks_out"], sp)))


def row_permutation_zs(ctx, glb, o):
    from quotient_circuit import build

    lg = 6
    c = build(lg, seed=2)
    rng = np.random.default_rng(77)
    betas, gammas = (rng.integers(0, P, 2, dtype=np.uint64) for _ in range(2))
    want = o.permutation_zs(c["circuit"], c["k_is"], c["wires"], c["sigmas"], betas, gammas)
    cs = glb.PolynomialBatch.from_values(np.concatenate([c["constants"], c["sigmas"]]), 3, False, 4, ctx=ctx)
    wb = glb.PolynomialBatch.from_values(c["wires"], 3, False, 4, ctx=ctx)
    cd, _ = _circuit_ctypes(glb, c)
    k_is = np.ascontiguousarray(c["k_is"], dtype=np.uint64)
    grand = np.zeros(2, dtype=np.uint64)

    def call(sp, p, v):
        ctx.check(ctx._lib.gl_permutation_zs(ctx._h, C.byref(cd), k_is.ctypes.data, cs._h, wb._h, betas.ctypes.data,
                                             gammas.ctypes.data, p["zs_partial_products_out"], sp, grand.ctypes.data))
        return {"grand": grand.copy()}

    def done():
        cs.free()
        wb.free()

    return Case({}, {"zs_partial_products_out": want.nbytes}, call=call, done=done,
                want={"zs_partial_products_out": want, "grand": np.ones(2, dtype=np.uint64)})


def row_prove(ctx, glb, o):
    from quotient_circuit import build

    fri = importlib.import_module("plonky2-lib_b200.fri")
    lg, pis = 5, [3, 1, 4]
    c = build(lg, seed=lg)
    c["pih"] = o.hash_no_pad(np.asarray(pis, dtype=np.uint64))
    c["wires"][0:4, 0] = c["pih"]
    fp = fri.FriParams.for_degree(glb.FriConfig(), lg)
    cs = glb.PolynomialBatch.from_values(np.concatenate([c["constants"], c["sigmas"]]), 3, False, 4, ctx=ctx)
    digest = np.array([11, 22, 33, 44], dtype=np.uint64)
    shape = c["wires"].shape

    def call(sp, p, v):
        return {"proof": glb.host.prove(c["circuit"], c["gates"], c["k_is"], cs, digest, fp, v["wires"].reshape(shape), pis,
                                        ctx=ctx)["words"]}

    return Case({"wires": np.ascontiguousarray(c["wires"]).reshape(-1)}, {}, call=call, done=cs.free)


# (entries covered, case id, builder(ctx, glb, oracle) -> Case)
TABLE = []
for _m in (1, 4099):
    TABLE += [
        (("gl_poseidon_permute_batch",), f"m{_m}", lambda x, g, o, m=_m: row_permute(x, g, o, m)),
        (("gl_poseidon_two_to_one_batch",), f"m{_m}", lambda x, g, o, m=_m: row_two_to_one(x, g, o, m)),
        (("gl_smt_leaf_hash_batch",), f"m{_m}", lambda x, g, o, m=_m: row_smt_leaf_hash(x, g, o, m)),
        (("gl_smt_build",), f"m{_m}", lambda x, g, o, m=_m: row_smt_build(x, g, o, m)),
    ]
    TABLE += [(("gl_poseidon_hash_no_pad_batch",), f"m{_m}-len{_ln}", lambda x, g, o, m=_m, ln=_ln: row_hash_no_pad(x, g, o, m, ln))
              for _ln in (0, 8, 9)]
TABLE += [
    (("gl_smt_verify_process_batch",), "m64", row_smt_verify),
    (("gl_smt_set_proofs",), "m300", row_smt_set_proofs),
    (("gl_smt_find_batch",), "m300-q77", row_smt_find),
    (("gl_merkle_build",), "len7", lambda x, g, o: row_merkle_build(x, g, o, 7)),
    (("gl_merkle_build",), "len3", lambda x, g, o: row_merkle_build(x, g, o, 3)),
    (("gl_merkle_verify_batch",), "k5", row_merkle_verify),
]
for _e in ("gl_fft_batch", "gl_ifft_batch", "gl_coset_fft_batch", "gl_coset_ifft_batch"):
    TABLE += [((_e,), f"lg{_lg}", lambda x, g, o, e=_e, lg=_lg: row_fft(x, g, o, e, lg)) for _lg in (0, 1, 15, 16, 20)]
for _e in ("gl_commit_from_values", "gl_commit_from_coeffs"):
    TABLE += [((_e,), f"lg{_lg}", lambda x, g, o, e=_e, lg=_lg: row_commit(x, g, o, e, lg)) for _lg in (0, 1, 15, 16, 20)]
for _e in ("gl_commit_from_values_ex", "gl_commit_from_coeffs_ex"):
    TABLE += [((_e,), f"lg{_lg}-blinded", lambda x, g, o, e=_e, lg=_lg: row_commit(x, g, o, e, lg)) for _lg in (0, 16)]
TABLE += [
    (("gl_commit_add_coeffs", "gl_commit_finish"), "stream", row_commit_stream),
    (("gl_commit_coeffs", "gl_commit_eval", "gl_commit_download"), "resident", row_commit_reads),
    (("gl_commit_open",), "k3", row_commit_open),
    (("gl_commit_get_lde_values",), "k3", row_commit_lde_values),
    (("gl_fri_layer_tree",), "len512", row_fri_layer_tree),
    (("gl_fri_layer_commit",), "len512", row_fri_layer_commit),
    (("gl_fri_fold",), "len512", row_fri_fold),
    (("gl_fri_final_poly",), "lg5", row_fri_final_poly),
    (("gl_quotient_polys",), "lg5", row_quotient),
    (("gl_permutation_zs",), "lg6", row_permutation_zs),
    (("gl_prove",), "lg5", row_prove),
]
# the group entry points: test_group_device_buffers below
GROUP_ENTRIES = ("gl_group_commit_from_values", "gl_group_commit_from_coeffs", "gl_group_commit_open")


@pytest.mark.gpu
@pytest.mark.parametrize("entries,build", [pytest.param(e, b, id="-".join(x[3:] for x in e) + "-" + i) for e, i, b in TABLE])
def test_device_buffers(glb, ctx, oracle, entries, build):
    _exercise(ctx, glb, build(ctx, glb, oracle), entries)


@pytest.mark.gpu
@pytest.mark.parametrize("is_values", [True, False], ids=["from_values", "from_coeffs"])
def test_group_device_buffers(glb, oracle, is_values):
    """gl_group_commit_from_values / _from_coeffs with every rank's buffers as device views at a 16-byte offset, against the
    host-buffer group commit and the oracle; an 8-byte-offset view of any rank is refused with GL_E_ARG, and the group then
    still commits; gl_group_commit_open refuses GL_DEVICE.  Two ranks when two GPUs are visible, else the one-rank group
    (the same guard and the same device path without the exchange)."""
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    nranks = 2 if torch.cuda.device_count() >= 2 else 1
    N = glb._native
    lg, c, rb, h = 9, 11, 2, 2
    n = 1 << lg
    a = _columns(np.random.default_rng(55), c, n)
    w = (oracle.commit_from_values if is_values else oracle.commit_from_coeffs)(a, rb, h, want_leaves=False)
    g = glb.Group.local(list(range(nranks)))
    try:
        host = g.commit(a, rb, h, is_values=is_values)
        for cp in host.caps:
            assert np.array_equal(cp, w["cap"])
        host.free()

        def commit(lead_in, lead_out):
            """Device views [lead:] of sentinel-padded tensors on every rank; returns (caps, coeffs, bases)."""
            bases, ptr = [], {"in": [], "co": [], "cap": []}
            for r in range(nranks):
                dev = f"cuda:{r}"
                for key, words, init, lead in (("in", a.size, a.reshape(-1), lead_in[r]), ("co", a.size, None, lead_out[r]),
                                               ("cap", 4 << h, None, lead_out[r])):
                    base = np.full(words + lead + PAD, SENT, dtype=np.uint64)
                    if init is not None:
                        base[lead:lead + words] = init
                    t = torch.from_numpy(base.view(np.int64)).to(dev)
                    bases.append((key, r, lead, words, t, base))
                    ptr[key].append(t.data_ptr() + 8 * lead)
            arr = {k: (C.c_void_p * nranks)(*v) for k, v in ptr.items()}
            hs = (C.c_void_p * nranks)()
            if is_values:
                rc = g._lib.gl_group_commit_from_values(g._h, arr["in"], lg, c, rb, h, arr["co"], arr["cap"], hs, N.GL_DEVICE, 0)
            else:
                rc = g._lib.gl_group_commit_from_coeffs(g._h, arr["in"], lg, c, rb, h, arr["cap"], hs, N.GL_DEVICE, 0)
            for hd in hs:
                if hd:
                    g._lib.gl_commit_free(hd)
            return rc, bases

        rc, bases = commit([2] * nranks, [2] * nranks)
        g.check(rc)
        for key, r, lead, words, t, before in bases:
            after = t.cpu().numpy().view(np.uint64)
            if key == "in" or (key == "co" and not is_values):
                assert np.array_equal(after, before), f"rank {r}: {key} changed"
                continue
            assert (after[:lead] == SENT).all() and (after[lead + words:] == SENT).all(), f"rank {r}: bytes outside {key} changed"
            want = w["cap"] if key == "cap" else w["coeffs"]
            assert np.array_equal(after[lead:lead + words], want.reshape(-1)), f"rank {r}: {key} differs"
        last = nranks - 1
        for which in ("in", "out"):
            leads_in = [2] * nranks
            leads_out = [2] * nranks
            (leads_in if which == "in" else leads_out)[last] = 1
            rc, bases = commit(leads_in, leads_out)
            assert rc == N.GL_E_ARG
            msg = (g._lib.gl_group_last_error(g._h) or b"").decode()
            want_arg = ("values" if is_values else "coeffs") if which == "in" else ("coeffs_out" if is_values else "cap_out")
            assert f": {want_arg}[{last}]" in msg, msg
            for key, r, lead, words, t, before in bases:
                assert np.array_equal(t.cpu().numpy().view(np.uint64), before), "a refused call wrote to a buffer"
        again = g.commit(a, rb, h, is_values=is_values)
        for cp in again.caps:
            assert np.array_equal(cp, w["cap"])
        idx = np.array([0, 5], dtype=np.uint64)
        rows = np.zeros((2, c), dtype=np.uint64)
        rp = (C.c_void_p * nranks)(*[rows.ctypes.data] * nranks)
        hs = (C.c_void_p * nranks)(*[hd.value for hd in again._hs]) if hasattr(again, "_hs") else None
        if hs is not None:
            assert g._lib.gl_group_commit_open(g._h, hs, idx.ctypes.data, 2, rp, None, N.GL_DEVICE) == N.GL_E_ARG
        again.free()
    finally:
        g.close()


# ---- CPU: the table and the guard stay complete ---------------------------------------------------------------------------
def _header_space_functions():
    text = open(os.path.join(ROOT, "include", "gl_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    out = {}
    for m in re.finditer(r"\bint\s+(gl_\w+)\s*\(([^)]*)\)\s*;", text):
        if re.search(r"\bint\s+space\b", m.group(2)):
            out[m.group(1)] = m.group(2)
    return out


def _matching(text, i, open_ch, close_ch):
    depth = 0
    for j in range(i, len(text)):
        if text[j] == open_ch:
            depth += 1
        elif text[j] == close_ch:
            depth -= 1
            if depth == 0:
                return j
    raise ValueError("unbalanced")


def _function_bodies():
    src = ""
    for f in ("gl_b200.cu", "gl_group.inc.cu"):
        src += open(os.path.join(ROOT, "plonky2-lib_b200", "csrc", f)).read() + "\n"
    src = re.sub(r"//[^\n]*", "", src)
    bodies = {}
    for m in re.finditer(r'(?m)^(?:extern "C" |static )[^;{}()]*?\b(\w+)\s*\(', src):
        close = _matching(src, m.end() - 1, "(", ")")
        rest = src[close + 1:]
        k = len(rest) - len(rest.lstrip())
        if not rest[k:].startswith("{"):
            continue
        start = close + 1 + k
        bodies[m.group(1)] = src[start:_matching(src, start, "{", "}") + 1]
    return bodies


def _guard_calls(body):
    calls = []
    for m in re.finditer(r"\bcheck_device_ptr\s*\(", body):
        calls.append(body[m.start():_matching(body, m.end() - 1, "(", ")") + 1])
    return calls


def test_every_space_entry_point_has_a_row_and_checks_its_device_buffers():
    """Each header function with an `int space` parameter (a) has a row in the GPU table above and (b) calls the library's
    alignment guard -- in its body or in a helper it calls directly -- for every device buffer the row passes; a function
    that serves host buffers only must refuse every other space outright."""
    header = _header_space_functions()
    assert len(header) >= 30
    covered = {e for entries, _, _ in TABLE for e in entries} | set(GROUP_ENTRIES)
    assert set(header) == set(DEVICE_ARGS), "DEVICE_ARGS and the header's space entry points differ"
    assert covered == set(header), f"entry points without a row: {sorted(set(header) - covered)}"
    bodies = _function_bodies()
    for name, params in header.items():
        assert name in bodies, f"{name}: definition not found"
        body = bodies[name]
        calls = _guard_calls(body)
        for helper in set(re.findall(r"\b(\w+)\s*\(", body)) & set(bodies):
            if helper not in header and helper != name:
                calls += _guard_calls(bodies[helper])
        args = DEVICE_ARGS[name]
        if not args:
            assert re.search(r"if \(space != GL_HOST\) return", body), f"{name}: serves host buffers only but does not refuse GL_DEVICE"
            continue
        for a in args:
            assert re.search(rf"\b{a}\b", params), f"{name}: {a} is not a parameter"
            assert any(re.search(rf"\b{a}\b", call) for call in calls), f"{name}: device buffer {a} is not checked by check_device_ptr"
