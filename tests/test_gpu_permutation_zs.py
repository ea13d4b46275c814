"""gl_permutation_zs (all_wires_permutation_partial_products on the resident commits) against the oracle's restatement of the
prover's loop, bit for bit: on the reference circuits of tests/quotient_circuit.py, on synthetic instances of other
geometries and at full size; then the device-resident chain Z -> Z commit -> quotient -> quotient commit, corrupted
witnesses, the zero-denominator panic, argument checks and the C++ mirror."""
import importlib
import os
import subprocess

import numpy as np
import pytest

from conftest import P
from quotient_circuit import build

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
M32 = np.uint64(0xFFFFFFFF)


# ---- vectorised Goldilocks arithmetic for the instance builder (plonky2's reduce128) -----------------------------------
def _mulmod(a, b):
    a, b = np.broadcast_arrays(np.asarray(a, dtype=np.uint64), np.asarray(b, dtype=np.uint64))
    a0, a1, b0, b1 = a & M32, a >> np.uint64(32), b & M32, b >> np.uint64(32)
    ll, lh, hl, hh = a0 * b0, a0 * b1, a1 * b0, a1 * b1
    mid = lh + hl
    mid_carry = (mid < lh).astype(np.uint64)
    lo = ll + (mid << np.uint64(32))
    lo_carry = (lo < ll).astype(np.uint64)
    hi = hh + (mid >> np.uint64(32)) + (mid_carry << np.uint64(32)) + lo_carry
    hi_hi, hi_lo = hi >> np.uint64(32), hi & M32
    t0 = lo - hi_hi
    t0 = np.where(lo < hi_hi, t0 - M32, t0)
    t1 = hi_lo * M32
    t2 = t0 + t1
    t2 = np.where(t2 < t1, t2 + M32, t2)
    return np.where(t2 >= np.uint64(P), t2 - np.uint64(P), t2)


def _subgroup(lg_n):
    w = pow(pow(7, (P - 1) >> 32, P), 1 << (32 - lg_n), P)
    sub = np.ones(1 << lg_n, dtype=np.uint64)
    for k in range(lg_n):
        h = 1 << k
        sub[h:2 * h] = _mulmod(sub[:h], pow(w, h, P))
    return sub


def synthetic(lg_n, R=80, num_wires=135, num_constants=4, nch=2, deg=8, swaps=None, seed=0):
    """Identity sigmas sigma_j(i) = k_j w^i plus `swaps` random disjoint transpositions of routed positions whose two ends
    hold equal wire values: a witness that satisfies its copy constraints (numpy-vectorised, any size)."""
    rng = np.random.default_rng(seed)
    n = 1 << lg_n
    k_is = np.array([pow(7, j, P) for j in range(R)], dtype=np.uint64)
    sub = _subgroup(lg_n)
    sigmas = np.stack([_mulmod(k, sub) for k in k_is])
    wires = rng.integers(0, P, (num_wires, n), dtype=np.uint64)
    m = swaps if swaps is not None else max(1, min((R * n) // 16, 1 << 16))
    pos = rng.choice(R * n, 2 * m, replace=False)
    a, b = pos[:m], pos[m:]
    sf, wf = sigmas.reshape(-1), wires[:R].reshape(-1)
    sf[a], sf[b] = sf[b].copy(), sf[a].copy()
    wf[b] = wf[a]
    constants = rng.integers(0, P, (num_constants, n), dtype=np.uint64)
    circuit = (lg_n, num_wires, R, num_constants, 0, nch, deg, 0)
    betas, gammas = (rng.integers(0, P, nch, dtype=np.uint64) for _ in range(2))
    return {"circuit": circuit, "k_is": k_is, "constants": constants, "sigmas": sigmas, "wires": wires, "betas": betas,
            "gammas": gammas}


def _challenges(lg_n):
    rng = np.random.default_rng(1234 + lg_n)
    return tuple(rng.integers(0, P, 2, dtype=np.uint64) for _ in range(3))


def _commits(glb, ctx, c, wires_blinding=False, wires_from_coeffs=False, oracle=None):
    cs = glb.PolynomialBatch.from_values(np.concatenate([c["constants"], c["sigmas"]]), 3, False, 4, ctx=ctx)
    if wires_from_coeffs:
        coeffs = np.stack([oracle.ifft(col) for col in c["wires"]])     # the oracle transforms one polynomial at a time
        w = glb.PolynomialBatch.from_coeffs(coeffs, 3, wires_blinding, 4, ctx=ctx)
    else:
        w = glb.PolynomialBatch.from_values(c["wires"], 3, wires_blinding, 4, ctx=ctx)
    return cs, w


def _check_layout(got, c):
    lg_n, _, R, _, _, nch, deg, _ = c["circuit"]
    assert got.shape == (nch * -(-R // deg), 1 << lg_n)


# ---- 1. reference circuits --------------------------------------------------------------------------------------------
@pytest.mark.parametrize("lg_n", [3, 5, 8, 12, 14, 16])
def test_matches_oracle_on_reference_circuits(glb, ctx, oracle, lg_n):
    c = build(lg_n, seed=lg_n)
    betas, gammas, _ = _challenges(lg_n)
    cs, w = _commits(glb, ctx, c)
    got, grand = glb.host.permutation_zs(c["circuit"], c["k_is"], cs, w, betas, gammas, ctx=ctx)
    want = oracle.permutation_zs(c["circuit"], c["k_is"], c["wires"], c["sigmas"], betas, gammas)
    _check_layout(got, c)
    assert np.array_equal(got, want)
    assert grand.tolist() == [1, 1]
    cs.free()
    w.free()


# ---- 2. geometry variants -----------------------------------------------------------------------------------------------
VARIANTS = {
    "R75_deg8": dict(R=75, deg=8),
    "deg4": dict(deg=4),
    "one_chunk": dict(R=5, num_wires=9, deg=8),
    "nch1": dict(nch=1),
    "nch3": dict(nch=3),
    "nch4_deg2": dict(R=24, num_wires=30, nch=4, deg=2),
}


@pytest.mark.parametrize("name", sorted(VARIANTS))
def test_geometry_variants_match_oracle(glb, ctx, oracle, name):
    c = synthetic(10, seed=sorted(VARIANTS).index(name), **VARIANTS[name])
    cs, w = _commits(glb, ctx, c)
    got, grand = glb.host.permutation_zs(c["circuit"], c["k_is"], cs, w, c["betas"], c["gammas"], ctx=ctx)
    want = oracle.permutation_zs(c["circuit"], c["k_is"], c["wires"], c["sigmas"], c["betas"], c["gammas"])
    _check_layout(got, c)
    assert np.array_equal(got, want)
    assert grand.tolist() == [1] * c["circuit"][5]
    cs.free()
    w.free()


@pytest.mark.parametrize("blinding,from_coeffs", [(True, False), (False, True), (True, True)])
def test_blinded_and_from_coeffs_wires_commits(glb, ctx, oracle, blinding, from_coeffs):
    """The salt of a blinded commit lives only in its leaves; a from_coeffs commit holds the same coefficients."""
    c = synthetic(9, seed=11)
    cs, w = _commits(glb, ctx, c, wires_blinding=blinding, wires_from_coeffs=from_coeffs, oracle=oracle)
    got, grand = glb.host.permutation_zs(c["circuit"], c["k_is"], cs, w, c["betas"], c["gammas"], ctx=ctx)
    want = oracle.permutation_zs(c["circuit"], c["k_is"], c["wires"], c["sigmas"], c["betas"], c["gammas"])
    assert np.array_equal(got, want) and grand.tolist() == [1, 1]
    cs.free()
    w.free()


def test_device_buffer_output(glb, ctx, oracle):
    c = synthetic(11, seed=5)
    cs, w = _commits(glb, ctx, c)
    buf = glb.DeviceBuffer((2 * 10, 1 << 11), ctx)
    out, grand = glb.host.permutation_zs(c["circuit"], c["k_is"], cs, w, c["betas"], c["gammas"], out=buf, ctx=ctx)
    assert out is buf
    want = oracle.permutation_zs(c["circuit"], c["k_is"], c["wires"], c["sigmas"], c["betas"], c["gammas"])
    assert np.array_equal(buf.to_host(), want) and grand.tolist() == [1, 1]
    buf.free()
    cs.free()
    w.free()


# ---- 3. full size ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("lg_n", [18, 20])
def test_fullsize_matches_oracle(glb, ctx, oracle, lg_n):
    c = synthetic(lg_n, seed=lg_n)
    cs, w = _commits(glb, ctx, c)
    got, grand = glb.host.permutation_zs(c["circuit"], c["k_is"], cs, w, c["betas"], c["gammas"], ctx=ctx)
    cs.free()
    w.free()
    want = oracle.permutation_zs(c["circuit"], c["k_is"], c["wires"], c["sigmas"], c["betas"], c["gammas"])
    assert np.array_equal(got, want)
    assert grand.tolist() == [1, 1]


# ---- 4. the Z columns stay on the device ------------------------------------------------------------------------------
def _degree_bound_holds(chunks, n):
    return all(not chunks[ch * 8 + 7][n - 8:].any() for ch in range(2))


@pytest.mark.parametrize("lg_n", [12, 16])
def test_device_resident_prove_round(glb, ctx, oracle, lg_n):
    import torch

    c = build(lg_n, seed=lg_n)
    betas, gammas, alphas = _challenges(lg_n)
    cs, w = _commits(glb, ctx, c)
    n = 1 << lg_n
    zs_dev = torch.empty((2 * 10, n), dtype=torch.int64, device=f"cuda:{ctx.device}")
    _, grand = glb.host.permutation_zs(c["circuit"], c["k_is"], cs, w, betas, gammas, out=zs_dev, ctx=ctx)
    assert grand.tolist() == [1, 1]
    zb = glb.PolynomialBatch.from_values(zs_dev, 3, False, 4, ctx=ctx)
    got = glb.host.compute_quotient_polys(c["circuit"], c["gates"], c["k_is"], cs, w, zb, c["pih"], betas, gammas, alphas, ctx=ctx)
    qb = glb.PolynomialBatch.from_coeffs(got, 3, False, 4, ctx=ctx)
    zs = oracle.permutation_zs(c["circuit"], c["k_is"], c["wires"], c["sigmas"], betas, gammas)
    vals = [np.concatenate([c["constants"], c["sigmas"]]), c["wires"], zs]
    leaves = [oracle.commit_from_values(v, 3, 4)["leaves"] for v in vals]
    want = oracle.quotient_polys(c["circuit"], c["gates"], c["k_is"], *leaves, 3, c["pih"], betas, gammas, alphas)
    assert np.array_equal(got, want)
    assert np.array_equal(zb.merkle_tree.cap, oracle.commit_from_values(zs, 3, 4, want_leaves=False)["cap"])
    assert np.array_equal(qb.merkle_tree.cap, oracle.commit_from_coeffs(want, 3, 4, want_leaves=False)["cap"])
    assert _degree_bound_holds(got, n) and all(got[ch * 8 + 7][: n - 8].any() for ch in range(2))
    for b in (cs, w, zb, qb):
        b.free()


# ---- 5. corrupted witnesses ---------------------------------------------------------------------------------------------
def test_copy_violation_returns_columns_and_breaks_the_quotient(glb, ctx, oracle):
    lg_n = 7
    c = build(lg_n, seed=3, corrupt="copy")
    rng = np.random.default_rng(5)
    betas, gammas, alphas = (rng.integers(0, P, 2, dtype=np.uint64) for _ in range(3))
    cs, w = _commits(glb, ctx, c)
    zs, grand = glb.host.permutation_zs(c["circuit"], c["k_is"], cs, w, betas, gammas, ctx=ctx)
    assert any(int(g) != 1 for g in grand)
    assert zs.shape == (20, 1 << lg_n) and zs[0][0] == 1 and zs[1][0] == 1
    with pytest.raises(ValueError):          # the oracle stops at the open grand product
        oracle.permutation_zs(c["circuit"], c["k_is"], c["wires"], c["sigmas"], betas, gammas)
    zb = glb.PolynomialBatch.from_values(zs, 3, False, 4, ctx=ctx)
    got = glb.host.compute_quotient_polys(c["circuit"], c["gates"], c["k_is"], cs, w, zb, c["pih"], betas, gammas, alphas, ctx=ctx)
    assert not _degree_bound_holds(got, 1 << lg_n)
    for b in (cs, w, zb):
        b.free()


def test_gate_violation_keeps_the_copy_constraints(glb, ctx, oracle):
    c = build(7, seed=3, corrupt="bit")
    betas, gammas, _ = _challenges(7)
    cs, w = _commits(glb, ctx, c)
    got, grand = glb.host.permutation_zs(c["circuit"], c["k_is"], cs, w, betas, gammas, ctx=ctx)
    assert grand.tolist() == [1, 1]
    assert np.array_equal(got, oracle.permutation_zs(c["circuit"], c["k_is"], c["wires"], c["sigmas"], betas, gammas))
    cs.free()
    w.free()


# ---- 6. zero denominator ------------------------------------------------------------------------------------------------
def test_zero_denominator_panics(glb, ctx):
    c = synthetic(8, seed=21)
    row, j = 77, 13
    betas, gammas = c["betas"].copy(), c["gammas"].copy()
    gammas[1] = (-(int(c["wires"][j, row]) + int(betas[1]) * int(c["sigmas"][j, row]))) % P
    cs, w = _commits(glb, ctx, c)
    with pytest.raises(glb.GlPanic) as e:
        glb.host.permutation_zs(c["circuit"], c["k_is"], cs, w, betas, gammas, ctx=ctx)
    assert "zero" in str(e.value)
    # the ctx stays usable
    _, grand = glb.host.permutation_zs(c["circuit"], c["k_is"], cs, w, c["betas"], c["gammas"], ctx=ctx)
    assert grand.tolist() == [1, 1]
    cs.free()
    w.free()


# ---- 7. argument checks -------------------------------------------------------------------------------------------------
def test_argument_checks(glb, ctx):
    c = synthetic(6, seed=2)
    cs, w = _commits(glb, ctx, c)
    k, b, g = c["k_is"], c["betas"], c["gammas"]
    zs = glb.host.permutation_zs

    def bad(**kw):
        cd = list(c["circuit"])
        for i, key in enumerate(("degree_bits", "num_wires", "num_routed_wires", "num_constants", "num_selectors",
                                 "num_challenges", "quotient_degree_factor")):
            if key in kw:
                cd[i] = kw[key]
        return cd

    with pytest.raises(glb.GlPanic):
        zs(bad(num_wires=134), k, cs, w, b, g, ctx=ctx)                 # wires column count
    with pytest.raises(glb.GlPanic):
        zs(bad(num_constants=3), k, cs, w, b, g, ctx=ctx)               # constants_sigmas column count
    with pytest.raises(glb.GlPanic):
        zs(bad(num_challenges=0), k, cs, w, b, g, ctx=ctx)
    b5 = np.arange(1, 6, dtype=np.uint64)
    with pytest.raises(glb.GlPanic):
        zs(bad(num_challenges=5), k, cs, w, b5, b5, ctx=ctx)
    with pytest.raises(glb.GlPanic):
        zs(bad(quotient_degree_factor=6), k, cs, w, b, g, ctx=ctx)      # not a power of two
    with pytest.raises(glb.GlPanic):
        zs(bad(degree_bits=7), k, cs, w, b, g, ctx=ctx)                 # circuit degree differs from the commits'
    c7 = synthetic(7, seed=2)
    w7 = glb.PolynomialBatch.from_values(c7["wires"], 3, False, 4, ctx=ctx)
    with pytest.raises(glb.GlPanic):
        zs(c["circuit"], k, cs, w7, b, g, ctx=ctx)                      # commits of different degree
    w7.free()
    # a sharded commit
    sc = glb.Context(ctx.device)
    sc.set_shard(0, 2)
    s_cs, s_w = _commits(glb, sc, c)
    with pytest.raises(glb.GlPanic):
        zs(c["circuit"], k, s_cs, s_w, b, g, ctx=sc)
    s_cs.free()
    s_w.free()
    sc.close()
    # a handle of another ctx
    other = glb.Context(ctx.device)
    with pytest.raises(glb.GlPanic) as e:
        zs(c["circuit"], k, cs, w, b, g, ctx=other)
    assert e.value.code == 4
    other.close()
    # a FRI layer tree: a commit without polynomials
    fri = importlib.import_module("plonky2-lib_b200.fri")
    vals = glb.DeviceBuffer((1 << 8, 2), ctx).from_host(np.arange(1 << 9, dtype=np.uint64))
    tree = fri.FriLayerTree(vals, 1 << 8, 4, 2, ctx)
    with pytest.raises(glb.GlPanic) as e:
        zs(c["circuit"], k, cs, tree, b, g, ctx=ctx)
    assert e.value.code == 4
    tree.free()
    vals.free()
    cs.free()
    w.free()


# ---- 8. the C++ mirror ----------------------------------------------------------------------------------------------------
def test_cpp_mirror_matches_python_mirror(glb, ctx, tmp_path):
    """tests/cpp/permutation_zs_mirror_test.cpp commits a fixed instance through plonky2_b200.hpp and dumps the columns and
    grand products of all_wires_permutation_partial_products; the Python mirror computes the same instance."""
    exe, dump = str(tmp_path / "permutation_zs_mirror_test"), str(tmp_path / "zs.txt")
    libdir = os.path.join(ROOT, "plonky2-lib_b200")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-Wall", "-I", os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "tests", "cpp", "permutation_zs_mirror_test.cpp"), "-L", libdir, "-lgl_b200",
                           f"-Wl,-rpath,{libdir}", "-o", exe])
    out = subprocess.run([exe, dump], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stdout + out.stderr
    got = [int(x) for x in open(dump).read().split()]
    # the same instance as the C++ program: splitmix64 values, identity sigmas with a few swapped positions
    lg_n, R, num_wires, num_constants, deg = 6, 20, 24, 3, 4
    n = 1 << lg_n

    def splitmix(x):
        x = (x + 0x9E3779B97F4A7C15) & 0xFFFFFFFFFFFFFFFF
        x = ((x ^ (x >> 30)) * 0xBF58476D1CE4E5B9) & 0xFFFFFFFFFFFFFFFF
        x = ((x ^ (x >> 27)) * 0x94D049BB133111EB) & 0xFFFFFFFFFFFFFFFF
        x ^= x >> 31
        return x % P if x >= P else x

    wires = np.array([[splitmix((j << 32) + i) for i in range(n)] for j in range(num_wires)], dtype=np.uint64)
    consts = np.array([[splitmix(((100 + j) << 32) + i) for i in range(n)] for j in range(num_constants)], dtype=np.uint64)
    k_is = np.array([pow(7, j, P) for j in range(R)], dtype=np.uint64)
    sub = _subgroup(lg_n)
    sigmas = _mulmod(k_is[:, None], sub[None, :])
    for t in range(8):                      # swap (t, 2t + 1) <-> (t + 10, 5t + 3), equal wire values at both ends
        a, b = (t, 2 * t + 1), (t + 10, 5 * t + 3)
        sigmas[a], sigmas[b] = sigmas[b], sigmas[a]
        wires[b] = wires[a]
    circuit = (lg_n, num_wires, R, num_constants, 0, 2, deg, 0)
    cs = glb.PolynomialBatch.from_values(np.concatenate([consts, sigmas]), 3, False, 4, ctx=ctx)
    w = glb.PolynomialBatch.from_values(wires, 3, False, 4, ctx=ctx)
    zs, grand = glb.host.permutation_zs(circuit, k_is, cs, w, [11, 13], [17, 19], ctx=ctx)
    assert got == [int(x) for x in zs.reshape(-1)] + [int(x) for x in grand]
    assert grand.tolist() == [1, 1]
    cs.free()
    w.free()
