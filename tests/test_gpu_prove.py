"""gl_prove (plonky2::plonk::prover::prove from the witness on, one call) and plonk_verifier.verify_proof (the whole proof):
byte for byte against the oracle's restatement (oracle/plonk_oracle.py), every witness form, 0 / 1 / 9 public inputs, other
geometries and the older FRI form, full size, rejection of bad witnesses and tampered proofs, the argument checks and the
C++ mirror.  Instances come from tests/quotient_circuit.py with the PublicInputGate row's wires 0..3 set to
hash_no_pad(public_inputs): those wires are in no copy constraint, so the witness still satisfies every constraint."""
import ctypes as C
import importlib
import os
import subprocess

import numpy as np
import pytest

from conftest import P
from prove_circuit import identity_sigmas, large
from quotient_circuit import build

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DIGEST = np.array([11, 22, 33, 44], dtype=np.uint64)


@pytest.fixture(scope="module")
def mods(glb):
    return (importlib.import_module("plonky2-lib_b200.fri"), importlib.import_module("plonky2-lib_b200.wire"),
            importlib.import_module("plonky2-lib_b200.plonk_verifier"))


def _instance(oracle, lg_n, pis, seed=None, corrupt=None, nch=2):
    c = build(lg_n, seed=lg_n if seed is None else seed, corrupt=corrupt)
    pih = oracle.hash_no_pad(np.asarray(pis, dtype=np.uint64))
    c["wires"][0:4, 0] = pih
    c["pih"] = pih
    c["circuit"] = c["circuit"][:5] + (nch,) + c["circuit"][6:]
    c["num_pis"] = len(pis)
    return c


def _fri_params(fri, glb, lg_n, times_x=False):
    fp = fri.FriParams.for_degree(glb.FriConfig(), lg_n)
    fp.final_poly_times_x = times_x
    return fp


def _cs(glb, ctx, c, **kw):
    return glb.PolynomialBatch.from_values(np.concatenate([c["constants"], c["sigmas"]]), 3, False, 4, ctx=ctx, **kw)


def _bytes(wire, p):
    return wire.proof_with_public_inputs_to_bytes(p["caps"], p["openings"], p["opening_proof"], p["public_inputs"])


def _verify(pv, c, fp, cap, data):
    return pv.verify_proof(data, pv.CommonData(c["circuit"], c["gates"], c["k_is"], fp, c["num_pis"]), pv.VerifierData(cap, DIGEST))


def _prove(glb, ctx, c, fp, pis, cs=None, wires=None):
    own = cs is None
    cs = _cs(glb, ctx, c) if own else cs
    p = glb.host.prove(c["circuit"], c["gates"], c["k_is"], cs, DIGEST, fp, c["wires"] if wires is None else wires, pis, ctx=ctx)
    cap = cs.merkle_tree.cap.copy()
    if own:
        cs.free()
    return p, cap


def _oracle_bytes(wire, c, pis, times_x=False):
    from oracle import plonk_oracle

    o = plonk_oracle.prove(c["circuit"], c["gates"], c["k_is"], c["constants"], c["sigmas"], DIGEST, c["wires"], pis, times_x=times_x)
    return _bytes(wire, o), o["constants_sigmas_cap"]


# ---- 1. the oracle, byte for byte --------------------------------------------------------------------------------------
@pytest.mark.parametrize("lg_n", [5, 8, 12])
def test_matches_oracle_byte_for_byte(glb, ctx, oracle, mods, lg_n):
    fri, wire, pv = mods
    pis = [3, 1, 4]
    c = _instance(oracle, lg_n, pis)
    fp = _fri_params(fri, glb, lg_n)
    p, cap = _prove(glb, ctx, c, fp, pis)
    got = _bytes(wire, p)
    want, want_cap = _oracle_bytes(wire, c, pis)
    assert np.array_equal(cap, want_cap)
    assert got == want
    assert _verify(pv, c, fp, cap, got) and _verify(pv, c, fp, want_cap, want)


# ---- 2. witness forms and public inputs -----------------------------------------------------------------------------------
def test_witness_forms_give_identical_proofs(glb, ctx, oracle, mods):
    import torch

    fri, wire, pv = mods
    pis = [9, 8]
    c = _instance(oracle, 7, pis)
    fp = _fri_params(fri, glb, 7)
    cs = _cs(glb, ctx, c)
    host, _ = _prove(glb, ctx, c, fp, pis, cs=cs)
    cols, _ = _prove(glb, ctx, c, fp, pis, cs=cs, wires=[np.ascontiguousarray(w) for w in c["wires"]])
    dev_t = torch.from_numpy(c["wires"].view(np.int64)).to(f"cuda:{ctx.device}")
    tens, _ = _prove(glb, ctx, c, fp, pis, cs=cs, wires=dev_t)
    buf = glb.DeviceBuffer(c["wires"].shape, ctx).from_host(c["wires"])
    dbuf, _ = _prove(glb, ctx, c, fp, pis, cs=cs, wires=buf)
    buf.free()
    for other in (cols, tens, dbuf):
        assert np.array_equal(other["words"], host["words"])
    assert _verify(pv, c, fp, cs.merkle_tree.cap, _bytes(wire, host))
    cs.free()


@pytest.mark.parametrize("num_pis", [0, 1, 9])
def test_public_inputs(glb, ctx, oracle, mods, num_pis):
    fri, wire, pv = mods
    pis = [(1000003 * i + 17) % P for i in range(num_pis)]
    c = _instance(oracle, 6, pis, seed=40 + num_pis)
    fp = _fri_params(fri, glb, 6)
    p, cap = _prove(glb, ctx, c, fp, pis)
    data = _bytes(wire, p)
    assert _verify(pv, c, fp, cap, data)
    assert p["public_inputs"].tolist() == pis
    if num_pis == 0:
        assert not c["pih"].any()      # hash_n_to_m_no_pad of nothing


# ---- 3. geometry ------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("nch,times_x", [(1, False), (3, False), (2, True)])
def test_geometry_variants(glb, ctx, oracle, mods, nch, times_x):
    fri, wire, pv = mods
    pis = [5]
    c = _instance(oracle, 6, pis, nch=nch)
    fp = _fri_params(fri, glb, 6, times_x)
    p, cap = _prove(glb, ctx, c, fp, pis)
    got = _bytes(wire, p)
    assert p["openings"]["plonk_zs"].shape == (nch, 2) and p["openings"]["quotient_polys"].shape == (8 * nch, 2)
    assert got == _oracle_bytes(wire, c, pis, times_x)[0]
    assert _verify(pv, c, fp, cap, got)


# ---- 4. full size -----------------------------------------------------------------------------------------------------------
def test_reference_circuit_2_16_caps_match_oracle_stages(glb, ctx, oracle, mods):
    from oracle import fri_oracle

    fri, wire, pv = mods
    lg_n, pis = 16, [7, 7, 7]
    c = _instance(oracle, lg_n, pis)
    fp = _fri_params(fri, glb, lg_n)
    p, cap = _prove(glb, ctx, c, fp, pis)
    assert _verify(pv, c, fp, cap, _bytes(wire, p))
    # the oracle's stages on the transcript the proof's caps imply
    ch = fri_oracle.Challenger()
    ch.observe_hash(DIGEST)
    ch.observe_hash(c["pih"])
    w = oracle.commit_from_values(c["wires"], 3, 4)
    assert np.array_equal(p["caps"][0], w["cap"])
    ch.observe_cap(w["cap"])
    betas, gammas = [ch.get_challenge() for _ in range(2)], [ch.get_challenge() for _ in range(2)]
    zs = oracle.permutation_zs(c["circuit"], c["k_is"], c["wires"], c["sigmas"], betas, gammas)
    z = oracle.commit_from_values(zs, 3, 4)
    assert np.array_equal(p["caps"][1], z["cap"])
    ch.observe_cap(z["cap"])
    alphas = [ch.get_challenge() for _ in range(2)]
    cs_leaves = oracle.commit_from_values(np.concatenate([c["constants"], c["sigmas"]]), 3, 4)["leaves"]
    q = oracle.quotient_polys(c["circuit"], c["gates"], c["k_is"], cs_leaves, w["leaves"], z["leaves"], 3, c["pih"], betas, gammas, alphas)
    assert np.array_equal(p["caps"][2], oracle.commit_from_coeffs(q, 3, 4, want_leaves=False)["cap"])


@pytest.mark.parametrize("lg_n", [18, 20])
def test_fullsize_vectorised_instance_verifies(glb, ctx, oracle, mods, lg_n):
    fri, wire, pv = mods
    pis = [1, 2, 3, 4, 5]
    c = large(lg_n, pis, seed=lg_n)
    fp = _fri_params(fri, glb, lg_n)
    p, cap = _prove(glb, ctx, c, fp, pis)
    assert _verify(pv, c, fp, cap, _bytes(wire, p))


# ---- 5. rejection -----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("corrupt", ["bit", "copy"])
def test_bad_witness_proves_and_is_rejected(glb, ctx, oracle, mods, corrupt):
    fri, wire, pv = mods
    pis = [2]
    c = _instance(oracle, 7, pis, seed=3, corrupt=corrupt)
    fp = _fri_params(fri, glb, 7)
    p, cap = _prove(glb, ctx, c, fp, pis)        # GL_OK: upstream's prover does not check the witness
    with pytest.raises(pv.PlonkVerifyError):
        _verify(pv, c, fp, cap, _bytes(wire, p))


def _flip(data, byte_offset):
    v = int.from_bytes(data[byte_offset:byte_offset + 8], "little")
    return data[:byte_offset] + ((v + 1) % P).to_bytes(8, "little") + data[byte_offset + 8:]


@pytest.mark.parametrize("where", ["cap", "opening", "quotient_opening", "fri", "public_input"])
def test_tampered_proof_is_rejected(glb, ctx, oracle, mods, where):
    fri, wire, pv = mods
    pis = [6, 28]
    lg_n = 8
    c = _instance(oracle, lg_n, pis, seed=9)
    fp = _fri_params(fri, glb, lg_n)
    p, cap = _prove(glb, ctx, c, fp, pis)
    data = _bytes(wire, p)
    assert _verify(pv, c, fp, cap, data)
    lens = glb.host.opening_set_lengths(c["circuit"])
    caps_b = 3 * (4 << 4) * 8
    before = lambda f: caps_b + 16 * sum(lens[g] for g in wire.OPENING_SET_FIELDS[:wire.OPENING_SET_FIELDS.index(f)])  # noqa: E731
    off = {"cap": 8 * 5, "opening": before("wires") + 16 * 3, "quotient_opening": before("quotient_polys") + 16 * 5 + 8,
           "fri": caps_b + 16 * sum(lens.values()) + 8 * 7, "public_input": len(data) - 8}[where]
    with pytest.raises(pv.PlonkVerifyError):
        _verify(pv, c, fp, cap, _flip(data, off))


def test_wrong_number_of_public_inputs_is_rejected(glb, ctx, oracle, mods):
    fri, wire, pv = mods
    pis = [4, 5]
    c = _instance(oracle, 6, pis, seed=12)
    fp = _fri_params(fri, glb, 6)
    p, cap = _prove(glb, ctx, c, fp, pis)
    data = _bytes(wire, p)
    for count in (1, 3):
        with pytest.raises(pv.PlonkVerifyError):
            pv.verify_proof(data, pv.CommonData(c["circuit"], c["gates"], c["k_is"], fp, count), pv.VerifierData(cap, DIGEST))


# ---- 6. argument checks -------------------------------------------------------------------------------------------------------
def _raw(glb, ctx, fri, c, cs, fp, out_words=None, digest=DIGEST):
    cd = glb._native.Circuit(*[int(v) for v in c["circuit"]])
    gates = (glb._native.Gate * len(c["gates"]))(*[glb._native.Gate(*[int(v) for v in g[:5]], 0) for g in c["gates"]])
    prm = fri.c_params(fp)
    words = C.c_uint64(0)
    out = np.empty(out_words or 1, dtype=np.uint64)
    rc = ctx._lib.gl_prove(ctx._h, C.byref(cd), gates, c["k_is"].ctypes.data, cs._h, None if digest is None else digest.ctypes.data,
                           C.byref(prm), c["wires"].ctypes.data, None, 0, None, 0, out.ctypes.data if out_words else None,
                           out_words or 0, C.byref(words))
    return rc, words.value


def test_argument_checks(glb, ctx, oracle, mods):
    fri, wire, pv = mods
    c = _instance(oracle, 6, [])
    fp = _fri_params(fri, glb, 6)
    cs = _cs(glb, ctx, c)
    rc, words = _raw(glb, ctx, fri, c, cs, fp)                       # no buffer: the size is still reported
    assert rc == 1 and words > 0
    assert _raw(glb, ctx, fri, c, cs, fp, out_words=words - 1) == (1, words)    # one word short
    assert _raw(glb, ctx, fri, c, cs, fp, out_words=words)[0] == 0
    assert _raw(glb, ctx, fri, c, cs, fp, out_words=words, digest=None)[0] == 1  # NULL argument
    short = glb.PolynomialBatch.from_values(np.concatenate([c["constants"], c["sigmas"][:-1]]), 3, False, 4, ctx=ctx)
    assert _raw(glb, ctx, fri, c, short, fp, out_words=words)[0] == 1           # num_constants + R - 1 columns
    short.free()
    for cfg in (glb.FriConfig(rate_bits=2), glb.FriConfig(cap_height=3)):       # prm does not match constants_sigmas
        other = fri.FriParams.for_degree(cfg, 6)
        assert _raw(glb, ctx, fri, c, cs, other, out_words=1 << 22)[0] == 1
    blinded = glb.PolynomialBatch.from_values(np.concatenate([c["constants"], c["sigmas"]]), 3, True, 4, ctx=ctx)
    assert _raw(glb, ctx, fri, c, blinded, fp, out_words=1 << 22)[0] == 1
    blinded.free()
    with pytest.raises(glb.GlPanic) as e:                            # the same through the mirror
        glb.host.prove((6, 135, 80, 5, 2, 2, 8, 6), c["gates"], c["k_is"], cs, DIGEST, fp, c["wires"], [], ctx=ctx)
    assert e.value.code == 1
    # a witness the library would read past: every form is checked in the mirror
    import torch

    short = [c["wires"][:, :32], c["wires"][:134], [np.ascontiguousarray(w) for w in c["wires"][:134]],
             [np.ascontiguousarray(w[:32]) for w in c["wires"]], torch.zeros((134, 64), dtype=torch.int64, device=f"cuda:{ctx.device}"),
             glb.DeviceBuffer((135, 32), ctx)]
    for w in short:
        with pytest.raises(glb.GlPanic) as e:
            glb.host.prove(c["circuit"], c["gates"], c["k_is"], cs, DIGEST, fp, w, [], ctx=ctx)
        assert e.value.code == 1
    short[-1].free()
    # the ctx proves the next instance correctly
    p, cap = _prove(glb, ctx, c, fp, [], cs=cs)
    assert _verify(pv, c, fp, cap, _bytes(wire, p))
    cs.free()


# ---- 7. the C++ mirror --------------------------------------------------------------------------------------------------------
def test_cpp_mirror_matches_python_mirror(glb, ctx, mods, tmp_path):
    """tests/cpp/prove_mirror_test.cpp proves a fixed instance through plonky2_b200.hpp and dumps the words; the Python mirror
    proves the same instance."""
    fri, wire, pv = mods
    exe, dump = str(tmp_path / "prove_mirror_test"), str(tmp_path / "proof.txt")
    libdir = os.path.join(ROOT, "plonky2-lib_b200")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-Wall", "-I", os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "tests", "cpp", "prove_mirror_test.cpp"), "-L", libdir, "-lgl_b200",
                           f"-Wl,-rpath,{libdir}", "-o", exe])
    out = subprocess.run([exe, dump], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stdout + out.stderr
    got = [int(x) for x in open(dump).read().split()]

    def splitmix(x):
        x = (x + 0x9E3779B97F4A7C15) & 0xFFFFFFFFFFFFFFFF
        x = ((x ^ (x >> 30)) * 0xBF58476D1CE4E5B9) & 0xFFFFFFFFFFFFFFFF
        x = ((x ^ (x >> 27)) * 0x94D049BB133111EB) & 0xFFFFFFFFFFFFFFFF
        x ^= x >> 31
        return x % P if x >= P else x

    lg_n, R, num_wires, num_constants = 6, 20, 24, 3
    n = 1 << lg_n
    pis = [5, 6, 7]
    wires = np.array([[splitmix((j << 32) + i) for i in range(n)] for j in range(num_wires)], dtype=np.uint64)
    cs = np.zeros((num_constants + R, n), dtype=np.uint64)
    cs[0, 0] = 2
    wires[0:4, 0] = glb.PoseidonHash.hash_no_pad(np.array(pis, dtype=np.uint64), ctx=ctx)
    for i in range(1, n):
        if i % 5 == 1:
            cs[0, i] = 1
            cs[1, i] = wires[0, i] = splitmix((200 << 32) + i)
            cs[2, i] = wires[1, i] = splitmix((201 << 32) + i)
    k_is = np.array([pow(7, j, P) for j in range(R)], dtype=np.uint64)
    cs[num_constants:] = identity_sigmas(k_is, lg_n)
    for t in range(8):
        a, b = (num_constants + t + 4, 2 * t + 3), (num_constants + t + 10, 5 * t + 7)
        cs[a], cs[b] = cs[b], cs[a]
        wires[t + 10, 5 * t + 7] = wires[t + 4, 2 * t + 3]
    circuit = (lg_n, num_wires, R, num_constants, 1, 2, 8, 3)
    gates = [(0, 0, 0, 0, 3, 0), (1, 2, 0, 0, 3, 0), (2, 0, 0, 0, 3, 0)]
    csb = glb.PolynomialBatch.from_values(cs, 3, False, 4, ctx=ctx)
    fp = _fri_params(fri, glb, lg_n)
    p = glb.host.prove(circuit, gates, k_is, csb, np.array([1, 2, 3, 4], dtype=np.uint64), fp, wires, pis, ctx=ctx)
    assert got == [int(x) for x in p["words"]]
    assert pv.verify_proof(_bytes(wire, p), pv.CommonData(circuit, gates, k_is, fp, len(pis)),
                           pv.VerifierData(csb.merkle_tree.cap, np.array([1, 2, 3, 4], dtype=np.uint64)))
    csb.free()
