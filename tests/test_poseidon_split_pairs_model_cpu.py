"""The fused partial-round pairs of csrc/poseidon.cuh with lanes 1..11 carried in split form, restated bit for bit in numpy:

  * poseidon_renorm: the pair's accumulators A = a0 + 2^32 a1, B = b0 + 2^32 b1 of lanes 1..11 become
    L = a0 - b1 + 2^32, H = a1 - 1 + b0 + b1 (L + 2^32 H = A + 2^32 B - b1 p), the next pair's layer inputs;
  * the rank-one lane-0 terms in the frequency domain: z = CIRC (CIRC x~ + (w + sigma) e0) + 8 sigma e0 + K, applied by
    poseidon_circ12<1, true> after the kernel multiply;
  * lane 0 and, after the last pair, every lane folded as before.

The S-box, the fold, the full rounds and the constant tables are the ones tests/test_poseidon_schedule_model_cpu.py
restates; this file reuses them and adds the permutation against the oracle, an exact interval analysis of every FP64
intermediate of the new pair (the lane ranges are the fixed point of what the renormalisation hands the next pair), and
the preconditions of the renormalisation and the fold."""
import numpy as np
import pytest

import test_poseidon_schedule_model_cpu as base
from oracle import pyoracle as o

P = base.P
M32, S32 = base.M32, base.S32
mds, c0, den, fold, handoff = base.mds, base.c0, base.den, base.fold, base.handoff
K0, K2, KR, KI, IDX = base.K0, base.K2, base.KR, base.KI, base.IDX


@pytest.fixture(scope="module")
def rc():
    return [int(v) for v in o.round_constants()]


def circ12_e0(x, e, ops=None):
    """poseidon_circ12<1, true>(x, y, e) in the device's operation order: CIRC^2 x + CIRC (e e0)."""
    rec = (lambda v: (ops.append(v), v)[1]) if ops is not None else (lambda v: v)
    U0, U2, UR, UI = [None] * 3, [None] * 3, [None] * 3, [None] * 3
    for b in range(3):
        p0, p1, p2, p3 = (x[IDX[a][b]] for a in range(4))
        t0, t1 = rec(p0 + p2), rec(p1 + p3)
        U0[b], U2[b] = rec(t0 + t1), rec(t0 - t1)
        UR[b], UI[b] = rec(p0 - p2), rec(p3 - p1)
    y = [None] * 12
    for b in range(3):
        b1, b2 = (b + 2) % 3, (b + 1) % 3
        v0 = rec(rec(rec(rec(K0[1][0] * U0[b]) + rec(K0[1][1] * U0[b1])) + rec(K0[1][2] * U0[b2])))
        v2 = rec(rec(rec(K2[1][0] * U2[b]) + rec(K2[1][1] * U2[b1])) + rec(K2[1][2] * U2[b2]))
        vr, vi = rec(KR[1][0] * UR[b]), rec(KR[1][0] * UI[b])
        for kk, (src_r, src_i) in enumerate(((UR[b], UI[b]), (UR[b1], UI[b1]), (UR[b2], UI[b2]))):
            if kk:
                vr = rec(vr + rec(KR[1][kk] * src_r))
                vi = rec(vi + rec(KR[1][kk] * src_i))
            vr = rec(vr + rec(-KI[1][kk] * src_i))
            vi = rec(vi + rec(KI[1][kk] * src_r))
        # the image of e e0 under the single circulant's kernel: 1 in U0, U2, UR of class 0
        v0, v2 = rec(v0 + rec(K0[0][b] * e)), rec(v2 + rec(K2[0][b] * e))
        vr, vi = rec(vr + rec(KR[0][b] * e)), rec(vi + rec(KI[0][b] * e))
        sm, df = rec(v0 + v2), rec(v0 - v2)
        y[IDX[0][b]], y[IDX[2][b]] = rec(sm + vr), rec(sm - vr)
        y[IDX[1][b]], y[IDX[3][b]] = rec(df - vi), rec(df + vi)
    return y


def renorm(al, ah):
    """poseidon_renorm: (L, H) = (a0 - b1 + 2^32, a1 - 1 + b0 + b1) as float64 bit patterns."""
    A, B = al.view(np.uint64), ah.view(np.uint64)
    assert (al >= 0).all() and (ah >= 0).all()
    assert (A >= np.uint64(1 << 32)).all() and (A < np.uint64(1 << 50)).all() and (B < np.uint64(1 << 50)).all()
    a0, a1, b0, b1 = A & M32, A >> S32, B & M32, B >> S32
    return den(a0 + np.uint64(1 << 32) - b1), den(a1 - np.uint64(1) + b0 + b1)


def permute_model(states, rc, split, pk):
    """poseidon_permute on an (n, 12) uint64 array, with the split-form pairs."""
    s = [states[:, i].copy() for i in range(12)]
    with np.errstate(over="ignore"):
        for i in range(12):  # gl_add_c
            t = s[i] + np.uint64(rc[i])
            s[i] = t + np.where(t < s[i], np.uint64(0xFFFFFFFF), np.uint64(0))

        def full_round(s, rnd):
            hl = [handoff(v) for v in s]
            dl, dh = [den(h[0]) for h in hl], [den(h[1]) for h in hl]
            yl, yh = base.circ12(dl, 0), base.circ12(dh, 0)
            out = []
            for r in range(12):
                kx, ky = split[rnd * 12 + r]
                al, ah = yl[r] + den(np.uint64(kx)), yh[r] + den(np.uint64(ky))
                if r == 0:
                    al, ah = 8. * dl[0] + al, 8. * dh[0] + ah
                out.append(fold(al, ah))
            return out

        def partial_pair(s0, xl, xh, pair):
            yl, yh = float(mds(0, 1)) * xl[1], float(mds(0, 1)) * xh[1]
            for j in range(2, 12):
                yl, yh = float(mds(0, j)) * xl[j] + yl, float(mds(0, j)) * xh[j] + yh
            h0 = handoff(s0)
            xl[0], xh[0] = den(h0[0]), den(h0[1])
            yl, yh = float(mds(0, 0)) * xl[0] + yl, float(mds(0, 0)) * xh[0] + yh
            kx, ky = split[(5 + 2 * pair) * 12]
            wl, wh = 8. * xl[0] - yl, 8. * xh[0] - yh
            g = handoff(fold(yl + den(np.uint64(kx)), yh + den(np.uint64(ky))))
            gl, gh = den(g[0]), den(g[1])
            zl, zh = circ12_e0(xl, wl + gl), circ12_e0(xh, wh + gh)
            for r in range(12):
                kx, ky = pk[pair * 12 + r]
                al, ah = zl[r] + den(np.uint64(kx)), zh[r] + den(np.uint64(ky))
                if r == 0:
                    s0 = fold(8. * gl + al, 8. * gh + ah)
                else:
                    xl[r], xh[r] = renorm(al, ah)
            return s0

        for rnd in range(1, 5):
            s = full_round(s, rnd)
        xl = [None] + [den(v & M32) for v in s[1:]]
        xh = [None] + [den(v >> S32) for v in s[1:]]
        s0 = s[0]
        for pair in range(11):
            s0 = partial_pair(s0, xl, xh, pair)
        s = [s0] + [fold(xl[i], xh[i]) for i in range(1, 12)]
        for rnd in range(27, 31):
            s = full_round(s, rnd)
    out = np.stack(s, axis=1)
    return np.where(out >= np.uint64(P), out - np.uint64(P), out)  # gl_canon


# ---------------------------------------------------------------------------------------------------------------------
# the permutation against the oracle
# ---------------------------------------------------------------------------------------------------------------------
def test_model_matches_oracle_on_kat_extremes_and_random(rc):
    split, pk, _, _ = base.tables(rc)
    iota = np.arange(12, dtype=np.uint64)[None, :]
    got = permute_model(iota, rc, split, pk)
    assert got[0, :4].tolist() == [0xd64e1e3efc5b8e9e, 0x53666633020aaa47, 0xd40285597c6a8825, 0x613a4f81e81231d2]
    ext = base.extreme_states()
    assert np.array_equal(permute_model(ext, rc, split, pk), o.permute_batch(ext))
    rng = np.random.default_rng(4)
    states = rng.integers(0, 1 << 64, size=(100000, 12), dtype=np.uint64)
    assert np.array_equal(permute_model(states, rc, split, pk), o.permute_batch(states))


# ---------------------------------------------------------------------------------------------------------------------
# the two forms, exactly
# ---------------------------------------------------------------------------------------------------------------------
def test_renorm_is_the_value_less_a_multiple_of_p():
    rng = np.random.default_rng(5)
    A = rng.integers(1 << 32, 1 << 50, size=200000, dtype=np.uint64)
    B = rng.integers(0, 1 << 50, size=200000, dtype=np.uint64)
    b1max = (1 << 50) - 1 >> 32
    # the extremes: b1 at its maximum, a0 = 0, b0 = 0xffffffff, a1 = 1, and the corners of A and B
    A[:6] = [1 << 32, 1 << 32, (1 << 50) - 1, b1max << 32, 1 << 32, (1 << 50) - (1 << 32)]
    B[:6] = [(1 << 50) - 1, 0, (1 << 50) - 1, (b1max << 32) | 0xFFFFFFFF, 0xFFFFFFFF, b1max << 32]
    L, H = renorm(den(A), den(B))
    L, H = L.view(np.uint64), H.view(np.uint64)
    assert L.min() >= (1 << 32) - b1max and L.max() < 1 << 33 and H.max() < (1 << 32) + (1 << 19)
    for a, b, l, h in zip(A.tolist(), B.tolist(), L.tolist(), H.tolist()):
        assert l + (h << 32) == a + (b << 32) - (b >> 32) * P
    # and the fold after the last pair takes (L, H) as it is
    y = fold(den(L), den(H))
    for l, h, v in zip(L[:5000].tolist(), H[:5000].tolist(), y[:5000].tolist()):
        assert v % P == (l + (h << 32)) % P


def test_rank_one_terms_in_the_frequency_domain():
    """circ12_e0(x, e) + 8 sigma e0 is the old CIRC^2 x + col0(CIRC) w + M[.][0] sigma, as exact linear forms."""
    x = [Lin({j: 1}) for j in range(12)]
    w, g = Lin({"w": 1}), Lin({"g": 1})
    new = circ12_e0(x, w + g)
    old = base.circ12(x, 1)
    for r in range(12):
        a = new[r] + (8 * g if r == 0 else 0)
        b = old[r] + c0(r) * w + mds(r, 0) * g
        assert {k: v for k, v in a.c.items() if v} == {k: v for k, v in b.c.items() if v} and a.k == b.k


# ---------------------------------------------------------------------------------------------------------------------
# exact interval analysis of the new pair
# ---------------------------------------------------------------------------------------------------------------------
Lin = base.Lin
HALF_RANGE = base.HALF_RANGE  # a 32-bit half of a folded lane: the first pair's lanes 1..11


def union(a, b):
    return min(a[0], b[0]), max(a[1], b[1])


def pair_bounds(split, pk, lanes):
    """Every FP64 intermediate of one pair for lanes 1..11 in lanes[half]; returns the worst magnitude and the range of
    each half's accumulators handed to poseidon_renorm (rows 1..11), after checking every fold and renorm precondition."""
    worst, acc_range = 0, []
    for half, lane0 in ((0, base.DL_RANGE), (1, base.DH_RANGE)):
        x = [Lin({j: 1}) for j in range(12)]
        g = Lin({"g": 1})
        rng = {0: lane0, "g": lane0, **{j: lanes[half] for j in range(1, 12)}}
        ops = []
        y = mds(0, 1) * x[1]
        for j in list(range(2, 12)) + [0]:  # Yraw
            y = mds(0, j) * x[j] + y
            ops.append(y)
        for pair in range(11):  # y0: into the fold that feeds sigma's S-box
            lo, hi = (y + split[(5 + 2 * pair) * 12][half]).bounds(rng)
            assert 0 <= lo and hi < 1 << 50 and (half or lo >= 1 << 18)
        w = 8 * x[0] - y
        e = w + g
        ops += [w, e]
        z = circ12_e0(x, e, ops)
        lo_acc, hi_acc = 1 << 64, 0
        for pair in range(11):
            for r in range(12):
                acc = z[r] + pk[pair * 12 + r][half]
                ops.append(acc)
                if r == 0:
                    acc = 8 * g + acc
                    ops.append(acc)
                lo, hi = acc.bounds(rng)
                assert 0 <= lo and hi < 1 << 50
                if half == 0:
                    assert lo >= (1 << 32 if r else 1 << 18)  # renorm: a1 >= 1; fold: A - bh does not borrow
                if r:
                    lo_acc, hi_acc = min(lo_acc, lo), max(hi_acc, hi)
        acc_range.append((lo_acc, hi_acc))
        worst = max(worst, base.check_ops(ops, rng))
    return worst, acc_range


def test_interval_analysis_split_pairs(rc):
    split, pk, _, _ = base.tables(rc)
    lanes = [HALF_RANGE, HALF_RANGE]
    for _ in range(10):  # the lane ranges the renormalisation hands on, to their fixed point
        worst, ((alo, ahi), (blo, bhi)) = pair_bounds(split, pk, lanes)
        assert alo >= 1 << 32 and ahi < 1 << 50 and blo >= 0 and bhi < 1 << 50
        L = ((1 << 32) - (bhi >> 32), (1 << 33) - 1)
        H = ((alo >> 32) - 1, (ahi >> 32) - 1 + 0xFFFFFFFF + (bhi >> 32))
        new = [union(HALF_RANGE, L), union(HALF_RANGE, H)]
        if new == lanes:
            break
        lanes = new
    else:
        pytest.fail("lane ranges did not settle")
    assert worst < 1 << 50  # (2^49.6; exact below 2^53)
    assert lanes[0][1] < 1 << 33 and lanes[1][1] < (1 << 32) + (1 << 19)
    # the fold after the last pair: A = L >= 2^32 - 2^18 > B >> 32 (B = H < 2^33), both below 2^50
    assert L[0] >= 1 << 31 and H[1] < 1 << 33
