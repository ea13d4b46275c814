"""The Poseidon schedule of csrc/poseidon.cuh restated bit for bit in numpy, against the oracle's permutation:

  * gl_sqr's three-product chain and gl_reduce128, on 32-bit limbs with 64-bit wrap-around;
  * the S-box hand-off: (dl, dh) = (r0 - r2 - r3 + 2^33, r1 + r2) of the last 128-bit product, as 64-bit integers whose bit
    patterns are read as float64 denormals;
  * the constant tables of poseidon_constants.h (linear_layer_tables with the signed offsets and the hand-off bias taken
    back out), restated from the same formulas;
  * the full round and the fused partial pair through the 4 x 3 Good-Thomas FFT (poseidon_circ12) on float64 denormals
    (numpy does not flush denormals; every product and sum is exact, so a fused multiply-add and a multiply followed by
    an add give the same bits);
  * the fold (A - bh) + 2^32 (bh + b0) with its single wrap.

Next to the model: an exact interval analysis in Python integers of every FP64 intermediate of both layer kinds, and the
check that every table offset is 0 mod p.  The device itself is checked against the oracle in tests/test_gpu_parity.py and
tests/test_gpu_fullsize.py; tools/poseidon_bench checks the FFT form on the same extreme patterns on the GPU."""
import numpy as np
import pytest

from oracle import pyoracle as o

P = 0xFFFFFFFF00000001
M32 = np.uint64(0xFFFFFFFF)
S32 = np.uint64(32)
CIRC = [17, 15, 41, 16, 2, 28, 13, 13, 39, 18, 34, 20]
DIAG0 = 8
HANDOFF_BIAS = 1 << 33  # POSEIDON_HANDOFF_BIAS
FULL_OFF = ((1 << 42) + 1, 0xFFFFFFFF - (1 << 10))  # (A, B) offsets of one layer
PAIR_OFF = ((1 << 48) + (1 << 16), (1 << 16) * 0xFFFFFFFF - (1 << 16))  # of the fused pair


def mds(r, j):
    return CIRC[(j - r) % 12] + (DIAG0 if r == j == 0 else 0)


def pair_entry(r, j):  # N = M M' without the lane-0 path
    return sum(mds(r, i) * mds(i, j) for i in range(1, 12))


def circ2(r, j):
    return sum(CIRC[(m - r) % 12] * CIRC[(j - m) % 12] for m in range(12))


def c0(r):  # col0(CIRC)
    return mds(r, 0) - (DIAG0 if r == 0 else 0)


# ---------------------------------------------------------------------------------------------------------------------
# tables (poseidon_constants.h: linear_layer_tables(rc, CIRC, 8, true, split, pk, POSEIDON_HANDOFF_BIAS))
# ---------------------------------------------------------------------------------------------------------------------
def full_layer(rnd):
    return 1 <= rnd <= 4 or 27 <= rnd <= 30


def lane0_only(rnd):
    return 5 <= rnd <= 25 and rnd % 2 == 1


def split_weight(rnd, lane):  # total weight of the S-box outputs in the row this entry is added to
    if full_layer(rnd):
        return sum(mds(lane, j) for j in range(12))
    return mds(0, 0)


def pair_weight(lane):
    return pair_entry(lane, 0) + mds(lane, 0)


def tables(rc, bias=HANDOFF_BIAS):
    split = [[0, 0] for _ in range(31 * 12)]
    plain_split = [[0, 0] for _ in range(31 * 12)]
    for i in range(31 * 12):
        v = int(rc[i]) if i < 360 else 0
        split[i] = [v & 0xFFFFFFFF, v >> 32]
        plain_split[i] = list(split[i])
    for rnd in range(31):
        for lane in range(12):
            if full_layer(rnd) or (lane0_only(rnd) and lane == 0):
                split[rnd * 12 + lane][0] += FULL_OFF[0] - bias * split_weight(rnd, lane)
                split[rnd * 12 + lane][1] += FULL_OFF[1]
    pk, plain_pk = [], []
    for pair in range(11):
        r1 = rc[(5 + 2 * pair) * 12:(6 + 2 * pair) * 12]
        r2 = rc[(6 + 2 * pair) * 12:(7 + 2 * pair) * 12]
        for lane in range(12):
            lo = (int(r2[lane]) & 0xFFFFFFFF) + sum(mds(lane, i) * (int(r1[i]) & 0xFFFFFFFF) for i in range(1, 12))
            hi = (int(r2[lane]) >> 32) + sum(mds(lane, i) * (int(r1[i]) >> 32) for i in range(1, 12))
            plain_pk.append([lo, hi])
            pk.append([lo + PAIR_OFF[0] - bias * pair_weight(lane), hi + PAIR_OFF[1]])
    for t in split + pk:
        assert 0 <= t[0] < 1 << 52 and 0 <= t[1] < 1 << 52  # stored as non-negative denormal bit patterns
    return split, pk, plain_split, plain_pk


@pytest.fixture(scope="module")
def rc():
    return [int(v) for v in o.round_constants()]


# ---------------------------------------------------------------------------------------------------------------------
# the device's arithmetic on uint64 arrays
# ---------------------------------------------------------------------------------------------------------------------
def limbs(x):
    return x & M32, x >> S32


def mul128(a, b):
    """(lo, hi) of the 128-bit product, as gl_mul's IMAD.WIDE chain forms it."""
    a0, a1 = limbs(a)
    b0, b1 = limbs(b)
    p00, p01, p10, p11 = a0 * b0, a0 * b1, a1 * b0, a1 * b1
    t = (p00 >> S32) + (p01 & M32) + (p10 & M32)
    t2 = (t >> S32) + (p01 >> S32) + (p10 >> S32) + (p11 & M32)
    r3 = (t2 >> S32) + (p11 >> S32)
    return (p00 & M32) | ((t & M32) << S32), (t2 & M32) | (r3 << S32)


def sqr128(a):
    """gl_sqr: l + 2^32 (m + m) + 2^64 h, the cross product added twice by a 32-bit carry chain."""
    a0, a1 = limbs(a)
    l, m, h = a0 * a0, a0 * a1, a1 * a1
    c = (l >> S32) + (m & M32)  # add.cc  r1 = l1 + m0
    r1 = c & M32
    c = (c >> S32) + (h & M32) + (m >> S32)  # addc.cc r2 = h0 + m1
    r2 = c & M32
    r3 = ((c >> S32) + (h >> S32)) & M32  # addc
    c = r1 + (m & M32)  # add.cc  r1 += m0
    r1 = c & M32
    c = (c >> S32) + r2 + (m >> S32)  # addc.cc r2 += m1
    r2 = c & M32
    r3 = (r3 + (c >> S32)) & M32  # addc
    return (l & M32) | (r1 << S32), r2 | (r3 << S32)


def reduce128(lo, hi):
    """gl_reduce128: (r0 + 2^32 r1) + 2^32 r2 - (r2 + r3), the net wrap folded back as k (2^32 - 1), mod 2^64."""
    r2, r3 = limbs(hi)
    with np.errstate(over="ignore"):
        w = lo + (r2 << S32)
        k = (w < lo).astype(np.int64)
        g = r2 + r3
        w2 = w - g
        k -= (w < g).astype(np.int64)
        return w2 + (k * 0xFFFFFFFF).astype(np.uint64)


def gl_mul(a, b):
    return reduce128(*mul128(a, b))


def gl_sqr(a):
    return reduce128(*sqr128(a))


def handoff(x):
    """poseidon_sbox_split: x^7 as (dl, dh) bit patterns, dl = r0 - r2 - r3 + 2^33, dh = r1 + r2."""
    x2 = gl_sqr(x)
    x4 = gl_sqr(x2)
    x3 = gl_mul(x2, x)
    lo, hi = mul128(x3, x4)
    r0, r1 = limbs(lo)
    r2, r3 = limbs(hi)
    dl = np.uint64(HANDOFF_BIAS) + r0 - r2 - r3
    dh = r1 + r2
    return dl, dh


def fold(al, ah):
    """poseidon_fold on float64 accumulators: (A - bh) + 2^32 (bh + b0), one wrap folded back as 2^32 - 1."""
    A, B = al.view(np.uint64), ah.view(np.uint64)
    assert (A < np.uint64(1 << 50)).all() and (B < np.uint64(1 << 50)).all() and (al >= 0).all() and (ah >= 0).all()
    bh, b0 = B >> S32, B & M32
    assert (A >= bh).all()
    s = (A - bh) + ((bh + b0) << S32)  # mod 2^64
    c = (((A - bh) >> S32) + bh + b0) >> S32  # the wrap
    return s + c * np.uint64(0xFFFFFFFF)


def den(u):
    return np.ascontiguousarray(u, dtype=np.uint64).view(np.float64)


K0 = [[16., 32., 16.], [5120., 5120., 6144.]]
K2 = [[-1., 8., 2.], [132., -48., 240.]]
KR = [[2., -1., -16.], [54., 486., -162.]]
KI = [[1., 4., 1.], [-252., -36., -72.]]
IDX = [[0, 4, 8], [9, 1, 5], [6, 10, 2], [3, 7, 11]]


def circ12(x, sq, ops=None):
    """poseidon_circ12<SQ> in the device's operation order.  x: list of 12 arrays (float64, or Python-int linear forms when
    `ops` collects the intermediates for the interval analysis)."""
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
        v0 = rec(rec(rec(rec(K0[sq][0] * U0[b]) + rec(K0[sq][1] * U0[b1])) + rec(K0[sq][2] * U0[b2])))
        v2 = rec(rec(rec(K2[sq][0] * U2[b]) + rec(K2[sq][1] * U2[b1])) + rec(K2[sq][2] * U2[b2]))
        vr, vi = rec(KR[sq][0] * UR[b]), rec(KR[sq][0] * UI[b])
        for kk, (src_r, src_i) in enumerate(((UR[b], UI[b]), (UR[b1], UI[b1]), (UR[b2], UI[b2]))):
            if kk:
                vr = rec(vr + rec(KR[sq][kk] * src_r))
                vi = rec(vi + rec(KR[sq][kk] * src_i))
            vr = rec(vr + rec(-KI[sq][kk] * src_i))
            vi = rec(vi + rec(KI[sq][kk] * src_r))
        sm, df = rec(v0 + v2), rec(v0 - v2)
        y[IDX[0][b]], y[IDX[2][b]] = rec(sm + vr), rec(sm - vr)
        y[IDX[1][b]], y[IDX[3][b]] = rec(df - vi), rec(df + vi)
    return y


def permute_model(states, rc, split, pk):
    """poseidon_permute on an (n, 12) uint64 array, in the device's schedule."""
    s = [states[:, i].copy() for i in range(12)]
    with np.errstate(over="ignore"):
        for i in range(12):  # gl_add_c
            t = s[i] + np.uint64(rc[i])
            s[i] = t + np.where(t < s[i], np.uint64(0xFFFFFFFF), np.uint64(0))

        def full_round(s, rnd):
            hl = [handoff(v) for v in s]
            dl, dh = [den(h[0]) for h in hl], [den(h[1]) for h in hl]
            yl, yh = circ12(dl, 0), circ12(dh, 0)
            out = []
            for r in range(12):
                kx, ky = split[rnd * 12 + r]
                al, ah = yl[r] + den(np.uint64(kx)), yh[r] + den(np.uint64(ky))
                if r == 0:
                    al, ah = 8. * dl[0] + al, 8. * dh[0] + ah
                out.append(fold(al, ah))
            return out

        def partial_pair(s, pair):
            dl = [None] + [den(v & M32) for v in s[1:]]
            dh = [None] + [den(v >> S32) for v in s[1:]]
            yl, yh = float(mds(0, 1)) * dl[1], float(mds(0, 1)) * dh[1]
            for j in range(2, 12):
                yl, yh = float(mds(0, j)) * dl[j] + yl, float(mds(0, j)) * dh[j] + yh
            h0 = handoff(s[0])
            dl[0], dh[0] = den(h0[0]), den(h0[1])
            yl, yh = float(mds(0, 0)) * dl[0] + yl, float(mds(0, 0)) * dh[0] + yh
            kx, ky = split[(5 + 2 * pair) * 12]
            g = handoff(fold(yl + den(np.uint64(kx)), yh + den(np.uint64(ky))))
            gl, gh = den(g[0]), den(g[1])
            zl, zh = circ12(dl, 1), circ12(dh, 1)
            wl, wh = 8. * dl[0] - yl, 8. * dh[0] - yh
            out = []
            for r in range(12):
                kx, ky = pk[pair * 12 + r]
                tl, th = float(mds(r, 0)) * gl + den(np.uint64(kx)), float(mds(r, 0)) * gh + den(np.uint64(ky))
                tl, th = float(c0(r)) * wl + tl, float(c0(r)) * wh + th
                out.append(fold(zl[r] + tl, zh[r] + th))
            return out

        for rnd in range(1, 5):
            s = full_round(s, rnd)
        for pair in range(11):
            s = partial_pair(s, pair)
        for rnd in range(27, 31):
            s = full_round(s, rnd)
    out = np.stack(s, axis=1)
    return np.where(out >= np.uint64(P), out - np.uint64(P), out)  # gl_canon


# ---------------------------------------------------------------------------------------------------------------------
# tests
# ---------------------------------------------------------------------------------------------------------------------
def extreme_states():
    """The patterns tools/poseidon_bench uses, as whole 64-bit lanes: every 32-bit limb 0xffffffff, all zeros,
    alternating, one-hot; plus p - 1 and 2^64 - 1 (non-canonical inputs)."""
    rows = [[0xFFFFFFFFFFFFFFFF] * 12, [0] * 12, [P - 1] * 12, [0xFFFFFFFF00000000] * 12, [0xFFFFFFFF] * 12]
    for ph in range(2):
        rows.append([0xFFFFFFFFFFFFFFFF if (i + ph) & 1 else 0 for i in range(12)])
        rows.append([0xFFFFFFFF if (i + ph) & 1 else 0xFFFFFFFF00000000 for i in range(12)])
    for i in range(12):
        rows.append([0xFFFFFFFFFFFFFFFF if j == i else 0 for j in range(12)])
        rows.append([0xFFFFFFFF if j == i else 0 for j in range(12)])
    return np.array(rows, dtype=np.uint64)


def test_sqr_and_reduce_are_exact():
    rng = np.random.default_rng(1)
    a = rng.integers(0, 1 << 64, size=200000, dtype=np.uint64, endpoint=False)
    a[:6] = [0, 1, 0xFFFFFFFF, 0xFFFFFFFF00000000, P - 1, 0xFFFFFFFFFFFFFFFF]
    assert all(np.array_equal(u, v) for u, v in zip(sqr128(a), mul128(a, a)))
    got = gl_sqr(a)
    for x, y in zip(a[:2000].tolist(), got[:2000].tolist()):
        assert y % P == x * x % P


def test_handoff_value_and_range():
    rng = np.random.default_rng(2)
    x = rng.integers(0, 1 << 64, size=100000, dtype=np.uint64)
    x[:4] = [0, 1, P - 1, 0xFFFFFFFFFFFFFFFF]
    dl, dh = handoff(x)
    assert dl.min() >= 2 and dl.max() < 3 << 32 and dh.max() < 1 << 33
    for v, a, b in zip(x[:3000].tolist(), dl[:3000].tolist(), dh[:3000].tolist()):
        assert (a - HANDOFF_BIAS + (b << 32)) % P == pow(v, 7, P)


def test_table_offsets_are_zero_mod_p(rc):
    split, pk, plain_split, plain_pk = tables(rc)
    assert (FULL_OFF[0] + (FULL_OFF[1] << 32)) % P == 0 and (PAIR_OFF[0] + (PAIR_OFF[1] << 32)) % P == 0
    used = [(rnd, lane) for rnd in range(31) for lane in range(12) if full_layer(rnd) or (lane0_only(rnd) and lane == 0)]
    assert len(used) == 8 * 12 + 11
    for rnd, lane in used:
        (a, b), (a0, b0) = split[rnd * 12 + lane], plain_split[rnd * 12 + lane]
        # the offset the entry carries, plus what the hand-off bias adds to the accumulator it meets
        assert (a - a0 + HANDOFF_BIAS * split_weight(rnd, lane) + ((b - b0) << 32)) % P == 0
    for lane in range(12):
        for pair in range(11):
            (a, b), (a0, b0) = pk[pair * 12 + lane], plain_pk[pair * 12 + lane]
            assert (a - a0 + HANDOFF_BIAS * pair_weight(lane) + ((b - b0) << 32)) % P == 0
    # the pair's weight as the device forms it: CIRC^2 x~ + col0(CIRC) (8 x~_0 - Yraw) + M[.][0] sigma
    for r in range(12):
        assert circ2(r, 0) + c0(r) * (DIAG0 - mds(0, 0)) == pair_entry(r, 0)


def test_model_matches_oracle_on_kat_extremes_and_random(rc):
    split, pk, _, _ = tables(rc)
    iota = np.arange(12, dtype=np.uint64)[None, :]
    got = permute_model(iota, rc, split, pk)
    assert got[0, :4].tolist() == [0xd64e1e3efc5b8e9e, 0x53666633020aaa47, 0xd40285597c6a8825, 0x613a4f81e81231d2]
    ext = extreme_states()
    assert np.array_equal(permute_model(ext, rc, split, pk), o.permute_batch(ext))
    rng = np.random.default_rng(3)
    states = rng.integers(0, 1 << 64, size=(100000, 12), dtype=np.uint64)
    assert np.array_equal(permute_model(states, rc, split, pk), o.permute_batch(states))


# ---------------------------------------------------------------------------------------------------------------------
# exact interval analysis: every intermediate is a linear form in independent inputs with known ranges
# ---------------------------------------------------------------------------------------------------------------------
class Lin:
    """sum_i c_i x_i + k with exact integer coefficients; bounds() is exact for independent x_i in [lo_i, hi_i]."""

    def __init__(self, c=None, k=0):
        self.c, self.k = dict(c or {}), k

    def __add__(self, o):
        o = o if isinstance(o, Lin) else Lin(k=o)
        c = dict(self.c)
        for i, v in o.c.items():
            c[i] = c.get(i, 0) + v
        return Lin(c, self.k + o.k)

    def __neg__(self):
        return Lin({i: -v for i, v in self.c.items()}, -self.k)

    def __sub__(self, o):
        return self + (-o)

    def __rmul__(self, s):
        assert float(s).is_integer()
        s = int(s)
        return Lin({i: s * v for i, v in self.c.items()}, s * self.k)

    def bounds(self, rng):
        lo = hi = self.k
        for i, v in self.c.items():
            a, b = v * rng[i][0], v * rng[i][1]
            lo, hi = lo + min(a, b), hi + max(a, b)
        return lo, hi


DL_RANGE = (2, (3 << 32) - 1)  # r0 - r2 - r3 + 2^33
DH_RANGE = (0, (1 << 33) - 2)  # r1 + r2
HALF_RANGE = (0, 0xFFFFFFFF)  # a 32-bit half of a folded lane


def check_ops(ops, rng):
    worst = 0
    for v in ops:
        lo, hi = v.bounds(rng)
        worst = max(worst, abs(lo), abs(hi))
    assert worst < 1 << 53
    return worst


def fold_inputs_ok(A, B, rng):
    (alo, ahi), (blo, bhi) = A.bounds(rng), B.bounds(rng)
    assert 0 <= alo and ahi < 1 << 50 and 0 <= blo and bhi < 1 << 50
    assert alo >= 1 << 18  # A - bh never borrows (bh < 2^18)
    return alo, ahi, bhi


def test_interval_analysis_full_round(rc):
    split, _, _, _ = tables(rc)
    worst = 0
    for half, inp in ((0, DL_RANGE), (1, DH_RANGE)):
        x = [Lin({j: 1}) for j in range(12)]
        rng = {j: inp for j in range(12)}
        ops = []
        y = circ12(x, 0, ops)
        worst = max(worst, check_ops(ops, rng))
        for rnd in [r for r in range(31) if full_layer(r)]:
            for r in range(12):
                acc = y[r] + split[rnd * 12 + r][half]
                if r == 0:
                    acc = 8 * x[0] + acc
                lo, hi = acc.bounds(rng)
                assert 0 <= lo and hi < 1 << 50 and (half or lo >= 1 << 18)
                worst = max(worst, hi)
    assert worst < 1 << 45


def test_interval_analysis_fused_pair(rc):
    split, pk, _, _ = tables(rc)
    worst = 0
    for half, (lane0, other) in ((0, (DL_RANGE, HALF_RANGE)), (1, (DH_RANGE, HALF_RANGE))):
        x = [Lin({j: 1}) for j in range(12)]
        g = Lin({"g": 1})
        rng = {0: lane0, "g": lane0, **{j: other for j in range(1, 12)}}
        ops = []
        y = mds(0, 1) * x[1]
        for j in list(range(2, 12)) + [0]:  # lanes 1..11 first, lane 0 after its S-box: Yraw
            y = mds(0, j) * x[j] + y
            ops.append(y)
        for pair in range(11):  # y0: into the fold that feeds sigma's S-box
            acc = y + split[(5 + 2 * pair) * 12][half]
            lo, hi = acc.bounds(rng)
            assert 0 <= lo and hi < 1 << 50 and (half or lo >= 1 << 18)
        z = circ12(x, 1, ops)
        w = 8 * x[0] - y
        ops.append(w)
        for pair in range(11):
            for r in range(12):
                t = mds(r, 0) * g + pk[pair * 12 + r][half]
                t2 = c0(r) * w + t
                acc = z[r] + t2
                ops.extend([t, t2, acc])
                lo, hi = acc.bounds(rng)
                assert 0 <= lo and hi < 1 << 50 and (half or lo >= 1 << 18)
        worst = max(worst, check_ops(ops, rng))
    assert worst < 1 << 51
