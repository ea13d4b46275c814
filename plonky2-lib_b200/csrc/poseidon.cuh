// Poseidon-Goldilocks permutation (width 12, rate 8, x^7, 4 + 22 + 4 rounds), one state per thread.
//
// plonky2::hash::poseidon::{Poseidon::poseidon, PoseidonHash} -- SURVEY 8a P5.  Reached in the
// reference from PoseidonHash::two_to_one (src/smt/goldilocks_poseidon/mod.rs:165,
// src/zkdsa/account.rs:165, src/zkdsa/circuits/mod.rs:66-67), PoseidonHash::hash_pad
// (src/smt/goldilocks_poseidon/mod.rs:170) and, through data.prove(pw), from MerkleTree::new.
//
// B200 mapping (measured pipe rates: profiles/r1_pipe_peaks.json).  IMAD.WIDE.U32 issues at ~51
// lanes/clk/SM and does not overlap with ALU work, so the two halves of a round go to different
// pipes:
//   * S-box x^7: four 64x64 products (two of them squares of three 32x32 products each) = IMAD.WIDE.U32 on the
//     FMA-heavy pipe + shift-reduction on ALU; the last product is handed to the linear layer unreduced.
//   * MDS layer: on the FP64 pipe (B200 keeps full-rate DFMA).  A 32-bit half x of a lane is
//     reinterpreted as the double with bit pattern (hi = 0, lo = x), i.e. the denormal x * 2^-1074.
//     The circulant entries are <= 41 and each row sums to 264, so sum_i c_i * x_i < 2^42 stays below
//     2^52: every DFMA is exact and the accumulator's BIT PATTERN is the integer sum.  No int<->fp
//     conversion instruction is ever issued, in either direction.
//   * The next round's constants are the addend of the first DFMA of each row (a constant-bank
//     operand), so "add round constants" costs nothing.
//   * The 22 partial rounds run as 11 fused pairs (poseidon_partial_pair): two linear layers minus the
//     lane-0 path are one matrix N = M M' with entries < 2^14, still exact in FP64.  Between two pairs lanes 1..11
//     stay two doubles (poseidon_renorm), only lane 0 is folded to a 64-bit element for its S-box.
// The 12-lane state lives in 24 registers of one thread (46 during the partial rounds).  Measured: 1.39 G permutations/s on one B200.
#pragma once
#include "gl_field.cuh"

#define POSEIDON_WIDTH 12
#define POSEIDON_RATE 8
#define POSEIDON_FULL_HALF 4
#define POSEIDON_PARTIAL 22
#define POSEIDON_ROUNDS 30

// ALL_ROUND_CONSTANTS[round * 12 + lane]; filled by gl_poseidon_upload_constants() at ctx creation.
// Defined here (not extern): include this header from exactly one translation unit (hash_kernels.cu).
__constant__ u64 c_poseidon_rc[POSEIDON_ROUNDS * POSEIDON_WIDTH];
// The same constants split for the FP64 MDS: [round][lane] -> (double with bits rc & 0xffffffff,
// double with bits rc >> 32); one extra all-zero round so the last MDS adds nothing.
__constant__ double2 c_poseidon_rc_split[(POSEIDON_ROUNDS + 1) * POSEIDON_WIDTH];

#ifdef __CUDACC__
GL_D double u32_as_denormal(u32 x) { return __hiloint2double(0, (int)x); }
GL_D u64 double_bits(double d) { return (u64)__double_as_longlong(d); }

// x^7 handed to the FP64 linear layers without the last modular reduction.  The 128-bit product x^3 * x^4 =
// r0 + r1 phi + r2 phi^2 + r3 phi^3 (phi = 2^32, phi^2 = phi - 1, phi^3 = -1 mod p) is (r0 - r2 - r3) + (r1 + r2) phi.  Both
// coefficients are formed as 64-bit integers by carry chains (IADD3 / IADD3.X), and their bit patterns ARE the doubles the
// layers read (integers below 2^52 are exact denormals, no move or FP64 add is needed):
//   dl = r0 - r2 - r3 + POSEIDON_HANDOFF_BIAS in [2, 3 * 2^32),  dh = r1 + r2 in [0, 2^33).
// The bias keeps dl non-negative; the layers' constant tables take it back out (poseidon_constants.h: linear_layer_tables),
// so every accumulator the fold sees is the same integer as with the signed coefficient r0 - r2 - r3.
#define POSEIDON_HANDOFF_BIAS (1ULL << 33)
GL_D void poseidon_sbox_split(u64 x, double& dl, double& dh) {
    const u64 x2 = gl_sqr(x), x4 = gl_sqr(x2), x3 = gl_mul(x2, x);
    const unsigned __int128 p = (unsigned __int128)x3 * x4;
    const u64 lo = (u64)p, hi = (u64)(p >> 64);
    u32 l0, l1, h0, h1;
    asm("{\n\t"
        "sub.cc.u32 %0, %4, %6;\n\t"      // dl = (2 phi + r0) - r2 - r3, subtract family only
        "subc.u32 %1, 2, 0;\n\t"
        "sub.cc.u32 %0, %0, %7;\n\t"
        "subc.u32 %1, %1, 0;\n\t"
        "add.cc.u32 %2, %5, %6;\n\t"      // dh = r1 + r2
        "addc.u32 %3, 0, 0;\n\t"
        "}"
        : "=&r"(l0), "=&r"(l1), "=&r"(h0), "=&r"(h1)
        : "r"((u32)lo), "r"((u32)(lo >> 32)), "r"((u32)hi), "r"((u32)(hi >> 32)));
    dl = __longlong_as_double((long long)gl_pack(l0, l1));
    dh = __longlong_as_double((long long)gl_pack(h0, h1));
}
// (exactness: every operand is an integer multiple of 2^-1074, so FP64 sums and products are exact while they stay below
// 2^53 in magnitude.  A full round's layer sees inputs in [0, 3 * 2^32); the fused pair's CIRC^2 form sees lane 0 in
// [0, 3 * 2^32) and the other lanes in [0, 2^33) (poseidon_renorm's L and H).  tests/test_poseidon_schedule_model_cpu.py
// and tests/test_poseidon_split_pairs_model_cpu.py bound every intermediate exactly: all stay below 2^50.)

// MDS entries: M[r][j] = CIRC[(j - r) mod 12] + (r == j ? DIAG[r] : 0)
__host__ __device__ constexpr int poseidon_mds_entry(int r, int j) {
    constexpr int C[12] = {17, 15, 41, 16, 2, 28, 13, 13, 39, 18, 34, 20};
    return C[(j - r + 12) % 12] + ((r == 0 && j == 0) ? 8 : 0);
}
// N = M * M' with row 0 of M' zeroed: the part of two consecutive linear layers that does not pass through
// lane 0 (the only lane the S-box touches in a partial round).  Entries < 2^14.
__host__ __device__ constexpr int poseidon_pair_entry(int r, int j) {
    int acc = 0;
    for (int i = 1; i < 12; i++) acc += poseidon_mds_entry(r, i) * poseidon_mds_entry(i, j);
    return acc;
}

// Constants of the 11 fused pairs of partial rounds: K[pair][lane] = sum_{i>=1} M[lane][i] * rc[a+1][i] + rc[a+2][lane]
// (a = 4 + 2 * pair), split in 32-bit-half sums like c_poseidon_rc_split.
__constant__ double2 c_poseidon_pair_k[(POSEIDON_PARTIAL / 2) * POSEIDON_WIDTH];

// value = A + 2^32 B with A, B < 2^50 (integer bit patterns); bh = B >> 32 < 2^18, b0 = B mod 2^32.  2^64 = 2^32 - 1 (mod p):
//   A + 2^32 B = (A - bh) + 2^32 (bh + b0)  (mod p),
// one carry chain without a multiply.  A - bh does not borrow: the tables keep A >= 2^40 (their positive offsets).  The sum
// is below 2^64 + 2^51, so it wraps at most once; the wrap c is folded back as c * (2^32 - 1) = c * 2^32 - c, which cannot
// wrap again (the wrapped sum is below 2^51).  After the last fused pair it takes poseidon_renorm's (L, H) as they are:
// L >= 2^32 - 2^18 > H >> 32.
GL_D u64 poseidon_fold(double al, double ah) {
    const u64 A = double_bits(al), B = double_bits(ah);
    u32 y0, y1;
    asm("{\n\t"
        ".reg .u32 t, c;\n\t"
        "add.u32 t, %3, %5;\n\t"          // A1 + bh < 2^19
        "sub.cc.u32 %0, %2, %5;\n\t"      // A0 - bh
        "subc.u32 t, t, 0;\n\t"
        "add.cc.u32 %1, t, %4;\n\t"       // + b0: the wrap
        "addc.u32 c, 0, 0;\n\t"
        "add.u32 t, %1, c;\n\t"           // + c * 2^32 (no carry: after a wrap the high word is < 2^19)
        "sub.cc.u32 %0, %0, c;\n\t"       // - c
        "subc.u32 %1, t, 0;\n\t"
        "}"
        : "=&r"(y0), "=&r"(y1)
        : "r"((u32)A), "r"((u32)(A >> 32)), "r"((u32)B), "r"((u32)(B >> 32)));
    return gl_pack(y0, y1);
}

// Two consecutive partial rounds a, a + 1 in one pass over the FP64 pipe.  On entry the state holds the input
// of round a's S-box (constants already added).  With x~ = state after that S-box (lane 0 only):
//   y0 = M[0] . x~ + rc[a+1][0]                     -> S-box of round a + 1 -> sigma
//   z  = N x~ + K + M[.][0] * sigma                 (N = M M' without the lane-0 path)
// 2 folds (y0 and lane 0 of z) and 11 renormalisations instead of 24 folds; every partial sum stays below 2^50 (exact).
// ------------------------------------------------------------------------------------------------------------
// Circulant products through a 4 x 3 Good-Thomas FFT (exact, FP64 pipe).
//
// y_r = sum_i CIRC[i] x_{(i+r) mod 12} is a cyclic convolution over Z_12 = Z_4 x Z_3 (index n <-> (n mod 4, n mod 3),
// no twiddles).  A real FFT of length 4 along the Z_4 axis leaves, for the frequencies 0, 1 (complex) and 2, one
// length-3 cyclic convolution each; the inverse FFT's 1/4 is absorbed into the kernel, which stays integral
// because plonky2's MDS row was chosen that way: FFT4(row)/4 = {16,32,16}, {(2,1),(-1,4),(-16,1)}/.., {-1,8,2}.
// 90 FP64 operations per 12-vector instead of 144 multiply-adds; every intermediate is an integer below 2^50 in
// units of 2^-1074 (signed: differences can be negative denormals), so the arithmetic is exact and the final,
// non-negative results are again integer bit patterns.  SQ = 1 applies the circulant twice (kernel convolved with
// itself), which is what the fused partial-round pair needs.
// E0 adds CIRC (e e_0) = e col0(CIRC) to the result (the pair's rank-one lane-0 term): the forward FFT of e_0 is 1 in
// U0, U2 and UR of residue class b = 0, so its image after the single circulant's kernel is e {K0, K2, KR, KI}[0][b] in
// (v0, v2, vr, vi) of class b -- 12 FMAs after the kernel multiply instead of 12 multiply-adds per output lane.
template <int SQ, bool E0 = false>
GL_D void poseidon_circ12(const double x[12], double y[12], double e = 0.) {
    constexpr double K0[2][3] = {{16., 32., 16.}, {5120., 5120., 6144.}};
    constexpr double K2[2][3] = {{-1., 8., 2.}, {132., -48., 240.}};
    constexpr double KR[2][3] = {{2., -1., -16.}, {54., 486., -162.}};
    constexpr double KI[2][3] = {{1., 4., 1.}, {-252., -36., -72.}};
    constexpr int IDX[4][3] = {{0, 4, 8}, {9, 1, 5}, {6, 10, 2}, {3, 7, 11}};   // lane with (n mod 4, n mod 3) = (a, b)
    double U0[3], U2[3], UR[3], UI[3];
#pragma unroll
    for (int b = 0; b < 3; b++) {
        const double p0 = x[IDX[0][b]], p1 = x[IDX[1][b]], p2 = x[IDX[2][b]], p3 = x[IDX[3][b]];
        const double t0 = p0 + p2, t1 = p1 + p3;
        U0[b] = t0 + t1;
        U2[b] = t0 - t1;
        UR[b] = p0 - p2;      // F1 = (p0 - p2) + i (p3 - p1)
        UI[b] = p3 - p1;
    }
#pragma unroll
    for (int b = 0; b < 3; b++) {
        const int b1 = (b + 2) % 3, b2 = (b + 1) % 3;        // (b - 1) mod 3, (b - 2) mod 3
        double v0 = __fma_rn(K0[SQ][2], U0[b2], __fma_rn(K0[SQ][1], U0[b1], K0[SQ][0] * U0[b]));
        double v2 = __fma_rn(K2[SQ][2], U2[b2], __fma_rn(K2[SQ][1], U2[b1], K2[SQ][0] * U2[b]));
        double vr = KR[SQ][0] * UR[b], vi = KR[SQ][0] * UI[b];
        vr = __fma_rn(-KI[SQ][0], UI[b], vr);
        vi = __fma_rn(KI[SQ][0], UR[b], vi);
        vr = __fma_rn(KR[SQ][1], UR[b1], vr);
        vi = __fma_rn(KR[SQ][1], UI[b1], vi);
        vr = __fma_rn(-KI[SQ][1], UI[b1], vr);
        vi = __fma_rn(KI[SQ][1], UR[b1], vi);
        vr = __fma_rn(KR[SQ][2], UR[b2], vr);
        vi = __fma_rn(KR[SQ][2], UI[b2], vi);
        vr = __fma_rn(-KI[SQ][2], UI[b2], vr);
        vi = __fma_rn(KI[SQ][2], UR[b2], vi);
        if (E0) {
            v0 = __fma_rn(K0[0][b], e, v0);
            v2 = __fma_rn(K2[0][b], e, v2);
            vr = __fma_rn(KR[0][b], e, vr);
            vi = __fma_rn(KI[0][b], e, vi);
        }
        const double sm = v0 + v2, df = v0 - v2;
        y[IDX[0][b]] = sm + vr;
        y[IDX[2][b]] = sm - vr;
        y[IDX[1][b]] = df - vi;
        y[IDX[3][b]] = df + vi;
    }
}

// One full round: S-box on every lane, then out = CIRC x + 8 x_0 e_0 + rc through the FFT form (206 FP64
// operations instead of 290).
GL_D void poseidon_full_round(u64 s[12], const double2* __restrict__ rc) {
    double dl[12], dh[12], yl[12], yh[12];
#pragma unroll
    for (int j = 0; j < 12; j++) {
        poseidon_sbox_split(s[j], dl[j], dh[j]);
    }
    poseidon_circ12<0>(dl, yl);
    poseidon_circ12<0>(dh, yh);
#pragma unroll
    for (int r = 0; r < 12; r++) {
        const double2 k = rc[r];
        double al = yl[r] + k.x, ah = yh[r] + k.y;
        if (r == 0) {
            al = __fma_rn(8., dl[0], al);
            ah = __fma_rn(8., dh[0], ah);
        }
        s[r] = poseidon_fold(al, ah);
    }
}

// Lanes 1..11 between two fused pairs: the pair's accumulators A = a0 + 2^32 a1, B = b0 + 2^32 b1 (A in [2^32, 2^50),
// B < 2^50) are not folded to a field element, only brought back to two doubles the next pair's layers can read.
// 2^64 = 2^32 - 1 (mod p):
//   A + 2^32 B = (a0 - b1 + 2^32) + 2^32 (a1 - 1 + b0 + b1)  (mod p),
// L = a0 - b1 + 2^32 in [2^32 - 2^18, 2^33) (b1 < 2^18), H = a1 - 1 + b0 + b1 in [0, 2^32 + 2^19) (a1 >= 1).  The 2^32 in L
// is paid for by the -1 in H, so the value is congruent without any table offset.  Five two-input carry-chain
// instructions instead of the fold's eight plus the next pair's two zero-extensions.
GL_D void poseidon_renorm(double al, double ah, double& l, double& h) {
    const u64 A = double_bits(al), B = double_bits(ah);
    u32 l0, l1, h0, h1;
    asm("{\n\t"
        ".reg .u32 t;\n\t"
        "sub.cc.u32 %0, %4, %7;\n\t"      // L = 2^32 + a0 - b1
        "subc.u32 %1, 1, 0;\n\t"
        "add.u32 t, %5, %7;\n\t"          // a1 + b1 - 1 < 2^19
        "sub.u32 t, t, 1;\n\t"
        "add.cc.u32 %2, t, %6;\n\t"       // H = (a1 + b1 - 1) + b0
        "addc.u32 %3, 0, 0;\n\t"
        "}"
        : "=&r"(l0), "=&r"(l1), "=&r"(h0), "=&r"(h1)
        : "r"((u32)A), "r"((u32)(A >> 32)), "r"((u32)B), "r"((u32)(B >> 32)));
    l = __longlong_as_double((long long)gl_pack(l0, l1));
    h = __longlong_as_double((long long)gl_pack(h0, h1));
}

// Two consecutive partial rounds in FFT form.  With M = CIRC + 8 e0 e0^T and M' = M without its row 0,
//   N x~ = M M' x~ = CIRC^2 x~ + col0(CIRC) * (8 x~_0 - Yraw),   Yraw = M[0] . x~  (the unfolded y0 without its constant)
// and M[.][0] = col0(CIRC) + 8 e0, so
//   z = N x~ + M[.][0] sigma + K = CIRC (CIRC x~ + (w + sigma) e0) + 8 sigma e0 + K,   w = 8 x~_0 - Yraw:
// the rank-one lane-0 terms go into the frequency domain of poseidon_circ12<1, true>, 258 FP64 operations per pair.
// s0 is lane 0 as a 64-bit integer (the next S-box's input); lanes 1..11 enter and leave in split form, (xl, xh)[i] with
// value xl + 2^32 xh: the halves of a folded lane for the first pair, poseidon_renorm's (L, H) after that.
GL_D void poseidon_partial_pair(u64& s0, double xl[12], double xh[12], int pair) {
    // everything that does not depend on lane 0 first: the FP64 pipe works while lane 0 goes through its S-box
    double yl = (double)poseidon_mds_entry(0, 1) * xl[1], yh = (double)poseidon_mds_entry(0, 1) * xh[1];
#pragma unroll
    for (int j = 2; j < 12; j++) {
        yl = __fma_rn((double)poseidon_mds_entry(0, j), xl[j], yl);
        yh = __fma_rn((double)poseidon_mds_entry(0, j), xh[j], yh);
    }
    poseidon_sbox_split(s0, xl[0], xh[0]);
    yl = __fma_rn((double)poseidon_mds_entry(0, 0), xl[0], yl);      // Yraw
    yh = __fma_rn((double)poseidon_mds_entry(0, 0), xh[0], yh);
    const double2 ky = c_poseidon_rc_split[(POSEIDON_FULL_HALF + 2 * pair + 1) * 12];
    // w before sigma: across sigma's S-box only (wl, wh) stay live, not (x~_0, Yraw) as well
    const double wl = __fma_rn(8., xl[0], -yl), wh = __fma_rn(8., xh[0], -yh);
    double gl, gh;
    poseidon_sbox_split(poseidon_fold(yl + ky.x, yh + ky.y), gl, gh);
    const double el = wl + gl, eh = wh + gh;
    double zl[12], zh[12];
    poseidon_circ12<1, true>(xl, zl, el);
    poseidon_circ12<1, true>(xh, zh, eh);
    const double2* kk = c_poseidon_pair_k + pair * 12;
#pragma unroll
    for (int r = 0; r < 12; r++) {
        const double2 k = kk[r];
        const double al = zl[r] + k.x, ah = zh[r] + k.y;
        if (r == 0) s0 = poseidon_fold(__fma_rn(8., gl, al), __fma_rn(8., gh, ah));
        else poseidon_renorm(al, ah, xl[r], xh[r]);
    }
}

GL_D void poseidon_permute(u64 s[12]) {
#pragma unroll
    for (int i = 0; i < 12; i++) s[i] = gl_add_c(s[i], c_poseidon_rc[i]);
    // One copy of each block (full round, fused partial pair) keeps the kernel inside the instruction cache.
#pragma unroll 1
    for (int phase = 0; phase < 2; phase++) {
        // constants of round r + 1 go into the MDS of round r; round 30 is the all-zero row
        const double2* rc = c_poseidon_rc_split + 12 * (phase ? POSEIDON_FULL_HALF + POSEIDON_PARTIAL + 1 : 1);
#pragma unroll 1
        for (int r = 0; r < POSEIDON_FULL_HALF; r++, rc += 12) poseidon_full_round(s, rc);
        if (phase == 0) {
            double xl[12], xh[12];
#pragma unroll
            for (int i = 1; i < 12; i++) {
                xl[i] = u32_as_denormal((u32)s[i]);
                xh[i] = u32_as_denormal((u32)(s[i] >> 32));
            }
#pragma unroll 1
            for (int pair = 0; pair < POSEIDON_PARTIAL / 2; pair++) poseidon_partial_pair(s[0], xl, xh, pair);
            // the full rounds take 64-bit lanes: L + 2^32 H with L >= 2^32 - 2^18 > H >> 32, inside the fold's domain
#pragma unroll
            for (int i = 1; i < 12; i++) s[i] = poseidon_fold(xl[i], xh[i]);
        }
    }
}

// hashing::compress: state = l || r || 0000, permute, first four lanes
GL_D void poseidon_two_to_one(const u64 l[4], const u64 r[4], u64 out[4]) {
    u64 s[12];
#pragma unroll
    for (int i = 0; i < 4; i++) {
        s[i] = l[i];
        s[4 + i] = r[i];
        s[8 + i] = 0;
    }
    poseidon_permute(s);
#pragma unroll
    for (int i = 0; i < 4; i++) out[i] = gl_canon(s[i]);
}
#endif
