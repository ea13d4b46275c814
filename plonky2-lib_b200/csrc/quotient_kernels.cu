// N3: compute_quotient_polys on the device (plonky2::plonk::prover step 8, vanishing_poly.rs
// eval_vanishing_poly_base_batch): for every point of the n * 2^quotient_degree_bits coset, the alpha-reduced sum of
//   * the permutation argument: L_0(x) (Z(x) - 1) and the partial-product checks prev * prod(num) - next * prod(den),
//   * every gate's constraints times its selector filter (gate.rs compute_filter),
// divided by Z_H(x).  Gates: upstream's NoopGate / ConstantGate / PublicInputGate and the reference's own three:
//   U32InterleaveGate      /root/reference/src/u32/gates/interleave_u32.rs:89-126   (packed form :230-266)
//   UninterleaveToU32Gate  /root/reference/src/u32/gates/uninterleave_to_u32.rs:98-145
//   UninterleaveToB32Gate  /root/reference/src/u32/gates/uninterleave_to_b32.rs:101-149
// reached from every data.prove(pw) of a circuit that uses them (src/hash/keccak256.rs:248).
//
// One thread per LDE row, in LEAF order: the three oracles are resident column-major with leaf order along the fast axis
// (get_lde_values(i, step) = leaves[reverse_bits(i * step)], and the rows with i * step a multiple of step are the FIRST
// n << qdb leaves), so a warp reads 256 contiguous bytes per column and every LDE value is read once; only the nch
// quotient values per point are scattered to their natural index for the coset_ifft that follows.
// The terms are never materialised: term t of the list upstream hands to reduce_with_powers_multi enters as
// alpha_c^t * term (table apow), and a gate's slots as filter * sum_j alpha_c^(t0 + j) * constraint_j (linearity).
#include <cuda_runtime.h>

#include "gl_field.cuh"
#include "quotient_kernels.h"

#define Q_BLOCK 128
#define Q_UNUSED_SELECTOR 0xFFFFFFFFULL

unsigned quotient_gate_constraints(const gl_gate& g) {
    switch (g.kind) {
        case GL_GATE_CONSTANT: return g.num_ops;
        case GL_GATE_PUBLIC_INPUT: return 4;
        case GL_GATE_U32_INTERLEAVE: return g.num_ops * 34;
        case GL_GATE_UNINTERLEAVE_TO_U32:
        case GL_GATE_UNINTERLEAVE_TO_B32: return g.num_ops * 67;
        default: return 0;
    }
}

GL_D u64 q_inv(u64 a) { return gl_pow(a, GL_P - 2); }

// ---- 160-bit unreduced accumulators ---------------------------------------------------------------------------------------
// The alpha-weighted sums of a gate's constraints and the binary / base-4 recompositions of its bit wires are sums of
// hundreds of products: they are accumulated as plain integers (five 32-bit limbs, carry chains) and reduced mod p once,
// instead of one modular reduction + modular add per term.
struct acc160 {
    u32 w0, w1, w2, w3, w4;
};
GL_D acc160 acc_zero() { return {0u, 0u, 0u, 0u, 0u}; }
// acc += a * b  (a, b any u64; at most 2^31 such terms fit)
GL_D void acc_mad(acc160& c, u64 a, u64 b) {
    const unsigned __int128 p = (unsigned __int128)a * b;
    const u64 lo = (u64)p, hi = (u64)(p >> 64);
    asm("add.cc.u32 %0, %0, %5;\n\taddc.cc.u32 %1, %1, %6;\n\taddc.cc.u32 %2, %2, %7;\n\taddc.cc.u32 %3, %3, %8;\n\taddc.u32 %4, %4, 0;"
        : "+r"(c.w0), "+r"(c.w1), "+r"(c.w2), "+r"(c.w3), "+r"(c.w4)
        : "r"((u32)lo), "r"((u32)(lo >> 32)), "r"((u32)hi), "r"((u32)(hi >> 32)));
}
// acc = acc * 2^K + v  (K = 1 or 2: one Horner step of a binary / base-4 recomposition)
template <int K>
GL_D void acc_horner(acc160& c, u64 v) {
    const u32 n4 = __funnelshift_l(c.w3, c.w4, K), n3 = __funnelshift_l(c.w2, c.w3, K), n2 = __funnelshift_l(c.w1, c.w2, K),
              n1 = __funnelshift_l(c.w0, c.w1, K), n0 = c.w0 << K;
    asm("add.cc.u32 %0, %5, %10;\n\taddc.cc.u32 %1, %6, %11;\n\taddc.cc.u32 %2, %7, 0;\n\taddc.cc.u32 %3, %8, 0;\n\taddc.u32 %4, %9, 0;"
        : "=r"(c.w0), "=r"(c.w1), "=r"(c.w2), "=r"(c.w3), "=r"(c.w4)
        : "r"(n0), "r"(n1), "r"(n2), "r"(n3), "r"(n4), "r"((u32)v), "r"((u32)(v >> 32)));
}
// w0 + w1 phi + w2 phi^2 + w3 phi^3 + w4 phi^4, phi = 2^32: phi^2 = phi - 1, phi^3 = -1, phi^4 = -phi
GL_D u64 acc_reduce(const acc160& c) {
    const u64 r = gl_reduce128(gl_pack(c.w0, c.w1), gl_pack(c.w2, c.w3));
    return gl_sub(r, (u64)c.w4 << 32);   // w4 * 2^32 < p
}

__global__ void __launch_bounds__(Q_BLOCK) k_quotient(const quotient_args a) {
    const u64 lde_size = (u64)1 << a.lg_lde;
    const u64 p = blockIdx.x * (u64)Q_BLOCK + threadIdx.x;
    if (p >= lde_size) return;
    const u64 i = a.lg_lde ? (__brevll(p) >> (64 - a.lg_lde)) : 0;      // natural index of this leaf
    const u64 i_next = (i + ((u64)1 << a.qdb)) & (lde_size - 1);
    const u64 p_next = a.lg_lde ? (__brevll(i_next) >> (64 - a.lg_lde)) : 0;
    const u64 x = gl_mul(7, gl_powtab(a.xtab, i));                       // shifted_x = coset_shift * w^i
    const unsigned nch = a.nch;
    const u64* __restrict__ W = a.wires + p;
    const u64* __restrict__ CS = a.cs + p;
    const u64* __restrict__ Z = a.zs + p;
    const u64* __restrict__ ZN = a.zs + p_next;
    acc160 res[QUOTIENT_MAX_CHALLENGES];
#pragma unroll
    for (int c = 0; c < QUOTIENT_MAX_CHALLENGES; c++) res[c] = acc_zero();
    const unsigned zi = (unsigned)(i & (((u64)1 << a.qdb) - 1));
    unsigned t = 0;
    // ---- vanishing_z_1_terms: L_0(x) (Z(x) - 1), L_0(x) = Z_H(x) / (n (x - 1))
    const u64 l0 = gl_mul(a.zh[zi], q_inv(gl_mul(a.n_field, gl_sub(x, 1))));
    for (unsigned c = 0; c < nch; c++, t++) {
        const u64 term = gl_mul(l0, gl_sub(Z[(u64)c * a.z_ld], 1));
        _Pragma("unroll") for (unsigned cc = 0; cc < QUOTIENT_MAX_CHALLENGES; cc++) if (cc < nch) acc_mad(res[cc], __ldg(a.apow + cc * a.nterms + t), term);
    }
    // ---- check_partial_products for every challenge
    for (unsigned c = 0; c < nch; c++) {
        const u64 beta = a.betas[c], gamma = a.gammas[c];
        const u64 bx = gl_mul(beta, x);
        const u64* pp = Z + (u64)(nch + c * a.num_prods) * a.z_ld;
        u64 prev = Z[(u64)c * a.z_ld];
        for (unsigned q = 0; q < a.chunks; q++, t++) {
            u64 num = 1, den = 1;
            const unsigned j1 = min((q + 1) * a.deg, a.R);
            for (unsigned j = q * a.deg; j < j1; j++) {
                const u64 wv = W[(u64)j * a.w_ld];
                const u64 sg = CS[(u64)(a.num_constants + j) * a.cs_ld];
                num = gl_mul(num, gl_mad2(bx, __ldg(a.k_is + j), wv, gamma));    // wire + beta * k_i * x + gamma
                den = gl_mul(den, gl_mad2(beta, sg, wv, gamma));                 // wire + beta * sigma + gamma
            }
            const u64 next = q == a.chunks - 1 ? ZN[(u64)c * a.z_ld] : pp[(u64)q * a.z_ld];
            const u64 term = gl_sub(gl_mul(prev, num), gl_mul(next, den));
            prev = next;
            _Pragma("unroll") for (unsigned cc = 0; cc < QUOTIENT_MAX_CHALLENGES; cc++) if (cc < nch) acc_mad(res[cc], __ldg(a.apow + cc * a.nterms + t), term);
        }
    }
    // ---- evaluate_gate_constraints_base_batch
    const bool many = a.num_selectors > 1;
    for (unsigned gi = 0; gi < a.num_gates; gi++) {
        const gl_gate g = a.gates[gi];
        if (g.kind == GL_GATE_NOOP) continue;
        const u64 s = CS[(u64)g.selector_index * a.cs_ld];
        u64 filter = 1;
        for (unsigned k = g.group_start; k < g.group_end; k++)
            if (k != gi) filter = gl_mul(filter, gl_sub((u64)k, s));
        if (many) filter = gl_mul(filter, gl_sub(Q_UNUSED_SELECTOR, s));
        acc160 acc[QUOTIENT_MAX_CHALLENGES];
#pragma unroll
        for (int c = 0; c < QUOTIENT_MAX_CHALLENGES; c++) acc[c] = acc_zero();
        const u64* ap = a.apow + a.gate_term0;
        unsigned k = 0;
#define Q_YIELD(v)                                                                                         \
    {                                                                                                      \
        const u64 v__ = (v);                                                                               \
        _Pragma("unroll") for (unsigned cc = 0; cc < QUOTIENT_MAX_CHALLENGES; cc++) if (cc < nch) acc_mad(acc[cc], __ldg(ap + cc * a.nterms + k), v__); \
        k++;                                                                                               \
    }
        if (g.kind == GL_GATE_CONSTANT) {
            for (unsigned o = 0; o < g.num_ops; o++) Q_YIELD(gl_sub(CS[(u64)(a.num_selectors + o) * a.cs_ld], W[(u64)o * a.w_ld]))
        } else if (g.kind == GL_GATE_PUBLIC_INPUT) {
            for (unsigned o = 0; o < 4; o++) Q_YIELD(gl_sub(W[(u64)o * a.w_ld], a.pih[o]))
        } else if (g.kind == GL_GATE_U32_INTERLEAVE) {
            for (unsigned o = 0; o < g.num_ops; o++) {
                const u64* bits = W + (u64)(g.num_ops * 2 + 32 * o) * a.w_ld;    // big-endian decomposition
                acc160 cx = acc_zero(), cxi = acc_zero();
                for (unsigned b = 0; b < 32; b++) {                             // Horner from the most significant bit
                    const u64 bit = bits[(u64)b * a.w_ld];
                    acc_horner<1>(cx, bit);                                     // sum bit * 2^(31 - b)  < 2^96
                    acc_horner<2>(cxi, bit);                                    // sum bit * 4^(31 - b)  < 2^128
                }
                Q_YIELD(gl_sub(acc_reduce(cx), W[(u64)(2 * o) * a.w_ld]))        // Check 1: decomposition matches x
                Q_YIELD(gl_sub(acc_reduce(cxi), W[(u64)(2 * o + 1) * a.w_ld]))   // Check 2: base-4 sum matches x_interleaved
                for (unsigned b = 0; b < 32; b++) {                             // Check 3: bit (bit - 1)
                    const u64 bit = bits[(u64)b * a.w_ld];
                    Q_YIELD(gl_mul(bit, gl_sub(bit, 1)))
                }
            }
        } else {   // GL_GATE_UNINTERLEAVE_TO_U32 / _TO_B32
            const bool b32 = g.kind == GL_GATE_UNINTERLEAVE_TO_B32;
            for (unsigned o = 0; o < g.num_ops; o++) {
                const u64* bits = W + (u64)(g.num_ops * 3 + 64 * o) * a.w_ld;
                acc160 cxi = acc_zero(), ev = acc_zero(), od = acc_zero();
                for (unsigned j = 0; j < 32; j++) {
                    const u64 e = bits[(u64)(2 * j) * a.w_ld], d = bits[(u64)(2 * j + 1) * a.w_ld];
                    acc_horner<1>(cxi, e);                                     // sum (2 e + d) * 4^(31 - j)  < 2^130
                    acc_horner<1>(cxi, d);
                    if (b32) {                                                 // coeff 4^(31 - j) ...
                        acc_horner<2>(ev, e);
                        acc_horner<2>(od, d);
                    } else {                                                   // ... or 2^(31 - j)
                        acc_horner<1>(ev, e);
                        acc_horner<1>(od, d);
                    }
                }
                Q_YIELD(gl_sub(acc_reduce(cxi), W[(u64)(3 * o) * a.w_ld]))
                Q_YIELD(gl_sub(acc_reduce(ev), W[(u64)(3 * o + 1) * a.w_ld]))
                Q_YIELD(gl_sub(acc_reduce(od), W[(u64)(3 * o + 2) * a.w_ld]))
                for (unsigned b = 0; b < 64; b++) {
                    const u64 bit = bits[(u64)b * a.w_ld];
                    Q_YIELD(gl_mul(bit, gl_sub(bit, 1)))
                }
            }
        }
#undef Q_YIELD
        _Pragma("unroll") for (unsigned cc = 0; cc < QUOTIENT_MAX_CHALLENGES; cc++) if (cc < nch) acc_mad(res[cc], filter, acc_reduce(acc[cc]));
    }
    // ---- divide by Z_H on the coset, scatter to the natural index
    const u64 zinv = a.zh_inv[zi];
#pragma unroll
    for (unsigned c = 0; c < QUOTIENT_MAX_CHALLENGES; c++)
        if (c < nch) a.out[(u64)c * lde_size + i] = gl_canon(gl_mul(acc_reduce(res[c]), zinv));
}

void launch_quotient(const quotient_args& a, cudaStream_t st) {
    const u64 lde_size = (u64)1 << a.lg_lde;
    k_quotient<<<(unsigned)((lde_size + Q_BLOCK - 1) / Q_BLOCK), Q_BLOCK, 0, st>>>(a);
    ++g_gl_launches;
}
