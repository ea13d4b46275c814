// The permutation argument's Z and partial-product columns on the device: plonky2::plonk::prover
// all_wires_permutation_partial_products / wires_permutation_partial_products_and_zs (SURVEY 3.2 step 5), reached from
// every data.prove(pw).  For row i (x = w^i), challenge c and chunk q of quotient_degree_factor routed wires:
//   N_q = prod_j (w_j + beta * k_j * x + gamma),  D_q = prod_j (w_j + beta * sigma_j + gamma),
//   rho_q(i) = prod_{q' <= q} N_q' / D_q',  r(i) = rho_{chunks-1}(i),
//   Z(i) = prod_{i' < i} r(i'),  partial product q at row i = Z(i) * rho_q(i)   (q < chunks - 1).
// Three launches:
//   k_perm_rows   one row per thread: the 2R values of the row are read once for every challenge; rho_q by Montgomery's
//                 trick over the chunks (prefix products, ONE Fermat inverse per row and challenge, then a backward walk);
//                 rho_q -> partial-product slots, r -> Z slot, and the product of r over the CTA's rows.
//   k_perm_scan   one CTA: exclusive prefix of the CTA products (each thread multiplies a contiguous run of them serially,
//                 so one CTA covers any row count) and the grand product.
//   k_perm_apply  Z(i) = (CTA prefix) * (exclusive in-CTA prefix of r, warp shuffles), partial products *= Z(i).
// Goldilocks multiplication is associative, commutative and exact, so this scan tree gives bit-for-bit the values of the
// prover's serial running product; every value written at the end is canonical.
#include <cuda_runtime.h>

#include "gl_field.cuh"
#include "permutation_kernels.h"

#define PERM_FULL_MASK 0xFFFFFFFFu
#define PERM_SCAN_THREADS 1024

// inclusive product scan over the lanes of a warp
GL_D u64 perm_warp_scan(u64 v, unsigned lane) {
#pragma unroll
    for (unsigned d = 1; d < 32; d <<= 1) {
        const u64 o = __shfl_up_sync(PERM_FULL_MASK, v, d);
        if (lane >= d) v = gl_mul(o, v);
    }
    return v;
}

__global__ void __launch_bounds__(PERM_BLOCK) k_perm_rows(const perm_args a) {
    extern __shared__ u64 perm_sm[];   // [2][nch * chunks][PERM_BLOCK]: D_q, then the prefix products of N
    __shared__ u64 wprod[PERM_MAX_CHALLENGES][PERM_BLOCK / 32];
    const unsigned t = threadIdx.x, lane = t & 31, wid = t >> 5;
    const u64 i = blockIdx.x * (u64)PERM_BLOCK + t;
    const unsigned nch = a.nch, chunks = a.chunks, slots = nch * chunks;
    u64* sD = perm_sm + t;
    u64* sN = perm_sm + (u64)slots * PERM_BLOCK + t;
    u64 r[PERM_MAX_CHALLENGES];
#pragma unroll
    for (unsigned c = 0; c < PERM_MAX_CHALLENGES; c++) r[c] = 1;
    if (i < a.n) {
        const u64 x = gl_powtab(a.xtab, i);
        u64 bx[PERM_MAX_CHALLENGES], pn[PERM_MAX_CHALLENGES], pd[PERM_MAX_CHALLENGES];
#pragma unroll
        for (unsigned c = 0; c < PERM_MAX_CHALLENGES; c++) {
            bx[c] = c < nch ? gl_mul(a.betas[c], x) : 0;
            pn[c] = pd[c] = 1;
        }
        const u64* __restrict__ W = a.wires + i;
        const u64* __restrict__ S = a.sigmas + i;
        for (unsigned q = 0; q < chunks; q++) {
            u64 num[PERM_MAX_CHALLENGES], den[PERM_MAX_CHALLENGES];
#pragma unroll
            for (unsigned c = 0; c < PERM_MAX_CHALLENGES; c++) num[c] = den[c] = 1;
            const unsigned j1 = min((q + 1) * a.deg, a.R);
            for (unsigned j = q * a.deg; j < j1; j++) {
                const u64 wv = W[(u64)j * a.n], sg = S[(u64)j * a.n], k = __ldg(a.k_is + j);
#pragma unroll
                for (unsigned c = 0; c < PERM_MAX_CHALLENGES; c++)
                    if (c < nch) {
                        num[c] = gl_mul(num[c], gl_mad2(bx[c], k, wv, a.gammas[c]));       // wire + beta * k_j * x + gamma
                        den[c] = gl_mul(den[c], gl_mad2(a.betas[c], sg, wv, a.gammas[c]));  // wire + beta * sigma + gamma
                    }
            }
#pragma unroll
            for (unsigned c = 0; c < PERM_MAX_CHALLENGES; c++)
                if (c < nch) {
                    pn[c] = gl_mul(pn[c], num[c]);
                    pd[c] = gl_mul(pd[c], den[c]);
                    sD[(u64)(c * chunks + q) * PERM_BLOCK] = den[c];
                    sN[(u64)(c * chunks + q) * PERM_BLOCK] = pn[c];
                }
        }
        const unsigned np = chunks - 1;
#pragma unroll
        for (unsigned c = 0; c < PERM_MAX_CHALLENGES; c++)
            if (c < nch) {
                // upstream's batch_multiplicative_inverse panics on a zero denominator: flag it, the host fails the call
                if (gl_canon(pd[c]) == 0) atomicOr(a.zero_den, 1u);
                u64 inv = gl_pow(pd[c], GL_P - 2);                                    // 1 / (D_0 .. D_{chunks-1})
                for (unsigned q = chunks; q-- > 0;) {
                    const u64 rho = gl_mul(sN[(u64)(c * chunks + q) * PERM_BLOCK], inv);
                    if (q == np) r[c] = rho;
                    else a.out[(u64)(nch + c * np + q) * a.n + i] = rho;
                    inv = gl_mul(inv, sD[(u64)(c * chunks + q) * PERM_BLOCK]);         // 1 / (D_0 .. D_{q-1})
                }
                a.out[(u64)c * a.n + i] = r[c];
            }
    }
    // product of r over the CTA's rows (rows past n contribute 1)
#pragma unroll
    for (unsigned c = 0; c < PERM_MAX_CHALLENGES; c++)
        if (c < nch) {
            u64 v = r[c];
#pragma unroll
            for (unsigned d = 16; d; d >>= 1) v = gl_mul(v, __shfl_xor_sync(PERM_FULL_MASK, v, d));
            if (lane == 0) wprod[c][wid] = v;
        }
    __syncthreads();
    if (t < nch) {
        u64 v = wprod[t][0];
#pragma unroll
        for (unsigned w = 1; w < PERM_BLOCK / 32; w++) v = gl_mul(v, wprod[t][w]);
        a.cta[(u64)t * a.nblocks + blockIdx.x] = v;
    }
}

__global__ void __launch_bounds__(PERM_SCAN_THREADS) k_perm_scan(const perm_args a) {
    __shared__ u64 wtot[PERM_SCAN_THREADS / 32];
    const unsigned t = threadIdx.x, lane = t & 31, wid = t >> 5;
    const unsigned per = (a.nblocks + PERM_SCAN_THREADS - 1) / PERM_SCAN_THREADS;
    const unsigned b0 = min(t * per, a.nblocks), b1 = min(b0 + per, a.nblocks);
    for (unsigned c = 0; c < a.nch; c++) {
        u64* v = a.cta + (u64)c * a.nblocks;
        u64 s = 1;
        for (unsigned b = b0; b < b1; b++) s = gl_mul(s, v[b]);
        const u64 inc = perm_warp_scan(s, lane);
        if (lane == 31) wtot[wid] = inc;
        __syncthreads();
        if (wid == 0) wtot[lane] = perm_warp_scan(wtot[lane], lane);
        __syncthreads();
        u64 excl = __shfl_up_sync(PERM_FULL_MASK, inc, 1);
        if (lane == 0) excl = 1;
        if (wid) excl = gl_mul(wtot[wid - 1], excl);
        for (unsigned b = b0; b < b1; b++) {
            const u64 p = v[b];
            v[b] = excl;
            excl = gl_mul(excl, p);
        }
        if (t == 0) a.grand[c] = gl_canon(wtot[PERM_SCAN_THREADS / 32 - 1]);
        __syncthreads();
    }
}

__global__ void __launch_bounds__(PERM_BLOCK) k_perm_apply(const perm_args a) {
    __shared__ u64 wtot[PERM_MAX_CHALLENGES][PERM_BLOCK / 32];
    const unsigned t = threadIdx.x, lane = t & 31, wid = t >> 5;
    const u64 i = blockIdx.x * (u64)PERM_BLOCK + t;
    const bool live = i < a.n;
    const unsigned nch = a.nch, np = a.chunks - 1;
    u64 excl[PERM_MAX_CHALLENGES];
#pragma unroll
    for (unsigned c = 0; c < PERM_MAX_CHALLENGES; c++) {
        excl[c] = 1;
        if (c < nch) {
            const u64 inc = perm_warp_scan(live ? a.out[(u64)c * a.n + i] : 1, lane);
            excl[c] = __shfl_up_sync(PERM_FULL_MASK, inc, 1);
            if (lane == 0) excl[c] = 1;
            if (lane == 31) wtot[c][wid] = inc;
        }
    }
    __syncthreads();
    if (!live) return;
#pragma unroll
    for (unsigned c = 0; c < PERM_MAX_CHALLENGES; c++)
        if (c < nch) {
            u64 z = a.cta[(u64)c * a.nblocks + blockIdx.x];
            for (unsigned w = 0; w < wid; w++) z = gl_mul(z, wtot[c][w]);
            z = gl_canon(gl_mul(z, excl[c]));
            a.out[(u64)c * a.n + i] = z;
            for (unsigned q = 0; q < np; q++) {
                u64* pp = a.out + (u64)(nch + c * np + q) * a.n + i;
                *pp = gl_canon(gl_mul(*pp, z));
            }
        }
}

cudaError_t launch_permutation_zs(const perm_args& a, cudaStream_t st) {
    const size_t smem = 2 * (size_t)a.nch * a.chunks * PERM_BLOCK * sizeof(u64);
    cudaError_t e = cudaFuncSetAttribute(k_perm_rows, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    k_perm_rows<<<a.nblocks, PERM_BLOCK, smem, st>>>(a);
    k_perm_scan<<<1, PERM_SCAN_THREADS, 0, st>>>(a);
    k_perm_apply<<<a.nblocks, PERM_BLOCK, 0, st>>>(a);
    g_gl_launches += 3;
    return cudaGetLastError();
}
