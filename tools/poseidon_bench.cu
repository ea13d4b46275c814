// Throughput of the Poseidon permutation alone (state in registers, no memory traffic) + KAT check.
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -I plonky2-lib_b200/csrc -o tools/poseidon_bench tools/poseidon_bench.cu
#include <cuda_runtime.h>

#include <cstdio>

#include "poseidon.cuh"
#include "poseidon_constants.h"

#ifndef REPS
#define REPS 64
#endif
#ifndef BLOCK
#define BLOCK 256
#endif
#ifndef MINB
#define MINB 1
#endif

#ifdef TWO_STATES
// experiment: two independent states per thread, their rounds in the same basic block (does ptxas overlap the FP64 layers
// of one with the integer S-boxes of the other?)
__device__ __forceinline__ void poseidon_permute2(u64 s[12], u64 t[12]) {
#pragma unroll
    for (int i = 0; i < 12; i++) { s[i] = gl_add_c(s[i], c_poseidon_rc[i]); t[i] = gl_add_c(t[i], c_poseidon_rc[i]); }
#pragma unroll 1
    for (int phase = 0; phase < 2; phase++) {
        const double2* rc = c_poseidon_rc_split + 12 * (phase ? POSEIDON_FULL_HALF + POSEIDON_PARTIAL + 1 : 1);
#pragma unroll 1
        for (int r = 0; r < POSEIDON_FULL_HALF; r++, rc += 12) { poseidon_full_round(s, rc); poseidon_full_round(t, rc); }
        if (phase == 0) {
            double sl[12], sh[12], tl[12], th[12];
#pragma unroll
            for (int i = 1; i < 12; i++) {
                sl[i] = u32_as_denormal((u32)s[i]); sh[i] = u32_as_denormal((u32)(s[i] >> 32));
                tl[i] = u32_as_denormal((u32)t[i]); th[i] = u32_as_denormal((u32)(t[i] >> 32));
            }
#pragma unroll 1
            for (int pair = 0; pair < POSEIDON_PARTIAL / 2; pair++) {
                poseidon_partial_pair(s[0], sl, sh, pair);
                poseidon_partial_pair(t[0], tl, th, pair);
            }
#pragma unroll
            for (int i = 1; i < 12; i++) { s[i] = poseidon_fold(sl[i], sh[i]); t[i] = poseidon_fold(tl[i], th[i]); }
        }
    }
}
__global__ void __launch_bounds__(BLOCK, MINB) k_bench(u64* out, u64 seed) {
    u64 s[12], t[12];
#pragma unroll
    for (int i = 0; i < 12; i++) { s[i] = seed * (threadIdx.x + 1 + blockIdx.x * (u64)blockDim.x) + i; t[i] = s[i] ^ 0x5555; }
#pragma unroll 1
    for (int r = 0; r < REPS / 2; r++) poseidon_permute2(s, t);
    u64 acc = 0;
#pragma unroll
    for (int i = 0; i < 12; i++) acc ^= s[i] ^ t[i];
    out[blockIdx.x * (u64)blockDim.x + threadIdx.x] = acc;
}
#else
__global__ void __launch_bounds__(BLOCK, MINB) k_bench(u64* out, u64 seed) {
    u64 s[12];
#pragma unroll
    for (int i = 0; i < 12; i++) s[i] = seed * (threadIdx.x + 1 + blockIdx.x * (u64)blockDim.x) + i;
#pragma unroll 1
    for (int r = 0; r < REPS; r++) poseidon_permute(s);
    u64 acc = 0;
#pragma unroll
    for (int i = 0; i < 12; i++) acc ^= s[i];
    out[blockIdx.x * (u64)blockDim.x + threadIdx.x] = acc;
}

#endif

__global__ void k_kat(u64* io) {
    u64 s[12];
    for (int i = 0; i < 12; i++) s[i] = io[i];
    poseidon_permute(s);
    for (int i = 0; i < 12; i++) io[i] = gl_canon(s[i]);
}

// exactness of the FP64 linear layers at the extremes: every 32-bit half at 0xffffffff / 0 / random, compared with
// 128-bit integer arithmetic on the device
__global__ void k_circ_extremes(const u64* halves, int cases, int* bad) {
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= cases) return;
    const u64* h = halves + 12 * t;
    double x[12], y1[12], y2[12];
    for (int i = 0; i < 12; i++) x[i] = u32_as_denormal((u32)h[i]);
    poseidon_circ12<0>(x, y1);
    poseidon_circ12<1>(x, y2);
    const int C[12] = {17, 15, 41, 16, 2, 28, 13, 13, 39, 18, 34, 20};
    u64 c1[12], c2[12];
    for (int r = 0; r < 12; r++) {
        u64 acc = 0;
        for (int i = 0; i < 12; i++) acc += (u64)C[i] * h[(i + r) % 12];
        c1[r] = acc;
    }
    for (int r = 0; r < 12; r++) {
        u64 acc = 0;
        for (int i = 0; i < 12; i++) acc += (u64)C[i] * c1[(i + r) % 12];
        c2[r] = acc;
    }
    for (int r = 0; r < 12; r++)
        if (double_bits(y1[r]) != c1[r] || double_bits(y2[r]) != c2[r]) atomicAdd(bad, 1);
}

// The same check for the inputs the S-box hand-off gives the layers: lanes in [0, 3 * 2^32) (dl = r0 - r2 - r3 + 2^33) for one
// layer (SQ = 0); lane 0 in that range and lanes 1..11 in [0, 2^33) for the fused pair (SQ = 1, the range of poseidon_renorm's
// (L, H)), with the rank-one term e e0 (e = 8 x_0 - M[0] . x + sigma, signed) applied in the frequency domain.
// ab[t][i] = (a, b): lane 0 (and every lane of SQ = 0) is a + 2 b, formed as an integer bit pattern the way
// poseidon_sbox_split forms it; lanes 1..11 of SQ = 1 are a + 2^32 (b >> 31).
__global__ void k_circ_handoff(const u32* ab, int cases, int* bad) {
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= cases) return;
    const u32* h = ab + 24 * t;
    const int C[12] = {17, 15, 41, 16, 2, 28, 13, 13, 39, 18, 34, 20};
    for (int sq = 0; sq < 2; sq++) {
        double x[12], y[12];
        u64 xi[12], c1[12], c2[12];
        for (int i = 0; i < 12; i++) {
            xi[i] = (sq == 0 || i == 0) ? (u64)h[2 * i] + 2 * (u64)h[2 * i + 1] : (u64)h[2 * i] + ((u64)(h[2 * i + 1] >> 31) << 32);
            x[i] = __longlong_as_double((long long)xi[i]);
        }
        long long e = 8 * (long long)xi[0] + (long long)(xi[1] ^ xi[5]);   // + sigma, any value in the lanes' range
        for (int j = 0; j < 12; j++) e -= (long long)(C[j] + (j == 0 ? 8 : 0)) * (long long)xi[j];
        if (sq == 0) poseidon_circ12<0>(x, y);
        else poseidon_circ12<1, true>(x, y, e < 0 ? -__longlong_as_double(-e) : __longlong_as_double(e));
        for (int r = 0; r < 12; r++) {
            u64 acc = 0;
            for (int i = 0; i < 12; i++) acc += (u64)C[i] * xi[(i + r) % 12];
            c1[r] = acc;
        }
        for (int r = 0; r < 12; r++) {
            u64 acc = 0;
            for (int i = 0; i < 12; i++) acc += (u64)C[i] * c1[(i + r) % 12];
            c2[r] = acc;
        }
        for (int r = 0; r < 12; r++) {
            // without the pair's table offsets z can be negative: compare signed integers
            const long long got = y[r] < 0 ? -(long long)double_bits(-y[r]) : (long long)double_bits(y[r]);
            if (got != (sq ? (long long)c2[r] + C[(12 - r) % 12] * e : (long long)c1[r])) atomicAdd(bad, 1);
        }
    }
}

// The integer forms at their extremes against 128-bit arithmetic: the S-box hand-off (dl - 2^33 + 2^32 dh = x^7 mod p) and
// the fold (A + 2^32 B mod p for A in [2^18, 2^50), B in [0, 2^50), the range the tables guarantee).  w[t] = (x, A, B).
__global__ void k_forms(const u64* w, int cases, int* bad) {
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= cases) return;
    typedef unsigned __int128 u128;
    const u64 x = w[3 * t], A = w[3 * t + 1], B = w[3 * t + 2];
    double dl, dh;
    poseidon_sbox_split(x, dl, dh);
    u64 x7 = 1;
    for (int i = 0; i < 7; i++) x7 = (u64)((u128)x7 * (x % GL_P) % GL_P);
    const u64 l = double_bits(dl), h = double_bits(dh);
    if (l < 2 || l >= (3ULL << 32) || h >= (1ULL << 33)) atomicAdd(bad, 1);
    if ((u64)(((u128)l + ((u128)h << 32) + (u128)GL_P * 4 - POSEIDON_HANDOFF_BIAS) % GL_P) != x7) atomicAdd(bad, 1);
    const u64 y = poseidon_fold(__longlong_as_double((long long)A), __longlong_as_double((long long)B));
    if (y % GL_P != (u64)(((u128)A + ((u128)B << 32)) % GL_P)) atomicAdd(bad, 1);
}

// poseidon_renorm at its extremes against 128-bit arithmetic: A in [2^32, 2^50), B in [0, 2^50) give L in [2^32 - 2^18, 2^33),
// H < 2^32 + 2^19 with L + 2^32 H = A + 2^32 B (mod p), and the fold after the last pair takes (L, H).  w[t] = (A, B).
__global__ void k_renorm(const u64* w, int cases, int* bad) {
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= cases) return;
    typedef unsigned __int128 u128;
    const u64 A = w[2 * t], B = w[2 * t + 1];
    double dl, dh;
    poseidon_renorm(__longlong_as_double((long long)A), __longlong_as_double((long long)B), dl, dh);
    const u64 l = double_bits(dl), h = double_bits(dh), want = (u64)(((u128)A + ((u128)B << 32)) % GL_P);
    if (l < (1ULL << 32) - (1ULL << 18) || l >= (1ULL << 33) || h >= (1ULL << 32) + (1ULL << 19)) atomicAdd(bad, 1);
    if ((u64)(((u128)l + ((u128)h << 32)) % GL_P) != want) atomicAdd(bad, 1);
    if (poseidon_fold(dl, dh) % GL_P != want) atomicAdd(bad, 1);
}

int main() {
    u64 rc[360];
    if (!poseidon_constants::generate(rc)) { printf("constants fingerprint mismatch\n"); return 1; }
    cudaMemcpyToSymbol(c_poseidon_rc, rc, sizeof rc);
    static u64 split[31 * 12 * 2], pk[11 * 12 * 2];
    static const int circ[12] = {17, 15, 41, 16, 2, 28, 13, 13, 39, 18, 34, 20};
    poseidon_constants::linear_layer_tables(rc, circ, 8, true, split, pk, POSEIDON_HANDOFF_BIAS);
    cudaMemcpyToSymbol(c_poseidon_rc_split, split, sizeof split);
    cudaMemcpyToSymbol(c_poseidon_pair_k, pk, sizeof pk);
    u64 h[12], *d;
    cudaMalloc(&d, 96);
    const u64 want_iota[4] = {0xd64e1e3efc5b8e9eULL, 0x53666633020aaa47ULL, 0xd40285597c6a8825ULL, 0x613a4f81e81231d2ULL};
    const u64 want_max[4] = {0xbe0085cfc57a8357ULL, 0xd95af71847d05c09ULL, 0xcf55a13d33c1c953ULL, 0x95803a74f4530e82ULL};
    int ok = 1;
    for (int i = 0; i < 12; i++) h[i] = i;
    cudaMemcpy(d, h, 96, cudaMemcpyHostToDevice);
    k_kat<<<1, 1>>>(d);
    cudaMemcpy(h, d, 96, cudaMemcpyDeviceToHost);
    for (int i = 0; i < 4; i++) ok &= h[i] == want_iota[i];
    for (int i = 0; i < 12; i++) h[i] = 0xFFFFFFFF00000000ULL;
    cudaMemcpy(d, h, 96, cudaMemcpyHostToDevice);
    k_kat<<<1, 1>>>(d);
    cudaMemcpy(h, d, 96, cudaMemcpyDeviceToHost);
    for (int i = 0; i < 4; i++) ok &= h[i] == want_max[i];
    {
        const int cases = 1 << 16;
        u64* hh = (u64*)malloc((size_t)cases * 12 * 8);
        u64 st = 88172645463325252ULL;
        for (int t = 0; t < cases; t++)
            for (int i = 0; i < 12; i++) {
                st ^= st << 13; st ^= st >> 7; st ^= st << 17;
                u64 v = st & 0xFFFFFFFFULL;
                int mode = t & 7;   // 0: all max, 1: all zero, 2: alternating, 3: one hot max, 4..7: random with extremes
                if (mode == 0) v = 0xFFFFFFFFULL;
                else if (mode == 1) v = 0;
                else if (mode == 2) v = ((i + (t >> 3)) & 1) ? 0xFFFFFFFFULL : 0;
                else if (mode == 3) v = (i == (t >> 3) % 12) ? 0xFFFFFFFFULL : 0;
                else if (mode == 4 && (st >> 40) % 3 == 0) v = 0xFFFFFFFFULL;
                hh[(size_t)t * 12 + i] = v;
            }
        u64* dh;
        int *dbad, hbad = 0;
        cudaMalloc(&dh, (size_t)cases * 96);
        cudaMalloc(&dbad, 4);
        cudaMemcpy(dh, hh, (size_t)cases * 96, cudaMemcpyHostToDevice);
        cudaMemset(dbad, 0, 4);
        k_circ_extremes<<<cases / 128, 128>>>(dh, cases, dbad);
        cudaMemcpy(&hbad, dbad, 4, cudaMemcpyDeviceToHost);
        printf("{\"circ12_extreme_cases\": %d, \"mismatches\": %d}\n", cases, hbad);
        ok &= hbad == 0;
        free(hh);
    }
    {
        const int cases = 1 << 16;
        u32* hh = (u32*)malloc((size_t)cases * 24 * 4);
        u64 st = 0x9E3779B97F4A7C15ULL;
        for (int t = 0; t < cases; t++)
            for (int i = 0; i < 24; i++) {
                st ^= st << 13; st ^= st >> 7; st ^= st << 17;
                u32 v = (u32)st;
                const int mode = t & 7;   // all limbs max, all zero, alternating lanes, one-hot lane, random with extremes
                if (mode == 0) v = 0xFFFFFFFFu;
                else if (mode == 1) v = 0;
                else if (mode == 2) v = (((i >> 1) + (t >> 3)) & 1) ? 0xFFFFFFFFu : 0u;
                else if (mode == 3) v = ((i >> 1) == (t >> 3) % 12) ? 0xFFFFFFFFu : 0u;
                else if (mode == 4 && (st >> 40) % 3 == 0) v = 0xFFFFFFFFu;
                hh[(size_t)t * 24 + i] = v;
            }
        u32* dh;
        int *dbad, hbad = 0;
        cudaMalloc(&dh, (size_t)cases * 96);
        cudaMalloc(&dbad, 4);
        cudaMemcpy(dh, hh, (size_t)cases * 96, cudaMemcpyHostToDevice);
        cudaMemset(dbad, 0, 4);
        k_circ_handoff<<<cases / 128, 128>>>(dh, cases, dbad);
        cudaMemcpy(&hbad, dbad, 4, cudaMemcpyDeviceToHost);
        printf("{\"circ12_handoff_cases\": %d, \"mismatches\": %d}\n", cases, hbad);
        ok &= hbad == 0;
        free(hh);
    }
    {
        const int cases = 1 << 16;
        u64* hw = (u64*)malloc((size_t)cases * 24);
        u64 st = 0x2545F4914F6CDD1DULL;
        const u64 X[6] = {0, 1, GL_P - 1, 0xFFFFFFFFFFFFFFFFULL, 0xFFFFFFFF00000000ULL, 0xFFFFFFFFULL};
        const u64 AMIN = 1ULL << 18, AMAX = (1ULL << 50) - 1, BMAX = (1ULL << 50) - 1;
        for (int t = 0; t < cases; t++) {
            u64 r[3];
            for (int k = 0; k < 3; k++) { st ^= st << 13; st ^= st >> 7; st ^= st << 17; r[k] = st; }
            const int mode = t & 7;   // extremes of x, A, B (b0 = 0xffffffff, bh max, A at both ends), then random
            u64 x = r[0], A = AMIN + r[1] % (AMAX - AMIN + 1), B = r[2] & BMAX;
            if (mode < 6) x = X[mode];
            if (mode == 0) { A = AMAX; B = BMAX; }
            else if (mode == 1) { A = AMIN; B = BMAX; }
            else if (mode == 2) { A = AMIN; B = 0; }
            else if (mode == 3) { A = AMAX; B = 0xFFFFFFFFULL; }
            else if (mode == 4) { A = AMIN; B = BMAX & ~0xFFFFFFFFULL; }
            else if (mode == 5) B |= 0xFFFFFFFFULL;
            hw[3 * t] = x; hw[3 * t + 1] = A; hw[3 * t + 2] = B;
        }
        u64* dw;
        int *dbad, hbad = 0;
        cudaMalloc(&dw, (size_t)cases * 24);
        cudaMalloc(&dbad, 4);
        cudaMemcpy(dw, hw, (size_t)cases * 24, cudaMemcpyHostToDevice);
        cudaMemset(dbad, 0, 4);
        k_forms<<<cases / 128, 128>>>(dw, cases, dbad);
        cudaMemcpy(&hbad, dbad, 4, cudaMemcpyDeviceToHost);
        printf("{\"handoff_fold_cases\": %d, \"mismatches\": %d}\n", cases, hbad);
        ok &= hbad == 0;
        free(hw);
    }
    {
        const int cases = 1 << 16;
        u64* hw = (u64*)malloc((size_t)cases * 16);
        u64 st = 0x6A09E667F3BCC909ULL;
        const u64 AMIN = 1ULL << 32, AMAX = (1ULL << 50) - 1, BMAX = (1ULL << 50) - 1;
        for (int t = 0; t < cases; t++) {
            u64 r[2];
            for (int k = 0; k < 2; k++) { st ^= st << 13; st ^= st >> 7; st ^= st << 17; r[k] = st; }
            const int mode = t & 7;   // b1 at its maximum, a0 = 0, b0 = 0xffffffff, a1 = 1, A and B at their ends, then random
            u64 A = AMIN + r[0] % (AMAX - AMIN + 1), B = r[1] & BMAX;
            if (mode == 0) { A &= ~0xFFFFFFFFULL; B = BMAX; }
            else if (mode == 1) { A = AMIN; B = BMAX; }
            else if (mode == 2) { A = AMAX; B = 0; }
            else if (mode == 3) { A = AMIN; B = 0xFFFFFFFFULL; }
            else if (mode == 4) { A &= ~0xFFFFFFFFULL; B |= 0xFFFFFFFFULL; }
            else if (mode == 5) B |= 0xFFFFFFFFULL;
            hw[2 * t] = A; hw[2 * t + 1] = B;
        }
        u64* dw;
        int *dbad, hbad = 0;
        cudaMalloc(&dw, (size_t)cases * 16);
        cudaMalloc(&dbad, 4);
        cudaMemcpy(dw, hw, (size_t)cases * 16, cudaMemcpyHostToDevice);
        cudaMemset(dbad, 0, 4);
        k_renorm<<<cases / 128, 128>>>(dw, cases, dbad);
        cudaMemcpy(&hbad, dbad, 4, cudaMemcpyDeviceToHost);
        printf("{\"renorm_cases\": %d, \"mismatches\": %d}\n", cases, hbad);
        ok &= hbad == 0;
        free(hw);
    }
    cudaDeviceProp p;
    cudaGetDeviceProperties(&p, 0);
    int blocks = p.multiProcessorCount * 16;
    u64* out;
    cudaMalloc(&out, (size_t)blocks * BLOCK * 8);
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0);
    cudaEventCreate(&e1);
    k_bench<<<blocks, BLOCK>>>(out, 3);
    cudaDeviceSynchronize();
    float best = 1e30f;
    for (int r = 0; r < 3; r++) {
        cudaEventRecord(e0);
        k_bench<<<blocks, BLOCK>>>(out, 5 + r);
        cudaEventRecord(e1);
        cudaEventSynchronize(e1);
        float ms;
        cudaEventElapsedTime(&ms, e0, e1);
        if (ms < best) best = ms;
    }
    cudaError_t e = cudaGetLastError();
    double perms = (double)blocks * BLOCK * REPS;
    printf("{\"kat_ok\": %d, \"perms_per_s\": %.4e, \"ms\": %.3f, \"block\": %d, \"minb\": %d, \"err\": \"%s\"}\n", ok, perms / (best * 1e-3), best,
           BLOCK, MINB, cudaGetErrorString(e));
    return ok ? 0 : 2;
}
