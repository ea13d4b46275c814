// Internal interface of permutation_kernels.cu: the permutation argument's Z and partial-product columns
// (plonky2::plonk::prover all_wires_permutation_partial_products, SURVEY 3.2 step 5).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <atomic>

extern std::atomic<unsigned long long> g_gl_launches;

#define PERM_BLOCK 128            // rows per CTA of the row and apply kernels (one row per thread)
#define PERM_MAX_CHALLENGES 4
#define PERM_MAX_SLOTS 64         // num_challenges * chunks: 2 * slots * PERM_BLOCK * 8 bytes of shared memory per CTA

struct perm_args {
    const uint64_t *wires, *sigmas;   // [R][n] routed wire values and sigma values on the subgroup, natural order
    const uint64_t* k_is;             // [R], canonical
    const uint64_t* xtab;             // 3 x 1024 power table of w_n
    uint64_t* out;                    // [nch * chunks][n]: Z_0 .. Z_{nch-1}, then the partial products of challenge 0, 1, ..
    uint64_t* cta;                    // [nch][nblocks]: product of the row ratios of each CTA, then its exclusive prefix
    uint64_t* grand;                  // [nch]: product of all row ratios
    unsigned* zero_den;               // set when some wire + beta * sigma + gamma is zero
    uint64_t n;
    uint32_t R, deg, chunks, nch, nblocks;
    uint64_t betas[PERM_MAX_CHALLENGES], gammas[PERM_MAX_CHALLENGES];
};
// three launches on `st`: row ratios + CTA products, scan of the CTA products, apply
cudaError_t launch_permutation_zs(const perm_args& a, cudaStream_t st);
