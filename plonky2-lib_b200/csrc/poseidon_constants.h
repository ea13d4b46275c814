// Poseidon-Goldilocks round constants, regenerated at context creation.
//
// plonky2's ALL_ROUND_CONSTANTS (plonky2::hash::poseidon) are the first 360 draws of
// ChaCha8Rng::seed_from_u64(0).gen_range(0..p) (rand 0.8.5 / rand_chacha 0.3.1, the versions the
// reference locks at Cargo.lock:1135-1149).  No table of them exists in /root/reference, so the
// library derives them and refuses to start unless the derived table reproduces the fingerprints
// that the reference's own known-answer test implies (src/zkdsa/circuits/mod.rs:85-105 passes only
// with exactly this table; XOR / first / last words recorded in SURVEY.md 8c).
#pragma once
#include <cstdint>
#include <cstring>

namespace poseidon_constants {

struct ChaCha8Stream {
    uint32_t key[8];
    uint64_t block_counter = 0;
    uint32_t buf[16];
    int used = 16;

    static uint32_t rol(uint32_t v, int k) { return (v << k) | (v >> (32 - k)); }
    static void quarter(uint32_t* x, int a, int b, int c, int d) {
        x[a] += x[b]; x[d] = rol(x[d] ^ x[a], 16);
        x[c] += x[d]; x[b] = rol(x[b] ^ x[c], 12);
        x[a] += x[b]; x[d] = rol(x[d] ^ x[a], 8);
        x[c] += x[d]; x[b] = rol(x[b] ^ x[c], 7);
    }
    // rand_core::SeedableRng::seed_from_u64: a PCG32 stream stretches the u64 into the 256-bit key
    explicit ChaCha8Stream(uint64_t seed) {
        uint64_t pcg = seed;
        for (int i = 0; i < 8; i++) {
            pcg = pcg * 6364136223846793005ULL + 11634580027462260723ULL;
            uint32_t xorshifted = (uint32_t)(((pcg >> 18) ^ pcg) >> 27);
            unsigned rot = (unsigned)(pcg >> 59) & 31u;
            key[i] = rot ? ((xorshifted >> rot) | (xorshifted << (32 - rot))) : xorshifted;
        }
    }
    void refill() {
        uint32_t init[16] = {0x61707865u, 0x3320646eu, 0x79622d32u, 0x6b206574u};  // "expand 32-byte k"
        for (int i = 0; i < 8; i++) init[4 + i] = key[i];
        init[12] = (uint32_t)block_counter;
        init[13] = (uint32_t)(block_counter >> 32);
        init[14] = init[15] = 0;
        uint32_t x[16];
        std::memcpy(x, init, sizeof x);
        for (int dr = 0; dr < 4; dr++) {  // 8 rounds
            quarter(x, 0, 4, 8, 12); quarter(x, 1, 5, 9, 13); quarter(x, 2, 6, 10, 14); quarter(x, 3, 7, 11, 15);
            quarter(x, 0, 5, 10, 15); quarter(x, 1, 6, 11, 12); quarter(x, 2, 7, 8, 13); quarter(x, 3, 4, 9, 14);
        }
        for (int i = 0; i < 16; i++) buf[i] = x[i] + init[i];
        block_counter++;
        used = 0;
    }
    uint32_t next_u32() {
        if (used == 16) refill();
        return buf[used++];
    }
    uint64_t next_u64() {
        uint64_t lo = next_u32();
        uint64_t hi = next_u32();
        return lo | (hi << 32);
    }
};

// Fills rc[360]; returns false if the fingerprints do not match.
inline bool generate(uint64_t* rc) {
    const uint64_t P = 0xFFFFFFFF00000001ULL;
    ChaCha8Stream rng(0);
    int n = 0;
    while (n < 360) {
        // rand::distributions::uniform::UniformInt<u64>::sample_single(0, p): widening multiply with
        // rejection zone (p << leading_zeros(p)) - 1 = p - 1
        unsigned __int128 wide = (unsigned __int128)rng.next_u64() * P;
        if ((uint64_t)wide <= P - 1) rc[n++] = (uint64_t)(wide >> 64);
    }
    uint64_t x = 0;
    for (int i = 0; i < 360; i++) x ^= rc[i];
    return x == 0xd95d3c3bb2fe42e3ULL && rc[0] == 0xb585f766f2144405ULL && rc[359] == 0xbc8dfb627fe558fcULL;
}

// The constant tables of the FP64 linear layers (poseidon.cuh), as integer bit patterns of denormal doubles:
//   split[(round) * 12 + lane] = (rc & 0xffffffff, rc >> 32), one extra all-zero round 30;
//   pair_k[pair * 12 + lane]   = sum_{i>=1} M[lane][i] * rc[a+1][i] + rc[a+2][lane], a = 4 + 2 pair, by 32-bit halves.
// signed_sbox: the S-box hands the linear layer (r0 - r2 - r3, r1 + r2) of its last 128-bit product, the first of which
// can be as low as -2^33; every constant a sum with such a term meets then carries an offset that is 0 mod p and makes
// the low accumulator positive: value = A + 2^32 B, p = 1 + 2^32 (2^32 - 1), so (A, B) += (2^e + k, k (2^32 - 1) - 2^(e-32))
// with k = 1 (e = 42: one linear layer, gain <= 280) or k = 2^16 (e = 48: the fused pair, gain < 2^14.1 on lane 0).
// handoff_bias: the device's S-box hands over r0 - r2 - r3 + handoff_bias (non-negative) instead of the signed coefficient,
// so each low (A) entry loses handoff_bias times the total weight of the S-box outputs in its row.  Every accumulator the
// fold sees is then the same integer as with the signed coefficients (handoff_bias = 0 describes that schedule).
inline void linear_layer_tables(const uint64_t* rc, const int mds_circ[12], int mds_diag0, bool signed_sbox,
                                uint64_t* split /* [31 * 12 * 2] */, uint64_t* pair_k /* [11 * 12 * 2] */,
                                uint64_t handoff_bias = 0) {
    auto entry = [&](int r, int j) { return mds_circ[(j - r + 12) % 12] + ((r == 0 && j == 0) ? mds_diag0 : 0); };
    for (int i = 0; i < 31 * 12; i++) {
        const uint64_t v = i < 360 ? rc[i] : 0;
        split[2 * i] = v & 0xFFFFFFFFULL;
        split[2 * i + 1] = v >> 32;
    }
    if (signed_sbox) {
        const uint64_t offA = (1ULL << 42) + 1, offB = 0xFFFFFFFFULL - (1ULL << 10);
        for (int round = 0; round < 31; round++) {
            const bool full_layer = (round >= 1 && round <= 4) || (round >= 27 && round <= 30);   // added by a full round's layer
            const bool lane0_only = round >= 5 && round <= 25 && (round & 1);                   // y0 of a fused pair
            for (int lane = 0; lane < 12; lane++)
                if (full_layer || (lane0_only && lane == 0)) {
                    // a full round's row sees all twelve S-box outputs, y0 of a pair only lane 0's
                    uint64_t weight = 0;
                    for (int j = 0; j < (full_layer ? 12 : 1); j++) weight += (uint64_t)entry(lane, j);
                    split[2 * (round * 12 + lane)] += offA - handoff_bias * weight;
                    split[2 * (round * 12 + lane) + 1] += offB;
                }
        }
    }
    for (int pair = 0; pair < 11; pair++) {
        const uint64_t* r1 = rc + (4 + 2 * pair + 1) * 12;
        const uint64_t* r2 = rc + (4 + 2 * pair + 2) * 12;
        for (int lane = 0; lane < 12; lane++) {
            uint64_t lo = r2[lane] & 0xFFFFFFFFULL, hi = r2[lane] >> 32;
            for (int i = 1; i < 12; i++) {
                lo += (uint64_t)entry(lane, i) * (r1[i] & 0xFFFFFFFFULL);
                hi += (uint64_t)entry(lane, i) * (r1[i] >> 32);
            }
            if (signed_sbox) {
                // the S-box outputs of the pair reach row `lane` as N[lane][0] x~_0 (N = M M' without the lane-0 path:
                // CIRC^2 x~ + col0(CIRC) (8 x~_0 - Yraw) on the device) and M[lane][0] sigma
                uint64_t weight = (uint64_t)entry(lane, 0);
                for (int i = 1; i < 12; i++) weight += (uint64_t)entry(lane, i) * (uint64_t)entry(i, 0);
                lo += (1ULL << 48) + (1ULL << 16) - handoff_bias * weight;
                hi += (1ULL << 16) * 0xFFFFFFFFULL - (1ULL << 16);
            }
            pair_k[(pair * 12 + lane) * 2] = lo;
            pair_k[(pair * 12 + lane) * 2 + 1] = hi;
        }
    }
}

}  // namespace poseidon_constants
