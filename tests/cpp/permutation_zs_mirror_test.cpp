// all_wires_permutation_partial_products through the C++ host mirror (include/plonky2_b200.hpp): commits a small fixed
// instance (splitmix64 wires and constants, identity sigmas k_j w^i with eight swapped pairs of routed positions that hold
// equal wire values), computes the Z and partial-product columns and writes them, then the grand products, to argv[1].
// tests/test_gpu_permutation_zs.py builds the same instance with the Python mirror and compares the two dumps.
#include <cstdio>

#include "plonky2_b200.hpp"

using namespace plonky2_b200;

static const uint64_t P = 0xFFFFFFFF00000001ULL;

static uint64_t splitmix(uint64_t x) {
    x += 0x9E3779B97F4A7C15ULL;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ULL;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBULL;
    x ^= x >> 31;
    return x >= P ? x - P : x;
}
static uint64_t mulmod(uint64_t a, uint64_t b) { return (uint64_t)((unsigned __int128)a * b % P); }

int main(int argc, char** argv) {
    if (argc < 2) return 2;
    Context ctx(0);
    const uint32_t lg_n = 6, R = 20, num_wires = 24, num_constants = 3, deg = 4;
    const size_t n = (size_t)1 << lg_n;
    std::vector<std::vector<F>> wires(num_wires, std::vector<F>(n)), cs(num_constants + R, std::vector<F>(n));
    for (uint32_t j = 0; j < num_wires; j++)
        for (size_t i = 0; i < n; i++) wires[j][i] = splitmix(((uint64_t)j << 32) + i);
    for (uint32_t j = 0; j < num_constants; j++)
        for (size_t i = 0; i < n; i++) cs[j][i] = splitmix(((uint64_t)(100 + j) << 32) + i);
    std::vector<F> k_is(R);
    const F w = detail::pow_mod(detail::pow_mod(7, (P - 1) >> 32), 1ull << (32 - lg_n));
    for (uint32_t j = 0; j < R; j++) {
        k_is[j] = detail::pow_mod(7, j);
        F x = 1;
        for (size_t i = 0; i < n; i++, x = mulmod(x, w)) cs[num_constants + j][i] = mulmod(k_is[j], x);
    }
    for (uint32_t t = 0; t < 8; t++) {   // (t, 2t + 1) <-> (t + 10, 5t + 3)
        std::swap(cs[num_constants + t][2 * t + 1], cs[num_constants + t + 10][5 * t + 3]);
        wires[t + 10][5 * t + 3] = wires[t][2 * t + 1];
    }
    const CircuitConfig cfg;
    PolynomialBatch csb = PolynomialBatch::from_values(ctx, cs, cfg.fri_config.rate_bits, false, cfg.fri_config.cap_height);
    PolynomialBatch wb = PolynomialBatch::from_values(ctx, wires, cfg.fri_config.rate_bits, false, cfg.fri_config.cap_height);
    gl_circuit circuit = {};
    circuit.degree_bits = lg_n;
    circuit.num_wires = num_wires;
    circuit.num_routed_wires = R;
    circuit.num_constants = num_constants;
    circuit.num_challenges = 2;
    circuit.quotient_degree_factor = deg;
    PermutationZs z = all_wires_permutation_partial_products(ctx, circuit, k_is, csb, wb, {11, 13}, {17, 19});

    FILE* f = std::fopen(argv[1], "w");
    if (!f) return 3;
    for (auto& col : z.zs_partial_products)
        for (F v : col) std::fprintf(f, "%llu\n", (unsigned long long)v);
    for (F g : z.grand_products) std::fprintf(f, "%llu\n", (unsigned long long)g);
    std::fclose(f);
    std::printf("permutation_zs_mirror_test ok: %zu columns\n", z.zs_partial_products.size());
    return 0;
}
