// plonky2::plonk::prover::prove through the C++ host mirror (include/plonky2_b200.hpp): commits the constants / sigmas of
// a small fixed circuit (a PublicInputGate row, ConstantGate rows, NoopGate rows; splitmix64 wires; identity sigmas k_j w^i
// with eight swapped pairs of routed positions that hold equal wire values), proves it and writes the proof's words to
// argv[1].  tests/test_gpu_prove.py builds the same instance with the Python mirror and compares the two dumps.
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
    const uint32_t lg_n = 6, R = 20, num_wires = 24, num_constants = 3;
    const size_t n = (size_t)1 << lg_n;
    std::vector<std::vector<F>> wires(num_wires, std::vector<F>(n)), cs(num_constants + R, std::vector<F>(n, 0));
    for (uint32_t j = 0; j < num_wires; j++)
        for (size_t i = 0; i < n; i++) wires[j][i] = splitmix(((uint64_t)j << 32) + i);
    const std::vector<F> public_inputs = {5, 6, 7};
    const HashOut pih = PoseidonHash::hash_no_pad(ctx, public_inputs);
    cs[0][0] = 2;                                   // row 0: PublicInputGate
    for (int e = 0; e < 4; e++) wires[e][0] = pih.elements[e];
    for (size_t i = 1; i < n; i++) {
        if (i % 5 == 1) {                           // ConstantGate { num_consts: 2 }
            cs[0][i] = 1;
            cs[1][i] = wires[0][i] = splitmix(((uint64_t)200 << 32) + i);
            cs[2][i] = wires[1][i] = splitmix(((uint64_t)201 << 32) + i);
        }                                           // else NoopGate: selector 0
    }
    std::vector<F> k_is(R);
    const F w = detail::pow_mod(detail::pow_mod(7, (P - 1) >> 32), 1ull << (32 - lg_n));
    for (uint32_t j = 0; j < R; j++) {
        k_is[j] = detail::pow_mod(7, j);
        F x = 1;
        for (size_t i = 0; i < n; i++, x = mulmod(x, w)) cs[num_constants + j][i] = mulmod(k_is[j], x);
    }
    for (uint32_t t = 0; t < 8; t++) {   // (t + 4, 2t + 3) <-> (t + 10, 5t + 7): neither end is in a gate's wires
        std::swap(cs[num_constants + t + 4][2 * t + 3], cs[num_constants + t + 10][5 * t + 7]);
        wires[t + 10][5 * t + 7] = wires[t + 4][2 * t + 3];
    }
    const CircuitConfig cfg;
    PolynomialBatch csb = PolynomialBatch::from_values(ctx, cs, cfg.fri_config.rate_bits, false, cfg.fri_config.cap_height);
    gl_circuit circuit = {};
    circuit.degree_bits = lg_n;
    circuit.num_wires = num_wires;
    circuit.num_routed_wires = R;
    circuit.num_constants = num_constants;
    circuit.num_selectors = 1;
    circuit.num_challenges = 2;
    circuit.quotient_degree_factor = 8;
    circuit.num_gates = 3;
    const std::vector<gl_gate> gates = {{GL_GATE_NOOP, 0, 0, 0, 3, 0}, {GL_GATE_CONSTANT, 2, 0, 0, 3, 0},
                                        {GL_GATE_PUBLIC_INPUT, 0, 0, 0, 3, 0}};
    const HashOut digest = {{1, 2, 3, 4}};
    const FriParams fp = FriParams::for_degree(cfg.fri_config, lg_n);
    ProofWithPublicInputs proof = prove(ctx, circuit, gates, k_is, csb, digest, fp, wires, public_inputs);

    FILE* f = std::fopen(argv[1], "w");
    if (!f) return 3;
    for (uint64_t v : proof.words) std::fprintf(f, "%llu\n", (unsigned long long)v);
    std::fclose(f);
    std::printf("prove_mirror_test ok: %zu words, %zu query rounds\n", proof.words.size(), proof.opening_proof.query_round_proofs.size());
    return 0;
}
