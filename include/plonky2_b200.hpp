// plonky2_b200.hpp -- header-only C++ host mirror of the plonky2 plugin surface that Plonky2-lib reaches,
// over the C ABI of gl_b200.h.  The reference's host language is Rust (no cargo/rustc in this image), so the
// host side above the C ABI is C++ with the SAME names, argument meaning and error behaviour as upstream:
//
//   plonky2::fri::oracle::PolynomialBatch::{from_values, from_coeffs, get_lde_values}
//   plonky2::hash::merkle_tree::MerkleTree::{new, get, prove}        (MerkleTree::build here: `new` is a keyword)
//   plonky2::hash::poseidon::PoseidonHash::{hash_no_pad, hash_pad, hash_or_noop, two_to_one}
//   plonky2::fri::FriConfig / plonk::circuit_data::CircuitConfig presets
//   plonky2::iop::challenger::Challenger, plonky2::fri::prover::fri_proof, PolynomialBatch::prove_openings (N1)
//   src/smt/goldilocks_poseidon/mod.rs:158-184  PoseidonNodeHash::calc_node_hash
//
// Upstream is infallible and panics on contract violations; here a violation throws plonky2_b200::Panic.
// Nothing in this header computes field arithmetic: every result comes from libgl_b200.so.
#pragma once
#include <cstdint>
#include <memory>
#include <stdexcept>
#include <array>
#include <string>
#include <utility>
#include <cstring>
#include <vector>

#include "gl_b200.h"

namespace plonky2_b200 {

using F = uint64_t;  // GoldilocksField, canonical u64

struct Panic : std::runtime_error {
    int code;
    Panic(int c, const std::string& m) : std::runtime_error(m), code(c) {}
};

struct HashOut {
    F elements[4];
    bool operator==(const HashOut& o) const {
        return elements[0] == o.elements[0] && elements[1] == o.elements[1] && elements[2] == o.elements[2] &&
               elements[3] == o.elements[3];
    }
    // WrappedHashOut's text form (src/smt/goldilocks_poseidon/hash/mod.rs:84-119): "0x" + the 32 bytes of to_bytes()
    // (4 x u64 little endian) in reverse order, i.e. elements[3] first, each as 16 hex digits
    std::string to_hex() const {
        static const char* d = "0123456789abcdef";
        std::string s = "0x";
        for (int e = 3; e >= 0; e--)
            for (int sh = 60; sh >= 0; sh -= 4) s.push_back(d[(elements[e] >> sh) & 15]);
        return s;
    }
};
using MerkleCap = std::vector<HashOut>;
struct MerkleProof {
    std::vector<HashOut> siblings;
};

class Context {
   public:
    explicit Context(int device = 0) {
        int rc = gl_ctx_create(device, &ctx_);
        if (rc) throw Panic(rc, gl_last_error(nullptr));
    }
    ~Context() { gl_ctx_destroy(ctx_); }
    Context(const Context&) = delete;
    Context& operator=(const Context&) = delete;
    gl_ctx* raw() const { return ctx_; }
    void check(int rc) const {
        if (rc) throw Panic(rc, gl_last_error(ctx_));
    }
    void set_shard(uint32_t index, uint32_t count) { check(gl_ctx_set_shard(ctx_, index, count)); }

   private:
    gl_ctx* ctx_ = nullptr;
};

// ---- FriConfig / CircuitConfig presets (the only configuration Plonky2-lib passes down) -------------
struct FriReductionStrategy {  // ConstantArityBits(arity_bits, final_poly_bits)
    uint32_t arity_bits = 4, final_poly_bits = 5;
    std::vector<uint32_t> reduction_arity_bits(uint32_t degree_bits, uint32_t rate_bits, uint32_t cap_height) const {
        std::vector<uint32_t> out;
        while (degree_bits > final_poly_bits && degree_bits + rate_bits - arity_bits >= cap_height) {
            out.push_back(arity_bits);
            degree_bits -= arity_bits;
        }
        return out;
    }
};
struct FriConfig {
    uint32_t rate_bits = 3, cap_height = 4, proof_of_work_bits = 16;
    FriReductionStrategy reduction_strategy;
    uint32_t num_query_rounds = 28;
};
struct CircuitConfig {
    uint32_t num_wires = 135, num_routed_wires = 80, num_constants = 2, num_challenges = 2;
    bool zero_knowledge = false;
    uint32_t max_quotient_degree_factor = 8;
    FriConfig fri_config;
    static CircuitConfig standard_recursion_config() { return {}; }
    static CircuitConfig standard_ecc_config() {
        CircuitConfig c;
        c.num_wires = 136;
        return c;
    }
    static CircuitConfig wide_ecc_config() {
        CircuitConfig c;
        c.num_wires = 234;
        return c;
    }
};

// ---- PoseidonHash (Hasher<F>) -----------------------------------------------------------------------
struct PoseidonHash {
    static constexpr size_t HASH_SIZE = 32, SPONGE_WIDTH = 12, SPONGE_RATE = 8;

    // batch forms: the single-shot forms below call them with m = 1
    static std::vector<HashOut> hash_no_pad_batch(const Context& c, const F* inputs, uint32_t len_each, uint64_t m) {
        std::vector<HashOut> out(m);
        c.check(gl_poseidon_hash_no_pad_batch(c.raw(), inputs, len_each, m, &out[0].elements[0], GL_HOST));
        return out;
    }
    static std::vector<HashOut> two_to_one_batch(const Context& c, const HashOut* l, const HashOut* r, uint64_t m) {
        std::vector<HashOut> out(m);
        c.check(gl_poseidon_two_to_one_batch(c.raw(), &l[0].elements[0], &r[0].elements[0], &out[0].elements[0], m, GL_HOST));
        return out;
    }
    static HashOut hash_no_pad(const Context& c, const std::vector<F>& input) {
        return hash_no_pad_batch(c, input.data(), (uint32_t)input.size(), 1)[0];
    }
    static HashOut two_to_one(const Context& c, const HashOut& l, const HashOut& r) { return two_to_one_batch(c, &l, &r, 1)[0]; }
    // pad 1, 0*, 1 to a multiple of SPONGE_WIDTH (this fork generation: src/smt/goldilocks_poseidon/mod.rs:167-181
    // must equal src/smt/gadgets/common.rs:87-101)
    static HashOut hash_pad(const Context& c, const std::vector<F>& input) {
        std::vector<F> p(input);
        p.push_back(1);
        while ((p.size() + 1) % SPONGE_WIDTH) p.push_back(0);
        p.push_back(1);
        return hash_no_pad(c, p);
    }
    static HashOut hash_or_noop(const Context& c, const std::vector<F>& input) {
        if (input.size() <= 4) {
            HashOut h{{0, 0, 0, 0}};
            for (size_t i = 0; i < input.size(); i++) h.elements[i] = input[i] % 0xFFFFFFFF00000001ULL;
            return h;
        }
        return hash_no_pad(c, input);
    }
};

// src/smt/goldilocks_poseidon/mod.rs:158-184
struct PoseidonNodeHash {
    static std::vector<HashOut> calc_leaf_hash_batch(const Context& c, const HashOut* keys, const HashOut* values, uint64_t m) {
        std::vector<HashOut> out(m);
        c.check(gl_smt_leaf_hash_batch(c.raw(), &keys[0].elements[0], &values[0].elements[0], &out[0].elements[0], m, GL_HOST));
        return out;
    }
    static HashOut calc_internal_hash(const Context& c, const HashOut& l, const HashOut& r) {
        return PoseidonHash::two_to_one(c, l, r);
    }
};

// ---- src/smt: batches over the sparse Merkle tree (P7, N2) ---------------------------------------------
// SparseMerkleProcessProof (src/smt/proof/process.rs): what `tree.set(key, value)` returns
struct SparseMerkleProcessProof {
    HashOut old_root, old_key, old_value, new_root, new_key, new_value;
    std::vector<HashOut> siblings;
    bool is_old0 = false;
    uint32_t fnc = 0;  // ProcessMerkleProofRole: 0 NoOp, 1 Update, 2 Insert, 3 Delete
};
struct SparseMerkleTreeBatch {
    // SparseMerkleProcessProof::check for every proof (src/smt/proof/process.rs:47-51): 0 = holds, k = its k-th assert fails
    static std::vector<int32_t> check_process_proofs(const Context& c, const std::vector<SparseMerkleProcessProof>& proofs) {
        const size_t m = proofs.size();
        std::vector<gl_smt_proof_hdr> hdr(m);
        std::vector<uint64_t> off(m + 1, 0), pool;
        for (size_t t = 0; t < m; t++) {
            const SparseMerkleProcessProof& p = proofs[t];
            for (int e = 0; e < 4; e++) {
                hdr[t].old_root[e] = p.old_root.elements[e]; hdr[t].old_key[e] = p.old_key.elements[e];
                hdr[t].old_value[e] = p.old_value.elements[e]; hdr[t].new_root[e] = p.new_root.elements[e];
                hdr[t].new_key[e] = p.new_key.elements[e]; hdr[t].new_value[e] = p.new_value.elements[e];
            }
            hdr[t].is_old0 = p.is_old0;
            hdr[t].fnc = p.fnc;
            for (auto& sb : p.siblings) pool.insert(pool.end(), sb.elements, sb.elements + 4);
            off[t + 1] = off[t] + p.siblings.size();
        }
        std::vector<int32_t> status(m);
        if (pool.empty()) pool.resize(4);
        c.check(gl_smt_verify_process_batch(c.raw(), hdr.data(), pool.data(), off.data(), m, status.data(), GL_HOST));
        return status;
    }
    // root after `tree.set(keys[t], values[t])` for every t on an empty tree (new keys only; src/smt/tree.rs:143-155)
    static HashOut root_of(const Context& c, const std::vector<HashOut>& keys, const std::vector<HashOut>& values) {
        HashOut root{{0, 0, 0, 0}};
        uint64_t count = 0;
        c.check(gl_smt_build(c.raw(), keys.empty() ? nullptr : &keys[0].elements[0], values.empty() ? nullptr : &values[0].elements[0],
                             keys.size(), root.elements, nullptr, 0, &count, nullptr, GL_HOST));
        return root;
    }
    // the proofs those `set` calls return, in call order
    static std::vector<SparseMerkleProcessProof> set_proofs(const Context& c, const std::vector<HashOut>& keys,
                                                               const std::vector<HashOut>& values) {
        const size_t m = keys.size();
        std::vector<SparseMerkleProcessProof> out(m);
        if (!m) return out;
        std::vector<gl_smt_proof_hdr> hdr(m);
        std::vector<uint64_t> off(m + 1), pool((size_t)4 * 32 * m);
        uint64_t total = 0;
        for (;;) {
            c.check(gl_smt_set_proofs(c.raw(), &keys[0].elements[0], &values[0].elements[0], m, hdr.data(), pool.data(),
                                         pool.size() / 4, off.data(), &total, GL_HOST));
            if (total * 4 <= pool.size()) break;
            pool.resize(total * 4);
        }
        for (size_t t = 0; t < m; t++) {
            SparseMerkleProcessProof& p = out[t];
            for (int e = 0; e < 4; e++) {
                p.old_root.elements[e] = hdr[t].old_root[e]; p.old_key.elements[e] = hdr[t].old_key[e];
                p.old_value.elements[e] = hdr[t].old_value[e]; p.new_root.elements[e] = hdr[t].new_root[e];
                p.new_key.elements[e] = hdr[t].new_key[e]; p.new_value.elements[e] = hdr[t].new_value[e];
            }
            p.is_old0 = hdr[t].is_old0 != 0;
            p.fnc = hdr[t].fnc;
            for (uint64_t s = off[t]; s < off[t + 1]; s++) {
                HashOut h;
                for (int e = 0; e < 4; e++) h.elements[e] = pool[4 * s + e];
                p.siblings.push_back(h);
            }
        }
        return out;
    }
};

// ---- MerkleTree ---------------------------------------------------------------------------------------
struct MerkleTree {
    std::vector<std::vector<F>> leaves;
    std::vector<HashOut> digests;
    MerkleCap cap;
    uint32_t cap_height = 0;

    // MerkleTree::new(leaves, cap_height)
    static MerkleTree build(const Context& c, std::vector<std::vector<F>> leaves, uint32_t cap_height) {
        MerkleTree t;
        const uint64_t n = leaves.size();
        const uint32_t len = n ? (uint32_t)leaves[0].size() : 0;
        std::vector<F> flat;
        flat.reserve(n * len);
        for (auto& row : leaves) {
            if (row.size() != len) throw Panic(GL_E_ARG, "MerkleTree::new: ragged leaves");
            flat.insert(flat.end(), row.begin(), row.end());
        }
        uint64_t nd = n >= (1ull << cap_height) ? 2 * (n - (1ull << cap_height)) : 0;
        t.digests.resize(nd);
        t.cap.resize(1ull << cap_height);
        c.check(gl_merkle_build(c.raw(), flat.data(), n, len, cap_height, nd ? &t.digests[0].elements[0] : nullptr,
                                &t.cap[0].elements[0], GL_HOST));
        t.leaves = std::move(leaves);
        t.cap_height = cap_height;
        return t;
    }
    const std::vector<F>& get(size_t i) const { return leaves[i]; }
    // verify_merkle_proof_to_cap (plonky2::hash::merkle_proofs) for a batch of openings against one cap; every proof
    // must have the same length (they do when they come from one tree)
    static std::vector<bool> verify_batch(const Context& c, const std::vector<std::vector<F>>& rows, const std::vector<uint64_t>& idx,
                                          const std::vector<MerkleProof>& proofs, const MerkleCap& cap) {
        const size_t k = rows.size();
        std::vector<bool> out(k);
        if (!k) return out;
        const uint32_t len = (uint32_t)rows[0].size(), L = (uint32_t)proofs[0].siblings.size();
        std::vector<F> flat, paths;
        for (size_t i = 0; i < k; i++) {
            if (rows[i].size() != len || proofs[i].siblings.size() != L) throw Panic(GL_E_ARG, "verify_batch: ragged openings");
            flat.insert(flat.end(), rows[i].begin(), rows[i].end());
            for (auto& s : proofs[i].siblings) paths.insert(paths.end(), s.elements, s.elements + 4);
        }
        uint32_t h = 0;
        while ((1ull << h) < cap.size()) h++;
        std::vector<int32_t> ok(k);
        if (paths.empty()) paths.resize(4);
        c.check(gl_merkle_verify_batch(c.raw(), flat.data(), len, idx.data(), paths.data(), L, &cap[0].elements[0], h, k, ok.data(), GL_HOST));
        for (size_t i = 0; i < k; i++) out[i] = ok[i] != 0;
        return out;
    }
    MerkleProof prove(size_t leaf_index) const {
        MerkleProof p;
        size_t n = leaves.size();
        uint32_t lg = 0;
        while ((1ull << lg) < n) lg++;
        uint32_t L = lg - cap_height;
        if (L == 0) return p;
        size_t per = 2 * ((1ull << L) - 1), sub = leaf_index >> L, pair = leaf_index & ((1ull << L) - 1);
        const HashOut* buf = digests.data() + sub * per;
        for (uint32_t i = 0; i < L; i++) {
            size_t parity = pair & 1;
            pair >>= 1;
            p.siblings.push_back(buf[2 * ((pair << (i + 1)) + (1ull << i) - 1) + (1 - parity)]);
        }
        return p;
    }
};

// ---- PolynomialBatch (resident mode) ------------------------------------------------------------------
class PolynomialBatch {
   public:
    std::vector<std::vector<F>> polynomials;  // coefficients
    MerkleCap cap;                            // merkle_tree.cap
    uint32_t degree_log = 0, rate_bits = 0, cap_height = 0;
    bool blinding = false;
    uint32_t leaf_len = 0;   // merkle_tree.leaves[i].len(): polynomials.size() + SALT_SIZE when blinding

    // values: one Vec per polynomial (Vec<PolynomialValues<F>>); `timing` / `fft_root_table` of the upstream
    // signature have no meaning on the device and are not taken.
    static PolynomialBatch from_values(const Context& c, const std::vector<std::vector<F>>& values, uint32_t rate_bits,
                                       bool blinding, uint32_t cap_height) {
        return make(c, values, true, rate_bits, blinding, cap_height);
    }
    static PolynomialBatch from_coeffs(const Context& c, const std::vector<std::vector<F>>& coeffs, uint32_t rate_bits,
                                       bool blinding, uint32_t cap_height) {
        return make(c, coeffs, false, rate_bits, blinding, cap_height);
    }
    // (tree.get(i), tree.prove(i)) for every i
    std::pair<std::vector<std::vector<F>>, std::vector<MerkleProof>> open(const std::vector<uint64_t>& idx) const {
        const uint32_t k = (uint32_t)idx.size(), cols = leaf_len;
        const uint32_t L = degree_log + rate_bits - cap_height;
        std::vector<F> rows((size_t)k * cols), paths((size_t)k * L * 4);
        ctx_->check(gl_commit_open(h_, idx.data(), k, rows.data(), paths.data(), GL_HOST));
        std::pair<std::vector<std::vector<F>>, std::vector<MerkleProof>> out;
        for (uint32_t q = 0; q < k; q++) {
            out.first.emplace_back(rows.begin() + (size_t)q * cols, rows.begin() + (size_t)(q + 1) * cols);
            MerkleProof p;
            for (uint32_t l = 0; l < L; l++) {
                HashOut d;
                for (int e = 0; e < 4; e++) d.elements[e] = paths[((size_t)q * L + l) * 4 + e];
                p.siblings.push_back(d);
            }
            out.second.push_back(std::move(p));
        }
        return out;
    }
    // OpeningSet::new for this batch: every polynomial at the extension point (a0, a1) -> [columns] x (c0, c1)
    std::vector<std::array<F, 2>> eval_at(const F point[2]) const {
        std::vector<std::array<F, 2>> out(polynomials.size());
        ctx_->check(gl_commit_eval(h_, point, &out[0][0], GL_HOST));
        return out;
    }
    std::vector<F> get_lde_values(uint64_t index, uint64_t step) const {
        std::vector<F> row(polynomials.size());
        ctx_->check(gl_commit_get_lde_values(h_, &index, 1, step, row.data(), GL_HOST));
        return row;
    }
    // mirror mode: MerkleTree.leaves / .digests exactly as upstream lays them out
    void download(std::vector<F>* leaves_row_major, std::vector<HashOut>* digests) const {
        uint64_t lo, hi;
        gl_commit_info(h_, nullptr, nullptr, nullptr, nullptr, &lo, &hi);
        if (leaves_row_major) leaves_row_major->resize((hi - lo) * leaf_len);
        uint64_t caps_local = (uint64_t)cap.size() * (hi - lo) >> (degree_log + rate_bits);
        if (digests) digests->resize(2 * ((hi - lo) - caps_local));
        ctx_->check(gl_commit_download(h_, leaves_row_major ? leaves_row_major->data() : nullptr,
                                       digests && !digests->empty() ? &(*digests)[0].elements[0] : nullptr, GL_HOST));
    }
    gl_commit* raw_handle() const { return h_; }  // the resident commit (for the FRI functions below)
    PolynomialBatch(PolynomialBatch&& o) noexcept { *this = std::move(o); }
    PolynomialBatch& operator=(PolynomialBatch&& o) noexcept {
        std::swap(polynomials, o.polynomials);
        std::swap(cap, o.cap);
        std::swap(degree_log, o.degree_log);
        std::swap(rate_bits, o.rate_bits);
        std::swap(cap_height, o.cap_height);
        std::swap(blinding, o.blinding);
        std::swap(leaf_len, o.leaf_len);
        std::swap(h_, o.h_);
        std::swap(ctx_, o.ctx_);
        return *this;
    }
    ~PolynomialBatch() {
        if (h_) gl_commit_free(h_);
    }

   private:
    PolynomialBatch() = default;
    static PolynomialBatch make(const Context& c, const std::vector<std::vector<F>>& polys, bool is_values,
                                uint32_t rate_bits, bool blinding, uint32_t cap_height) {
        if (polys.empty()) throw Panic(GL_E_ARG, "PolynomialBatch: empty batch");
        const size_t n = polys[0].size();
        if (n == 0 || (n & (n - 1))) throw Panic(GL_E_ARG, "log2_strict: polynomial length is not a power of two");
        uint32_t lg = 0;
        while ((1ull << lg) < n) lg++;
        // one pointer per polynomial, exactly where the caller's Vecs lie (gl_commit_from_values_cols): no flattening
        std::vector<const uint64_t*> cols;
        for (auto& p : polys) {
            if (p.size() != n) throw Panic(GL_E_ARG, "assert_eq!(p.len(), degree)");
            cols.push_back(p.data());
        }
        PolynomialBatch b;
        b.ctx_ = &c;
        b.degree_log = lg;
        b.rate_bits = rate_bits;
        b.cap_height = cap_height;
        b.cap.resize(1ull << cap_height);
        int rc;
        if (is_values) {
            b.polynomials.assign(polys.size(), std::vector<F>(n));
            std::vector<uint64_t*> outs;
            for (auto& p : b.polynomials) outs.push_back(p.data());
            rc = gl_commit_from_values_ex(c.raw(), nullptr, cols.data(), lg, (uint32_t)polys.size(), rate_bits, blinding ? 1 : 0,
                                          cap_height, nullptr, outs.data(), &b.cap[0].elements[0], &b.h_, GL_HOST);
        } else {
            rc = gl_commit_from_coeffs_ex(c.raw(), nullptr, cols.data(), lg, (uint32_t)polys.size(), rate_bits, blinding ? 1 : 0,
                                          cap_height, &b.cap[0].elements[0], &b.h_, GL_HOST);
            if (rc == GL_OK) b.polynomials = polys;
        }
        c.check(rc);
        b.blinding = blinding;
        c.check(gl_commit_leaf_len(b.h_, &b.leaf_len));
        return b;
    }
    gl_commit* h_ = nullptr;
    const Context* ctx_ = nullptr;
};

// ---- plonky2::iop::challenger::Challenger (host side of the Fiat-Shamir transcript) -----------------------------
class Challenger {
   public:
    explicit Challenger(const Context& c) : ctx_(&c) {
        for (auto& v : sponge_state) v = 0;
    }
    F sponge_state[12];
    std::vector<F> input_buffer, output_buffer;

    void observe_element(F e) {
        output_buffer.clear();  // any buffered outputs are now invalid
        input_buffer.push_back(e % 0xFFFFFFFF00000001ULL);
        if (input_buffer.size() == PoseidonHash::SPONGE_RATE) duplexing();
    }
    // same transcript as element-by-element observation; runs of full input buffers go to the device as one chain
    void observe_elements(const F* es, size_t n) {
        const size_t R = PoseidonHash::SPONGE_RATE;
        if ((input_buffer.size() + n) / R < 2) {
            for (size_t i = 0; i < n; i++) observe_element(es[i]);
            return;
        }
        std::vector<F> pending(input_buffer);
        for (size_t i = 0; i < n; i++) pending.push_back(es[i] % 0xFFFFFFFF00000001ULL);
        const size_t m = pending.size() / R;
        ctx_->check(gl_poseidon_duplex_chain(ctx_->raw(), sponge_state, pending.data(), m));
        input_buffer.assign(pending.begin() + m * R, pending.end());
        output_buffer.clear();
        if (input_buffer.empty()) output_buffer.assign(sponge_state, sponge_state + R);
    }
    void observe_hash(const HashOut& h) { observe_elements(h.elements, 4); }
    void observe_cap(const MerkleCap& cap) {
        std::vector<F> flat;
        for (auto& h : cap) flat.insert(flat.end(), h.elements, h.elements + 4);
        observe_elements(flat.data(), flat.size());
    }
    void observe_extension_element(const F e[2]) { observe_elements(e, 2); }
    F get_challenge() {
        if (!input_buffer.empty() || output_buffer.empty()) duplexing();
        F v = output_buffer.back();
        output_buffer.pop_back();
        return v;
    }
    void get_extension_challenge(F out[2]) {
        out[0] = get_challenge();
        out[1] = get_challenge();
    }

   private:
    void duplexing() {
        for (size_t i = 0; i < input_buffer.size(); i++) sponge_state[i] = input_buffer[i];  // overwrite mode
        input_buffer.clear();
        ctx_->check(gl_poseidon_permute_batch(ctx_->raw(), sponge_state, 1, GL_HOST));
        output_buffer.assign(sponge_state, sponge_state + PoseidonHash::SPONGE_RATE);
    }
    const Context* ctx_;
};

// ---- plonky2::fri: FriParams, proof structures, fri_proof, PolynomialBatch::prove_openings ----------------------
struct FriParams {
    FriConfig config;
    bool hiding = false;
    uint32_t degree_bits = 0;
    std::vector<uint32_t> reduction_arity_bits;
    static FriParams for_degree(const FriConfig& cfg, uint32_t degree_bits) {
        FriParams p;
        p.config = cfg;
        p.degree_bits = degree_bits;
        p.reduction_arity_bits = cfg.reduction_strategy.reduction_arity_bits(degree_bits, cfg.rate_bits, cfg.cap_height);
        return p;
    }
};
struct FriBatchInfo {  // FriBatchInfo: polynomials (oracle_index, polynomial_index) opened at `point`
    F point[2];
    std::vector<std::pair<uint32_t, uint32_t>> polynomials;
};
struct FriQueryStep {
    std::vector<F> evals;  // arity extension elements, flattened
    MerkleProof merkle_proof;
};
struct FriQueryRound {
    uint64_t x_index = 0;
    std::vector<std::pair<std::vector<F>, MerkleProof>> initial_trees_proof;  // per oracle: (row, path)
    std::vector<FriQueryStep> steps;
};
struct FriProof {
    std::vector<MerkleCap> commit_phase_merkle_caps;
    std::vector<FriQueryRound> query_round_proofs;
    std::vector<F> final_poly;  // extension coefficients, flattened [len][2]
    F pow_witness = 0;
};

namespace detail {
struct DevBuf {  // gl_dev_alloc block
    const Context* c;
    void* p = nullptr;
    DevBuf(const Context& ctx, size_t bytes) : c(&ctx) { ctx.check(gl_dev_alloc(ctx.raw(), bytes, &p)); }
    ~DevBuf() { gl_dev_free(c->raw(), p); }
    DevBuf(const DevBuf&) = delete;
    DevBuf& operator=(const DevBuf&) = delete;
    uint64_t* u64() const { return static_cast<uint64_t*>(p); }
};
struct LayerTree {  // resident layer tree of fri_committed_trees
    gl_commit* h = nullptr;
    uint32_t arity_bits = 0, lg_leaves = 0;
    MerkleCap cap;
};
inline F pow_mod(F b, uint64_t e) {
    const unsigned __int128 P = 0xFFFFFFFF00000001ULL;
    unsigned __int128 r = 1, x = b % (F)P;
    while (e) {
        if (e & 1) r = r * x % P;
        x = x * x % P;
        e >>= 1;
    }
    return (F)r;
}
inline std::pair<std::vector<std::vector<F>>, std::vector<MerkleProof>> open_handle(const Context& c, gl_commit* h, uint32_t cols,
                                                                                   uint32_t path_len,
                                                                                   const std::vector<uint64_t>& idx) {
    const uint32_t k = (uint32_t)idx.size();
    std::vector<F> rows((size_t)k * cols), paths((size_t)k * path_len * 4 + 4);
    c.check(gl_commit_open(h, idx.data(), k, rows.data(), paths.data(), GL_HOST));
    std::pair<std::vector<std::vector<F>>, std::vector<MerkleProof>> out;
    for (uint32_t q = 0; q < k; q++) {
        out.first.emplace_back(rows.begin() + (size_t)q * cols, rows.begin() + (size_t)(q + 1) * cols);
        MerkleProof p;
        for (uint32_t l = 0; l < path_len; l++) {
            HashOut d;
            for (int e = 0; e < 4; e++) d.elements[e] = paths[((size_t)q * path_len + l) * 4 + e];
            p.siblings.push_back(d);
        }
        out.second.push_back(std::move(p));
    }
    return out;
}
}  // namespace detail

// plonky2::fri::prover::fri_proof on device-resident inputs: lde_coeffs / lde_values are gl_dev_alloc blocks of
// n extension elements ([n][2], natural order); the oracles answer the initial openings.  Commit phase
// (fri_committed_trees), proof of work (smallest witness; upstream: any) and the query rounds.
inline FriProof fri_proof_resident(const Context& c, const std::vector<const PolynomialBatch*>& oracles, uint64_t* lde_coeffs,
                                   uint64_t* lde_values, uint64_t n, Challenger& challenger, const FriParams& fp) {
    FriProof proof;
    std::vector<detail::LayerTree> trees;
    std::vector<std::unique_ptr<detail::DevBuf>> owned;  // folded coefficients / values of the layers
    uint64_t *coeffs = lde_coeffs, *values = lde_values, len = n;
    F shift = 7;  // F::MULTIPLICATIVE_GROUP_GENERATOR
    uint32_t lg = 0;
    while ((1ull << lg) < n) lg++;
    for (uint32_t arity_bits : fp.reduction_arity_bits) {
        detail::LayerTree t;
        t.arity_bits = arity_bits;
        t.lg_leaves = lg - arity_bits;
        t.cap.resize(1ull << fp.config.cap_height);
        detail::DevBuf cap_dev(c, t.cap.size() * 32);
        c.check(gl_fri_layer_commit(c.raw(), values, len, arity_bits, fp.config.cap_height, cap_dev.u64(), &t.h, GL_DEVICE));
        c.check(gl_copy(c.raw(), &t.cap[0].elements[0], GL_HOST, cap_dev.p, GL_DEVICE, t.cap.size() * 32));
        challenger.observe_cap(t.cap);
        proof.commit_phase_merkle_caps.push_back(t.cap);
        trees.push_back(t);
        F beta[2];
        challenger.get_extension_challenge(beta);
        shift = detail::pow_mod(shift, 1ull << arity_bits);
        const uint64_t out_len = len >> arity_bits;
        owned.emplace_back(new detail::DevBuf(c, out_len * 16));
        owned.emplace_back(new detail::DevBuf(c, out_len * 16));
        uint64_t* folded = owned[owned.size() - 2]->u64();
        uint64_t* next = owned[owned.size() - 1]->u64();
        c.check(gl_fri_fold(c.raw(), coeffs, len, arity_bits, beta, shift, folded, next, GL_DEVICE));
        coeffs = folded;
        values = next;
        len = out_len;
        lg -= arity_bits;
    }
    // the coefficients being removed here are always zero
    const uint64_t final_len = len >> fp.config.rate_bits;
    proof.final_poly.resize(final_len * 2);
    c.check(gl_copy(c.raw(), proof.final_poly.data(), GL_HOST, coeffs, GL_DEVICE, final_len * 16));
    challenger.observe_elements(proof.final_poly.data(), proof.final_poly.size());
    // fri_proof_of_work
    {
        F state[12];
        for (int i = 0; i < 12; i++) state[i] = challenger.sponge_state[i];
        const uint32_t pos = (uint32_t)challenger.input_buffer.size();
        for (uint32_t i = 0; i < pos; i++) state[i] = challenger.input_buffer[i];
        const uint32_t min_lz = fp.config.proof_of_work_bits;  // + (64 - F::order().bits()) = + 0
        c.check(gl_pow_grind(c.raw(), state, pos, min_lz, &proof.pow_witness));
        challenger.observe_element(proof.pow_witness);
        F response = challenger.get_challenge();
        if (min_lz && (response >> (64 - min_lz))) throw Panic(GL_E_STATE, "fri_proof_of_work: invalid response");
    }
    // fri_prover_query_rounds: the challenger is only read here, so every x_index is drawn first and each tree
    // answers all rounds with one gather
    const uint32_t rounds = fp.config.num_query_rounds;
    std::vector<uint64_t> xs(rounds);
    for (auto& x : xs) x = challenger.get_challenge() % n;
    proof.query_round_proofs.resize(rounds);
    for (uint32_t q = 0; q < rounds; q++) proof.query_round_proofs[q].x_index = xs[q];
    for (const PolynomialBatch* o : oracles) {
        auto opened = o->open(xs);
        for (uint32_t q = 0; q < rounds; q++)
            proof.query_round_proofs[q].initial_trees_proof.emplace_back(std::move(opened.first[q]), std::move(opened.second[q]));
    }
    std::vector<uint64_t> idx = xs;
    for (auto& t : trees) {
        for (auto& x : idx) x >>= t.arity_bits;
        auto opened = detail::open_handle(c, t.h, 2u << t.arity_bits, t.lg_leaves - fp.config.cap_height, idx);
        for (uint32_t q = 0; q < rounds; q++)
            proof.query_round_proofs[q].steps.push_back({std::move(opened.first[q]), std::move(opened.second[q])});
        gl_commit_free(t.h);
    }
    return proof;
}

// plonky2::fri::oracle::PolynomialBatch::prove_openings(instance, oracles, challenger, fri_params)
inline FriProof prove_openings(const Context& c, const std::vector<FriBatchInfo>& instance,
                               const std::vector<const PolynomialBatch*>& oracles, Challenger& challenger, const FriParams& fp) {
    F alpha[2];
    challenger.get_extension_challenge(alpha);
    std::vector<gl_fri_batch> batches;
    std::vector<gl_fri_poly> polys;
    for (auto& b : instance) {
        gl_fri_batch gb;
        gb.point[0] = b.point[0];
        gb.point[1] = b.point[1];
        gb.first_poly = (uint32_t)polys.size();
        gb.num_polys = (uint32_t)b.polynomials.size();
        for (auto& pr : b.polynomials) polys.push_back({pr.first, pr.second});
        batches.push_back(gb);
    }
    std::vector<gl_commit*> handles;
    for (auto* o : oracles) handles.push_back(o->raw_handle());
    const uint64_t n = (1ull << oracles[0]->degree_log) << fp.config.rate_bits;
    detail::DevBuf coeffs(c, n * 16), values(c, n * 16);
    c.check(gl_fri_final_poly(c.raw(), handles.data(), (uint32_t)handles.size(), batches.data(), (uint32_t)batches.size(),
                              polys.data(), alpha, fp.config.rate_bits, coeffs.u64(), values.u64(), GL_DEVICE));
    return fri_proof_resident(c, oracles, coeffs.u64(), values.u64(), n, challenger, fp);
}

namespace detail {
// The FRI proof word stream of gl_fri_prove (field order of include/gl_b200.h), starting at flat[at] and running to the end
// of flat -> FriProof; widths: the leaf width of every initial oracle.
inline FriProof fri_proof_from_words(const std::vector<uint64_t>& flat, size_t at, const std::vector<uint32_t>& widths,
                                     const FriParams& fp) {
    FriProof proof;
    const uint32_t h = fp.config.cap_height, lgN = fp.degree_bits + fp.config.rate_bits;
    auto take_path = [&](uint32_t len) {
        MerkleProof mp;
        for (uint32_t l = 0; l < len; l++) {
            HashOut d;
            for (int e = 0; e < 4; e++) d.elements[e] = flat[at++];
            mp.siblings.push_back(d);
        }
        return mp;
    };
    uint32_t lg = lgN;
    for (uint32_t ab : fp.reduction_arity_bits) {
        MerkleCap cap(1ull << h);
        for (auto& d : cap)
            for (int e = 0; e < 4; e++) d.elements[e] = flat[at++];
        proof.commit_phase_merkle_caps.push_back(std::move(cap));
        lg -= ab;
    }
    const size_t final_words = (size_t)2 << (lg - fp.config.rate_bits);
    proof.final_poly.assign(flat.begin() + at, flat.begin() + at + final_words);
    at += final_words;
    proof.pow_witness = flat[at++];
    proof.query_round_proofs.resize(fp.config.num_query_rounds);
    for (auto& rnd : proof.query_round_proofs) {
        rnd.x_index = flat[at++];
        for (uint32_t w : widths) {
            std::vector<F> row(flat.begin() + at, flat.begin() + at + w);
            at += w;
            MerkleProof mp = take_path(lgN - h);
            rnd.initial_trees_proof.emplace_back(std::move(row), std::move(mp));
        }
        uint32_t cur = lgN;
        for (uint32_t ab : fp.reduction_arity_bits) {
            FriQueryStep st;
            st.evals.assign(flat.begin() + at, flat.begin() + at + ((size_t)2 << ab));
            at += (size_t)2 << ab;
            cur -= ab;
            st.merkle_proof = take_path(cur - h);
            rnd.steps.push_back(std::move(st));
        }
    }
    if (at != flat.size()) throw Panic(GL_E_STATE, "gl_fri_prove: proof stream of unexpected length");
    return proof;
}

inline gl_fri_params fri_params_c(const FriParams& fp, bool final_poly_times_x) {
    if (fp.reduction_arity_bits.size() > GL_FRI_MAX_LAYERS) throw Panic(GL_E_ARG, "too many FRI reduction layers");
    gl_fri_params prm;
    std::memset(&prm, 0, sizeof prm);
    prm.rate_bits = fp.config.rate_bits;
    prm.cap_height = fp.config.cap_height;
    prm.proof_of_work_bits = fp.config.proof_of_work_bits;
    prm.num_query_rounds = fp.config.num_query_rounds;
    prm.num_reduction_layers = (uint32_t)fp.reduction_arity_bits.size();
    for (size_t i = 0; i < fp.reduction_arity_bits.size(); i++) prm.reduction_arity_bits[i] = fp.reduction_arity_bits[i];
    prm.flags = final_poly_times_x ? GL_COMPAT_FRI_FINAL_POLY_TIMES_X : 0;
    return prm;
}
}  // namespace detail

// PolynomialBatch::prove_openings + fri_proof through ONE C-ABI call (gl_fri_prove): the Fiat-Shamir transcript runs on the
// device from `challenger`'s current state and comes back advanced past the proof; one copy brings the proof back.
// final_poly_times_x selects the fork form of upstream PR #436 (GL_COMPAT_FRI_FINAL_POLY_TIMES_X).
inline FriProof prove_openings_device(const Context& c, const std::vector<FriBatchInfo>& instance,
                                      const std::vector<const PolynomialBatch*>& oracles, Challenger& challenger,
                                      const FriParams& fp, bool final_poly_times_x = false) {
    if (fp.reduction_arity_bits.size() > GL_FRI_MAX_LAYERS) throw Panic(GL_E_ARG, "too many FRI reduction layers");
    std::vector<gl_fri_batch> batches;
    std::vector<gl_fri_poly> polys;
    for (auto& b : instance) {
        gl_fri_batch gb;
        gb.point[0] = b.point[0];
        gb.point[1] = b.point[1];
        gb.first_poly = (uint32_t)polys.size();
        gb.num_polys = (uint32_t)b.polynomials.size();
        for (auto& pr : b.polynomials) polys.push_back({pr.first, pr.second});
        batches.push_back(gb);
    }
    const gl_fri_params prm = detail::fri_params_c(fp, final_poly_times_x);
    gl_challenger ch;
    std::memset(&ch, 0, sizeof ch);
    for (int i = 0; i < 12; i++) ch.sponge_state[i] = challenger.sponge_state[i];
    ch.input_len = (uint32_t)challenger.input_buffer.size();
    ch.output_len = (uint32_t)challenger.output_buffer.size();
    for (uint32_t i = 0; i < ch.input_len; i++) ch.input_buffer[i] = challenger.input_buffer[i];
    for (uint32_t i = 0; i < ch.output_len; i++) ch.output_buffer[i] = challenger.output_buffer[i];
    std::vector<gl_commit*> handles;
    std::vector<uint32_t> widths;
    for (auto* o : oracles) {
        handles.push_back(o->raw_handle());
        widths.push_back(o->leaf_len);
    }
    uint64_t words = 0;
    c.check(gl_fri_proof_words(&prm, widths.data(), (uint32_t)widths.size(), fp.degree_bits, &words));
    std::vector<uint64_t> flat(words);
    c.check(gl_fri_prove(c.raw(), handles.data(), (uint32_t)handles.size(), batches.data(), (uint32_t)batches.size(), polys.data(),
                         &prm, &ch, flat.data(), words, &words));
    for (int i = 0; i < 12; i++) challenger.sponge_state[i] = ch.sponge_state[i];
    challenger.input_buffer.assign(ch.input_buffer, ch.input_buffer + ch.input_len);
    challenger.output_buffer.assign(ch.output_buffer, ch.output_buffer + ch.output_len);
    return detail::fri_proof_from_words(flat, 0, widths, fp);
}

// plonky2::plonk::prover compute_quotient_polys on the three resident prove-time oracles (gl_quotient_polys): returns
// quotient_polys.flat_map(|p| p.chunks(degree)), num_challenges * quotient_degree_factor coefficient vectors of 2^degree_bits.
inline std::vector<std::vector<F>> compute_quotient_polys(const Context& c, const gl_circuit& circuit, const std::vector<gl_gate>& gates,
                                                          const std::vector<F>& k_is, const PolynomialBatch& constants_sigmas,
                                                          const PolynomialBatch& wires, const PolynomialBatch& zs_partial_products,
                                                          const HashOut& public_inputs_hash, const std::vector<F>& betas,
                                                          const std::vector<F>& gammas, const std::vector<F>& alphas) {
    const size_t n = (size_t)1 << circuit.degree_bits, chunks = (size_t)circuit.num_challenges * circuit.quotient_degree_factor;
    std::vector<F> flat(chunks * n);
    c.check(gl_quotient_polys(c.raw(), &circuit, gates.data(), k_is.data(), constants_sigmas.raw_handle(), wires.raw_handle(),
                              zs_partial_products.raw_handle(), public_inputs_hash.elements, betas.data(), gammas.data(),
                              alphas.data(), flat.data(), GL_HOST));
    std::vector<std::vector<F>> out;
    for (size_t i = 0; i < chunks; i++) out.emplace_back(flat.begin() + i * n, flat.begin() + (i + 1) * n);
    return out;
}

// plonky2::plonk::prover all_wires_permutation_partial_products on the two resident commits (gl_permutation_zs): returns
// the num_challenges * ceil(num_routed_wires / quotient_degree_factor) columns of values on the subgroup (Z_0 .. Z_{nch-1},
// then the partial products of challenge 0, 1, ..) and, per challenge, the product of the row ratios over all rows
// (1 exactly when the witness satisfies every copy constraint).
struct PermutationZs {
    std::vector<std::vector<F>> zs_partial_products;
    std::vector<F> grand_products;
};
inline PermutationZs all_wires_permutation_partial_products(const Context& c, const gl_circuit& circuit, const std::vector<F>& k_is,
                                                            const PolynomialBatch& constants_sigmas, const PolynomialBatch& wires,
                                                            const std::vector<F>& betas, const std::vector<F>& gammas) {
    if (k_is.size() < circuit.num_routed_wires || betas.size() < circuit.num_challenges || gammas.size() < circuit.num_challenges)
        throw Panic(GL_E_ARG, "all_wires_permutation_partial_products: fewer k_is / betas / gammas than the circuit needs");
    const uint32_t deg = circuit.quotient_degree_factor ? circuit.quotient_degree_factor : 1;
    const size_t n = (size_t)1 << circuit.degree_bits;
    const size_t cols = (size_t)circuit.num_challenges * ((circuit.num_routed_wires + deg - 1) / deg);
    std::vector<F> flat(cols * n);
    PermutationZs out;
    out.grand_products.assign(circuit.num_challenges, 0);
    c.check(gl_permutation_zs(c.raw(), &circuit, k_is.data(), constants_sigmas.raw_handle(), wires.raw_handle(), betas.data(),
                              gammas.data(), flat.data(), GL_HOST, out.grand_products.data()));
    for (size_t i = 0; i < cols; i++) out.zs_partial_products.emplace_back(flat.begin() + i * n, flat.begin() + (i + 1) * n);
    return out;
}

// plonky2::plonk::prover::prove from the witness on, in one C-ABI call (gl_prove): ProofWithPublicInputs field by field.
// `words` is the stream gl_prove returns (caps, OpeningSet, FRI proof); the other fields are views of it.
struct ProofWithPublicInputs {
    MerkleCap wires_cap, plonk_zs_partial_products_cap, quotient_polys_cap;
    // OpeningSet in declaration order: constants, plonk_sigmas, wires, plonk_zs, plonk_zs_next, partial_products,
    // quotient_polys; each entry (a0, a1)
    std::vector<std::vector<std::array<F, 2>>> openings;
    FriProof opening_proof;
    std::vector<F> public_inputs;
    std::vector<uint64_t> words;
};
// wires: num_wires columns of 2^degree_bits values (the witness); constants_sigmas: the resident prover-data commit.
inline ProofWithPublicInputs prove(const Context& c, const gl_circuit& circuit, const std::vector<gl_gate>& gates,
                                   const std::vector<F>& k_is, const PolynomialBatch& constants_sigmas, const HashOut& circuit_digest,
                                   const FriParams& fp, const std::vector<std::vector<F>>& wires, const std::vector<F>& public_inputs,
                                   bool final_poly_times_x = false) {
    if (k_is.size() < circuit.num_routed_wires || gates.size() < circuit.num_gates || wires.size() != circuit.num_wires)
        throw Panic(GL_E_ARG, "prove: fewer k_is than num_routed_wires or gates than num_gates, or a witness without num_wires columns");
    for (auto& w : wires)   // the library reads 2^degree_bits values of every column and cannot check the caller's sizes
        if (w.size() != ((size_t)1 << circuit.degree_bits)) throw Panic(GL_E_ARG, "prove: a witness column without 2^degree_bits values");
    const gl_fri_params prm = detail::fri_params_c(fp, final_poly_times_x);
    std::vector<const uint64_t*> cols;
    for (auto& w : wires) cols.push_back(w.data());
    ProofWithPublicInputs out;
    uint64_t words = 0;
    gl_prove(c.raw(), &circuit, gates.data(), k_is.data(), constants_sigmas.raw_handle(), circuit_digest.elements, &prm, nullptr,
             cols.data(), GL_HOST, public_inputs.data(), (uint32_t)public_inputs.size(), nullptr, 0, &words);   // size only
    out.words.resize(words);
    c.check(gl_prove(c.raw(), &circuit, gates.data(), k_is.data(), constants_sigmas.raw_handle(), circuit_digest.elements, &prm,
                     nullptr, cols.data(), GL_HOST, public_inputs.data(), (uint32_t)public_inputs.size(), out.words.data(), words,
                     &words));
    size_t at = 0;
    const size_t cap_len = (size_t)1 << fp.config.cap_height;
    for (MerkleCap* cap : {&out.wires_cap, &out.plonk_zs_partial_products_cap, &out.quotient_polys_cap}) {
        cap->resize(cap_len);
        for (auto& d : *cap)
            for (int e = 0; e < 4; e++) d.elements[e] = out.words[at++];
    }
    const uint32_t nch = circuit.num_challenges, qdf = circuit.quotient_degree_factor;
    const uint32_t zcols = nch * ((circuit.num_routed_wires + qdf - 1) / qdf);
    for (uint32_t k : {circuit.num_constants, circuit.num_routed_wires, circuit.num_wires, nch, nch, zcols - nch, nch * qdf}) {
        std::vector<std::array<F, 2>> field(k);
        for (auto& v : field) {
            v[0] = out.words[at++];
            v[1] = out.words[at++];
        }
        out.openings.push_back(std::move(field));
    }
    const std::vector<uint32_t> widths = {constants_sigmas.leaf_len, circuit.num_wires, zcols, nch * qdf};
    out.opening_proof = detail::fri_proof_from_words(out.words, at, widths, fp);
    out.public_inputs = public_inputs;
    return out;
}

// One commit sharded over the GPUs of a box (gl_group_*: NCCL behind the C ABI); this process holds every rank.
class Group {
   public:
    explicit Group(const std::vector<const Context*>& ctxs) : ctxs_(ctxs) {
        std::vector<gl_ctx*> raw;
        for (auto* c : ctxs) raw.push_back(c->raw());
        int rc = gl_group_create(raw.data(), (uint32_t)raw.size(), 0, (uint32_t)raw.size(), nullptr, &g_);
        if (rc) throw Panic(rc, gl_last_error(nullptr));
    }
    ~Group() { gl_group_destroy(g_); }
    Group(const Group&) = delete;
    Group& operator=(const Group&) = delete;
    void check(int rc) const {
        if (rc) throw Panic(rc, gl_group_last_error(g_));
    }
    struct Sharded {   // the local shards of one PolynomialBatch + the whole cap
        std::vector<gl_commit*> handles;
        MerkleCap cap;
        std::vector<F> coefficients;   // [c][n]: every rank writes its polynomials into the one array
        uint32_t c = 0, degree_log = 0, rate_bits = 0, cap_height = 0, leaf_len = 0;
    };
    // values: [c][n] contiguous host array shared by the ranks
    Sharded commit_from_values(const std::vector<F>& values, uint32_t c, uint32_t log_n, uint32_t rate_bits, uint32_t cap_height,
                               uint32_t flags = 0) {
        const size_t nl = ctxs_.size();
        Sharded s;
        s.c = c; s.degree_log = log_n; s.rate_bits = rate_bits; s.cap_height = cap_height;
        s.leaf_len = c + ((flags & GL_COMMIT_BLINDING) ? GL_SALT_SIZE : 0);
        s.coefficients.resize(values.size());
        s.handles.assign(nl, nullptr);
        std::vector<std::vector<F>> caps(nl, std::vector<F>((size_t)4 << cap_height));
        std::vector<const uint64_t*> in(nl, values.data());
        std::vector<uint64_t*> co(nl, s.coefficients.data()), cp;
        for (auto& v : caps) cp.push_back(v.data());
        check(gl_group_commit_from_values(g_, in.data(), log_n, c, rate_bits, cap_height, co.data(), cp.data(), s.handles.data(),
                                          GL_HOST, flags));
        s.cap.resize(1ull << cap_height);
        for (size_t i = 0; i < s.cap.size(); i++)
            for (int e = 0; e < 4; e++) s.cap[i].elements[e] = caps[0][4 * i + e];
        return s;
    }
    // rows [k][leaf_len] and paths [k][L][4] for GLOBAL leaf indices, whoever owns them
    void open(const Sharded& s, const std::vector<uint64_t>& idx, std::vector<F>* rows, std::vector<F>* paths) {
        const size_t nl = ctxs_.size(), k = idx.size(), L = s.degree_log + s.rate_bits - s.cap_height;
        std::vector<std::vector<F>> r(nl, std::vector<F>(k * s.leaf_len)), p(nl, std::vector<F>(k * L * 4 + 4));
        std::vector<uint64_t*> rp, pp;
        for (size_t i = 0; i < nl; i++) {
            rp.push_back(r[i].data());
            pp.push_back(p[i].data());
        }
        check(gl_group_commit_open(g_, s.handles.data(), idx.data(), (uint32_t)k, rp.data(), pp.data(), GL_HOST));
        if (rows) *rows = r[0];
        if (paths) {
            p[0].resize(k * L * 4);
            *paths = p[0];
        }
    }
    static void free(Sharded& s) {
        for (auto* h : s.handles)
            if (h) gl_commit_free(h);
        s.handles.clear();
    }

   private:
    std::vector<const Context*> ctxs_;
    gl_group* g_ = nullptr;
};

}  // namespace plonky2_b200
