// Poseidon batch / Merkle / SMT kernels (SURVEY 2c K4, K5, K8; 8a rows P4-P7, P10).
//
// Every kernel is "one Poseidon state per thread": the work is issue bound (about 1.7*10^4 SASS
// instructions per permutation, a third of them DFMA, against at most 1.1 KB of traffic per leaf), so the
// only memory rule that matters is that a warp's loads coalesce -- leaves are therefore kept
// COLUMN-major on the device ([column][leaf]) so that 32 consecutive leaves read 256 contiguous bytes
// per column.  Each kernel has ONE inlined permutation site (a second copy of the 33 KB round code
// pushes a kernel out of the instruction cache); kernels with several hash sites call it out of line.
#include <cuda_runtime.h>

#include "hash_kernels.h"
#include "poseidon.cuh"
#include "poseidon_constants.h"

#define HASH_BLOCK 128
#ifndef HASH_MIN_CTAS
#define HASH_MIN_CTAS 5   // 94 registers, no spills: 1.549 G permutations/s against 1.530 at 4 (tools/poseidon_bench, profiles/README.md)
#endif

int gl_poseidon_upload_constants(const u64* rc360) {
    cudaError_t e = cudaMemcpyToSymbol(c_poseidon_rc, rc360, sizeof(u64) * POSEIDON_ROUNDS * POSEIDON_WIDTH);
    if (e != cudaSuccess) return (int)e;
    // bit patterns of the constants the FP64 linear layers add (poseidon_constants.h: linear_layer_tables)
    static u64 split[(POSEIDON_ROUNDS + 1) * POSEIDON_WIDTH * 2];
    static u64 pk[(POSEIDON_PARTIAL / 2) * POSEIDON_WIDTH * 2];
    static const int circ[12] = {17, 15, 41, 16, 2, 28, 13, 13, 39, 18, 34, 20};
    poseidon_constants::linear_layer_tables(rc360, circ, 8, true, split, pk, POSEIDON_HANDOFF_BIAS);
    e = cudaMemcpyToSymbol(c_poseidon_rc_split, split, sizeof(split));
    if (e != cudaSuccess) return (int)e;
    return (int)cudaMemcpyToSymbol(c_poseidon_pair_k, pk, sizeof(pk));
}

// ---- position of node q of layer i inside one subtree's digest buffer (plonky2 in-order layout) ----
// MerkleTree::prove: sibling of (pair, parity) at layer i sits at 2*((pair << (i+1)) + 2^i - 1) + (1 - parity)
GL_D u64 digest_pos(unsigned layer, u64 q) {
    u64 pair = q >> 1, parity = q & 1;
    return 2 * ((pair << (layer + 1)) + ((u64)1 << layer) - 1) + parity;
}

GL_D void store_digest(u64* dst, const u64 d[4]) {
    ulonglong2* p = reinterpret_cast<ulonglong2*>(dst);
    p[0] = make_ulonglong2(d[0], d[1]);
    p[1] = make_ulonglong2(d[2], d[3]);
}
GL_D void load_digest(const u64* src, u64 d[4]) {
    const ulonglong2* p = reinterpret_cast<const ulonglong2*>(src);
    ulonglong2 a = p[0], b = p[1];
    d[0] = a.x; d[1] = a.y; d[2] = b.x; d[3] = b.y;
}

// ------------------------------------------------------------------------------------------------
// Poseidon batch entry points (P5, P6)
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(HASH_BLOCK, HASH_MIN_CTAS) k_permute_batch(u64* states, u64 m) {
    u64 i = blockIdx.x * (u64)HASH_BLOCK + threadIdx.x;
    if (i >= m) return;
    ulonglong2* p = reinterpret_cast<ulonglong2*>(states + 12 * i);
    u64 s[12];
#pragma unroll
    for (int k = 0; k < 6; k++) {
        ulonglong2 v = p[k];
        s[2 * k] = v.x;
        s[2 * k + 1] = v.y;
    }
    poseidon_permute(s);
#pragma unroll
    for (int k = 0; k < 6; k++) p[k] = make_ulonglong2(gl_canon(s[2 * k]), gl_canon(s[2 * k + 1]));
}

__global__ void __launch_bounds__(HASH_BLOCK, HASH_MIN_CTAS)
k_two_to_one_batch(const u64* __restrict__ l, const u64* __restrict__ r, u64* __restrict__ out, u64 m) {
    u64 i = blockIdx.x * (u64)HASH_BLOCK + threadIdx.x;
    if (i >= m) return;
    u64 a[4], b[4], d[4];
    load_digest(l + 4 * i, a);
    load_digest(r + 4 * i, b);
    poseidon_two_to_one(a, b, d);
    store_digest(out + 4 * i, d);
}

// hash_no_pad over m rows of `len` elements each, row-major input ([m][len]).
__global__ void __launch_bounds__(HASH_BLOCK, HASH_MIN_CTAS)
k_hash_no_pad_rows(const u64* __restrict__ in, u32 len, u64 m, u64* __restrict__ out) {
    u64 i = blockIdx.x * (u64)HASH_BLOCK + threadIdx.x;
    if (i >= m) return;
    const u64* row = in + (u64)len * i;
    u64 s[12];
#pragma unroll
    for (int k = 0; k < 12; k++) s[k] = 0;
    for (u32 off = 0; off < len; off += 8) {
        u32 k = len - off < 8 ? len - off : 8;
#pragma unroll
        for (int j = 0; j < 8; j++)
            if (j < k) s[j] = __ldg(row + off + j);
        poseidon_permute(s);
    }
    u64 d[4];
#pragma unroll
    for (int j = 0; j < 4; j++) d[j] = gl_canon(s[j]);
    store_digest(out + 4 * i, d);
}

// PoseidonNodeHash::calc_node_hash(Node::Leaf(k, v)) = hash_no_pad([k, v, 1, 1, 0, 1])
// (src/smt/goldilocks_poseidon/mod.rs:167-181 == src/smt/gadgets/common.rs:87-101): two permutations
GL_D void smt_leaf_hash(const u64 k[4], const u64 v[4], u64 out[4]) {
    u64 s[12];
#pragma unroll
    for (int i = 0; i < 4; i++) {
        s[i] = k[i];
        s[4 + i] = v[i];
        s[8 + i] = 0;
    }
#pragma unroll 1
    for (int chunk = 0; chunk < 2; chunk++) {
        if (chunk) { s[0] = 1; s[1] = 1; s[2] = 0; s[3] = 1; }  // second chunk overwrites lanes 0..3 only
        poseidon_permute(s);
    }
#pragma unroll
    for (int i = 0; i < 4; i++) out[i] = gl_canon(s[i]);
}

__global__ void __launch_bounds__(HASH_BLOCK, HASH_MIN_CTAS)
k_smt_leaf_hash_batch(const u64* __restrict__ keys, const u64* __restrict__ values, u64* __restrict__ out, u64 m) {
    u64 i = blockIdx.x * (u64)HASH_BLOCK + threadIdx.x;
    if (i >= m) return;
    u64 k[4], v[4], d[4];
    load_digest(keys + 4 * i, k);
    load_digest(values + 4 * i, v);
    smt_leaf_hash(k, v, d);
    store_digest(out + 4 * i, d);
}

// ------------------------------------------------------------------------------------------------
// Merkle tree (P4): leaf layer + one kernel per level, writing plonky2's digest layout directly
// ------------------------------------------------------------------------------------------------
// Destination of the digest of leaf / node q of `layer` when every subtree has 2^sub_bits leaves.
// layer == sub_bits means "subtree root" -> cap entry.
GL_D u64* node_slot(u64* digests, u64* cap, unsigned sub_bits, unsigned layer, u64 global_q) {
    unsigned span = sub_bits - layer;                 // log2(nodes of this layer per subtree)
    u64 subtree = global_q >> span;
    u64 q = global_q & (((u64)1 << span) - 1);
    if (layer == sub_bits) return cap + 4 * subtree;
    u64 per_subtree = 2 * (((u64)1 << sub_bits) - 1);  // digests per subtree
    return digests + 4 * (subtree * per_subtree + digest_pos(layer, q));
}

// leaves column-major: element (leaf i, column j) at lde[j * ld + i]
__global__ void __launch_bounds__(HASH_BLOCK, HASH_MIN_CTAS)
k_leaf_hash_cols(const u64* __restrict__ lde, u64 ld, u32 c, u64 num_leaves, unsigned sub_bits,
                 u64* __restrict__ digests, u64* __restrict__ cap) {
    u64 i = blockIdx.x * (u64)HASH_BLOCK + threadIdx.x;
    if (i >= num_leaves) return;
    u64 d[4];
    if (c <= 4) {  // hash_or_noop: zero padded copy
#pragma unroll
        for (int j = 0; j < 4; j++) d[j] = j < c ? gl_canon(lde[(u64)j * ld + i]) : 0;
    } else {
        u64 s[12];
#pragma unroll
        for (int k = 0; k < 12; k++) s[k] = 0;
        const u64* p = lde + i;
        // one call site for the permutation (a second inlined copy pushes the kernel past the instruction
        // cache): the ragged last chunk is handled by predicated loads
        const u32 chunks = (c + 7) / 8;
#pragma unroll 1
        for (u32 ch = 0; ch < chunks; ch++, p += 8 * ld) {
            const u32 k = c - 8 * ch;   // elements left (>= 1)
#pragma unroll
            for (int j = 0; j < 8; j++)
                if (j < k) s[j] = p[(u64)j * ld];
            poseidon_permute(s);
        }
#pragma unroll
        for (int j = 0; j < 4; j++) d[j] = gl_canon(s[j]);
    }
    store_digest(node_slot(digests, cap, sub_bits, 0, i), d);
}

// The same sponge fed in column blocks as they arrive (gl_commit_add_coeffs with GL_COMMIT_STREAM_HASH): absorbs the
// 8-column groups of [col_begin, col_end) into the per-leaf sponge state (state[k * num_leaves + i], k < 12), so the
// hashing of the polynomials that are already extended overlaps the arrival of the next ones.  col_begin is a multiple
// of 8; col_end is a multiple of 8 or c; `first` starts from the zero state, `last` (col_end == c) writes the digests.
__global__ void __launch_bounds__(HASH_BLOCK, HASH_MIN_CTAS)
k_leaf_absorb_cols(const u64* __restrict__ lde, u64 ld, u32 col_begin, u32 col_end, u64 num_leaves, unsigned sub_bits,
                   u64* __restrict__ state, int first, int last, u64* __restrict__ digests, u64* __restrict__ cap) {
    u64 i = blockIdx.x * (u64)HASH_BLOCK + threadIdx.x;
    if (i >= num_leaves) return;
    u64 s[12];
#pragma unroll
    for (int k = 0; k < 12; k++) s[k] = first ? 0 : state[(u64)k * num_leaves + i];
    const u64* col = lde + i + (u64)col_begin * ld;
#pragma unroll 1
    for (u32 off = col_begin; off < col_end; off += 8, col += 8 * ld) {
        const u32 k = col_end - off < 8 ? col_end - off : 8;
#pragma unroll
        for (int j = 0; j < 8; j++)
            if (j < k) s[j] = col[(u64)j * ld];
        poseidon_permute(s);
    }
    if (last) {
        u64 d[4];
#pragma unroll
        for (int j = 0; j < 4; j++) d[j] = gl_canon(s[j]);
        store_digest(node_slot(digests, cap, sub_bits, 0, i), d);
    } else {
#pragma unroll
        for (int k = 0; k < 12; k++) state[(u64)k * num_leaves + i] = s[k];
    }
}

// leaves row-major ([num_leaves][leaf_len]) -- MerkleTree::new(leaves: Vec<Vec<F>>, cap_height)
__global__ void __launch_bounds__(HASH_BLOCK, HASH_MIN_CTAS)
k_leaf_hash_rows(const u64* __restrict__ leaves, u32 leaf_len, u64 num_leaves, unsigned sub_bits,
                 u64* __restrict__ digests, u64* __restrict__ cap) {
    u64 i = blockIdx.x * (u64)HASH_BLOCK + threadIdx.x;
    if (i >= num_leaves) return;
    const u64* row = leaves + (u64)leaf_len * i;
    u64 d[4];
    if (leaf_len <= 4) {
#pragma unroll
        for (int j = 0; j < 4; j++) d[j] = j < leaf_len ? gl_canon(row[j]) : 0;
    } else {
        u64 s[12];
#pragma unroll
        for (int k = 0; k < 12; k++) s[k] = 0;
        for (u32 off = 0; off < leaf_len; off += 8) {
            u32 k = leaf_len - off < 8 ? leaf_len - off : 8;
#pragma unroll
            for (int j = 0; j < 8; j++)
                if (j < k) s[j] = __ldg(row + off + j);
            poseidon_permute(s);
        }
#pragma unroll
        for (int j = 0; j < 4; j++) d[j] = gl_canon(s[j]);
    }
    store_digest(node_slot(digests, cap, sub_bits, 0, i), d);
}

// layer >= 1: node q = two_to_one(children 2q, 2q+1 of layer-1); children are adjacent in the layout
__global__ void __launch_bounds__(HASH_BLOCK, HASH_MIN_CTAS)
k_merkle_level(u64* __restrict__ digests, u64* __restrict__ cap, unsigned sub_bits, unsigned layer, u64 num_nodes) {
    u64 g = blockIdx.x * (u64)HASH_BLOCK + threadIdx.x;
    if (g >= num_nodes) return;
    const u64* child = node_slot(digests, cap, sub_bits, layer - 1, 2 * g);
    u64 a[4], b[4], d[4];
    load_digest(child, a);
    load_digest(child + 4, b);
    poseidon_two_to_one(a, b, d);
    store_digest(node_slot(digests, cap, sub_bits, layer, g), d);
}

// ------------------------------------------------------------------------------------------------
// P10 fri_proof_of_work: candidates start .. start+count; atomicMin keeps the smallest hit
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(HASH_BLOCK, HASH_MIN_CTAS)
k_pow_grind(const u64* __restrict__ state12, unsigned pos, unsigned out_pos, unsigned min_lz, u64 start,
            u64 count, unsigned long long* __restrict__ best) {
    u64 k = blockIdx.x * (u64)HASH_BLOCK + threadIdx.x;
    if (k >= count) return;
    u64 cand = start + k;
    u64 s[12];
#pragma unroll
    for (int j = 0; j < 12; j++) s[j] = state12[j];
#pragma unroll
    for (int j = 0; j < 12; j++)
        if (j == (int)pos) s[j] = cand;
    poseidon_permute(s);
    u64 resp = 0;
#pragma unroll
    for (int j = 0; j < 12; j++)
        if (j == (int)out_pos) resp = gl_canon(s[j]);
    unsigned lz = resp ? (unsigned)__clzll((long long)resp) : 64u;
    if (lz >= min_lz) atomicMin(best, (unsigned long long)cand);
}

// ------------------------------------------------------------------------------------------------
// P7 verify_smt_process_proof over a batch (src/smt/proof/process.rs:153-337): one proof per thread,
// 256 levels x 2 compressions + 2 leaf hashes = 516 permutations, no divergence in the hash count.
// ------------------------------------------------------------------------------------------------
// Out-of-line permutation for kernels with several hash sites (one copy of the 33 KB round code; the state
// travels through local memory, 24 accesses against ~17k instructions).
__device__ __noinline__ void poseidon_permute_call(u64* state) {
    u64 s[12];
#pragma unroll
    for (int i = 0; i < 12; i++) s[i] = state[i];
    poseidon_permute(s);
#pragma unroll
    for (int i = 0; i < 12; i++) state[i] = s[i];
}

// Challenger::duplexing x m: a serial chain, one thread
__global__ void __launch_bounds__(32) k_duplex_chain(u64* __restrict__ state, const u64* __restrict__ chunks, u64 m) {
    if (threadIdx.x) return;
    u64 s[12];
#pragma unroll
    for (int k = 0; k < 12; k++) s[k] = state[k];
    for (u64 i = 0; i < m; i++) {
#pragma unroll
        for (int k = 0; k < 8; k++) s[k] = chunks[8 * i + k];
        poseidon_permute_call(s);
#pragma unroll
        for (int k = 0; k < 12; k++) s[k] = gl_canon(s[k]);
    }
#pragma unroll
    for (int k = 0; k < 12; k++) state[k] = s[k];
}

// plonky2::iop::challenger::Challenger resident on the device (gl_fri_prove: the Fiat-Shamir transcript never leaves HBM).
// One thread: observe `n_obs` elements read from device memory (observe_element semantics: outputs invalidated, duplexing
// when the rate is full), then pop `n_squeeze` challenges (duplexing first when inputs are pending or no output is left).
GL_D void challenger_duplex(gl_challenger* ch) {
    u64 s[12];
#pragma unroll
    for (int k = 0; k < 12; k++) s[k] = ch->sponge_state[k];
    for (u32 k = 0; k < ch->input_len; k++) s[k] = ch->input_buffer[k];
    ch->input_len = 0;
    poseidon_permute_call(s);
#pragma unroll
    for (int k = 0; k < 12; k++) ch->sponge_state[k] = gl_canon(s[k]);
#pragma unroll
    for (int k = 0; k < 8; k++) ch->output_buffer[k] = ch->sponge_state[k];
    ch->output_len = 8;
}
__global__ void __launch_bounds__(32)
k_challenger_step(gl_challenger* __restrict__ ch, const u64* __restrict__ observe, u32 n_obs, u64* __restrict__ squeeze, u32 n_squeeze,
                  u64* __restrict__ pow_state) {
    if (threadIdx.x) return;
    for (u32 i = 0; i < n_obs; i++) {
        ch->output_len = 0;
        ch->input_buffer[ch->input_len++] = gl_canon(observe[i]);
        if (ch->input_len == 8) challenger_duplex(ch);
    }
    for (u32 i = 0; i < n_squeeze; i++) {
        if (ch->input_len || ch->output_len == 0) challenger_duplex(ch);
        squeeze[i] = ch->output_buffer[--ch->output_len];
    }
    if (pow_state) {   // fri_proof_of_work: the duplex state the witness is absorbed into (input buffer applied)
        for (int k = 0; k < 12; k++) pow_state[k] = (u32)k < ch->input_len ? ch->input_buffer[k] : ch->sponge_state[k];
    }
}
void launch_challenger_step(gl_challenger* ch, const u64* observe, u32 n_obs, u64* squeeze, u32 n_squeeze, u64* pow_state,
                            cudaStream_t st) {
    k_challenger_step<<<1, 32, 0, st>>>(ch, observe, n_obs, squeeze, n_squeeze, pow_state);
    ++g_gl_launches;
}

GL_D void two_to_one_call(const u64 l[4], const u64 r[4], u64 out[4]) {
    u64 s[12];
#pragma unroll
    for (int i = 0; i < 4; i++) { s[i] = l[i]; s[4 + i] = r[i]; s[8 + i] = 0; }
    poseidon_permute_call(s);
#pragma unroll
    for (int i = 0; i < 4; i++) out[i] = gl_canon(s[i]);
}
GL_D void smt_leaf_hash_call(const u64 k[4], const u64 v[4], u64 out[4]) {
    u64 s[12];
#pragma unroll
    for (int i = 0; i < 4; i++) { s[i] = k[i]; s[4 + i] = v[i]; s[8 + i] = 0; }
    poseidon_permute_call(s);
    s[0] = 1; s[1] = 1; s[2] = 0; s[3] = 1;
    poseidon_permute_call(s);
#pragma unroll
    for (int i = 0; i < 4; i++) out[i] = gl_canon(s[i]);
}

// verify_merkle_proof_to_cap over a batch (plonky2::hash::merkle_proofs; the verifier's side of P11): one proof per
// thread -- hash_or_noop of the leaf row, then the sibling path up to the cap entry the index ends in.
__global__ void __launch_bounds__(128)
k_merkle_verify_batch(const u64* __restrict__ leaves, u32 leaf_len, const u64* __restrict__ leaf_indices,
                      const u64* __restrict__ paths, u32 path_len, const u64* __restrict__ cap, u32 cap_height, u64 k,
                      int* __restrict__ ok) {
    u64 t = blockIdx.x * (u64)blockDim.x + threadIdx.x;
    if (t >= k) return;
    const u64* row = leaves + (u64)leaf_len * t;
    u64 d[4];
    if (leaf_len <= 4) {
#pragma unroll
        for (int j = 0; j < 4; j++) d[j] = j < leaf_len ? gl_canon(row[j]) : 0;
    } else {
        u64 s[12];
#pragma unroll
        for (int j = 0; j < 12; j++) s[j] = 0;
        for (u32 off = 0; off < leaf_len; off += 8) {
            const u32 n = leaf_len - off < 8 ? leaf_len - off : 8;
#pragma unroll
            for (int j = 0; j < 8; j++)
                if (j < n) s[j] = row[off + j];
            poseidon_permute_call(s);
        }
#pragma unroll
        for (int j = 0; j < 4; j++) d[j] = gl_canon(s[j]);
    }
    u64 idx = leaf_indices[t];
    const u64* sib = paths + (u64)t * path_len * 4;
    for (u32 l = 0; l < path_len; l++, sib += 4, idx >>= 1) {
        u64 sb[4], nd[4];
        load_digest(sib, sb);
        if (idx & 1) two_to_one_call(sb, d, nd);
        else two_to_one_call(d, sb, nd);
#pragma unroll
        for (int j = 0; j < 4; j++) d[j] = nd[j];
    }
    int good = idx < ((u64)1 << cap_height);
    if (good) {
        const u64* c = cap + 4 * idx;
#pragma unroll
        for (int j = 0; j < 4; j++) good &= d[j] == gl_canon(c[j]);
    }
    ok[t] = good;
}

enum { ST_TOP = 0, ST_BOT = 1, ST_OLD0 = 2, ST_NEW1 = 3, ST_UPD = 4, ST_NA = 5 };

GL_D void load_digest_canon(const u64* src, u64 d[4]) {
    load_digest(src, d);
#pragma unroll
    for (int j = 0; j < 4; j++) d[j] = gl_canon(d[j]);
}
GL_D bool is_zero4(const u64 h[4]) { return (h[0] | h[1] | h[2] | h[3]) == 0; }
GL_D bool eq4(const u64 a[4], const u64 b[4]) {
    return a[0] == b[0] && a[1] == b[1] && a[2] == b[2] && a[3] == b[3];
}
GL_D int key_bit(const u64 k[4], unsigned i) {
    u64 w = (i >> 6) == 0 ? k[0] : (i >> 6) == 1 ? k[1] : (i >> 6) == 2 ? k[2] : k[3];
    return (int)((w >> (i & 63)) & 1);
}
GL_D void sel4(u64 dst[4], const u64 a[4], bool take_a, const u64 b[4]) {
#pragma unroll
    for (int j = 0; j < 4; j++) dst[j] = take_a ? a[j] : b[j];
}

__global__ void __launch_bounds__(128)
k_smt_verify_process(const gl_smt_proof_hdr* __restrict__ proofs, const u64* __restrict__ sib_pool,
                     const u64* __restrict__ sib_off, u64 m, int* __restrict__ status) {
    u64 t = blockIdx.x * (u64)blockDim.x + threadIdx.x;
    if (t >= m) return;
    const gl_smt_proof_hdr* pf = proofs + t;
    const u64* sibs = sib_pool + 4 * sib_off[t];
    const int LEVELS = 256;
    u32 fnc = pf->fnc;
    bool enabled = fnc != 0;
    bool flip = fnc == 3;  // a remove proof is an insert proof with old and new flipped
    if (flip) fnc = 2;
    u64 old_key[4], old_value[4], old_root[4], new_key[4], new_value[4], new_root[4];
#pragma unroll
    for (int j = 0; j < 4; j++) {
        // every header word is a field element: the reference reads key bits through HashOut::to_bytes (canonical,
        // src/smt/proof/process.rs:193-203) and compares roots / keys / values as field elements, so any u64 is taken mod p
        old_key[j] = gl_canon(flip ? pf->new_key[j] : pf->old_key[j]);
        old_value[j] = gl_canon(flip ? pf->new_value[j] : pf->old_value[j]);
        old_root[j] = gl_canon(flip ? pf->new_root[j] : pf->old_root[j]);
        new_key[j] = gl_canon(flip ? pf->old_key[j] : pf->new_key[j]);
        new_value[j] = gl_canon(flip ? pf->old_value[j] : pf->new_value[j]);
        new_root[j] = gl_canon(flip ? pf->old_root[j] : pf->new_root[j]);
    }
    u64 ns64 = sib_off[t + 1] - sib_off[t];
    if (ns64 >= (u64)LEVELS) { status[t] = 1; return; }   // assert!(siblings.len() < n2b_new.len())
    u32 ns = (u32)ns64;
    // siblings.resize(256, default): levels >= ns have an all-zero sibling
    // smt_lev_ins: the deepest level whose PARENT level has a non-zero sibling (root's parent counts)
    // scan from the bottom: first i (descending) with sibling[i-1] != 0, or 0 if none
    int ins_level = 0;
    for (int i = (int)ns; i >= 1; i--) {
        u64 sb[4];
        load_digest_canon(sibs + 4 * (i - 1), sb);
        if (!is_zero4(sb)) { ins_level = i; break; }
    }
    // assert!(is_zeros.last()) cannot fire: ns < 256, so level 255 holds a padded zero
    // state machine, top to bottom; remember the state of every level in 3 bits (packed)
    // levels above ins_level: lev_ins = 0 -> stay Top; at ins_level: transition; below: Bottom/NewOne/Na chain
    // We need sm[i] while walking bottom-up, so store them: 256 x 3 bits = 24 u32.
    u32 smw[26];
#pragma unroll
    for (int j = 0; j < 26; j++) smw[j] = 0;
    int prev = enabled ? ST_TOP : ST_NA;
    bool ins_or_rem = fnc == 2;
    bool is_old0 = pf->is_old0 != 0;
    // calc_old_new_root (src/smt/proof/process.rs:260-337) hashes twice at each of the 256 levels, but a level in
    // state Na passes zeros on, old_hash is read only in state Top and new_hash only in Top / Bottom / NewOne: the
    // discarded hashes are not computed here.  `last` = deepest level that is not Na (everything below it yields
    // prev_old = prev_new = 0); the leaf hashes are computed only if some level reads them.
    int last = -1;
    bool need_old1 = false, need_new1 = false;
    for (int i = 0; i < LEVELS; i++) {
        int diff = key_bit(old_key, i) ^ key_bit(new_key, i);
        bool lev_ins = (i == ins_level);
        int st;
        if (prev == ST_TOP) {
            if (!lev_ins) st = ST_TOP;
            else if (!ins_or_rem) st = ST_UPD;
            else if (is_old0) st = ST_OLD0;
            else st = diff ? ST_NEW1 : ST_BOT;
        } else if (prev == ST_BOT) {
            st = diff ? ST_NEW1 : ST_BOT;
        } else {
            st = ST_NA;
        }
        smw[i / 10] |= (u32)st << (3 * (i % 10));
        prev = st;
        if (st != ST_NA) last = i;
        need_old1 |= st == ST_BOT || st == ST_NEW1 || st == ST_UPD;
        need_new1 |= st == ST_NEW1 || st == ST_OLD0 || st == ST_UPD;
    }
    if (prev == ST_TOP || prev == ST_BOT) { status[t] = 3; return; }
    u64 old1_leaf[4] = {0, 0, 0, 0}, new1_leaf[4] = {0, 0, 0, 0};
    if (need_old1) smt_leaf_hash_call(old_key, old_value, old1_leaf);
    if (need_new1) smt_leaf_hash_call(new_key, new_value, new1_leaf);
    u64 prev_old[4] = {0, 0, 0, 0}, prev_new[4] = {0, 0, 0, 0};
    const u64 zero[4] = {0, 0, 0, 0};
#pragma unroll 1
    for (int i = last; i >= 0; i--) {
        int st = (int)((smw[i / 10] >> (3 * (i % 10))) & 7u);
        bool pos = key_bit(new_key, i) != 0;
        u64 sb[4];
        if ((u32)i < ns) load_digest_canon(sibs + 4 * i, sb);
        else { sb[0] = sb[1] = sb[2] = sb[3] = 0; }
        u64 l[4], r[4], old_hash[4] = {0, 0, 0, 0}, new_hash[4] = {0, 0, 0, 0};
        if (st == ST_TOP) {
            sel4(l, sb, pos, prev_old);
            sel4(r, prev_old, pos, sb);
            two_to_one_call(l, r, old_hash);
        }
        u64 n_left[4], n_right[4];
#pragma unroll
        for (int j = 0; j < 4; j++) {
            n_left[j] = (st == ST_TOP || st == ST_BOT) ? prev_new[j] : (st == ST_NEW1 ? new1_leaf[j] : 0);
            n_right[j] = st == ST_TOP ? sb[j] : (st == ST_NEW1 ? old1_leaf[j] : 0);
        }
        if (st == ST_TOP || st == ST_BOT || st == ST_NEW1) {
            sel4(l, n_right, pos, n_left);
            sel4(r, n_left, pos, n_right);
            two_to_one_call(l, r, new_hash);
        }
#pragma unroll
        for (int j = 0; j < 4; j++) {
            prev_old[j] = st == ST_TOP ? old_hash[j]
                          : (st == ST_BOT || st == ST_NEW1 || st == ST_UPD) ? old1_leaf[j] : zero[j];
            prev_new[j] = (st == ST_TOP || st == ST_BOT || st == ST_NEW1) ? new_hash[j]
                          : (st == ST_OLD0 || st == ST_UPD) ? new1_leaf[j] : zero[j];
        }
    }
    int rc = 0;
    if (enabled) {
        if (!eq4(prev_old, old_root)) rc = 4;
        else if (!eq4(prev_new, new_root)) rc = 5;
    } else {
        if (!eq4(old_root, new_root)) rc = 6;
        else if (!eq4(old_value, new_value)) rc = 7;
    }
    if (rc == 0 && (fnc == 1 || !enabled) && !eq4(old_key, new_key)) rc = 8;
    status[t] = rc;
}

// ------------------------------------------------------------------------------------------------
// launchers
// ------------------------------------------------------------------------------------------------
static inline unsigned nblk(u64 n, unsigned b) { return (unsigned)((n + b - 1) / b); }

void launch_permute_batch(u64* states, u64 m, cudaStream_t st) {
    if (m) { k_permute_batch<<<nblk(m, HASH_BLOCK), HASH_BLOCK, 0, st>>>(states, m); ++g_gl_launches; }
}
void launch_duplex_chain(u64* state, const u64* chunks, u64 m, cudaStream_t st) {
    k_duplex_chain<<<1, 32, 0, st>>>(state, chunks, m);
    ++g_gl_launches;
}
void launch_two_to_one_batch(const u64* l, const u64* r, u64* out, u64 m, cudaStream_t st) {
    if (m) { k_two_to_one_batch<<<nblk(m, HASH_BLOCK), HASH_BLOCK, 0, st>>>(l, r, out, m); ++g_gl_launches; }
}
void launch_hash_no_pad_rows(const u64* in, u32 len, u64 m, u64* out, cudaStream_t st) {
    if (m) { k_hash_no_pad_rows<<<nblk(m, HASH_BLOCK), HASH_BLOCK, 0, st>>>(in, len, m, out); ++g_gl_launches; }
}
void launch_smt_leaf_hash_batch(const u64* k, const u64* v, u64* out, u64 m, cudaStream_t st) {
    if (m) { k_smt_leaf_hash_batch<<<nblk(m, HASH_BLOCK), HASH_BLOCK, 0, st>>>(k, v, out, m); ++g_gl_launches; }
}
void launch_smt_verify_process(const gl_smt_proof_hdr* p, const u64* sib_pool, const u64* sib_off, u64 m,
                               int* status, cudaStream_t st) {
    if (m) { k_smt_verify_process<<<nblk(m, 128), 128, 0, st>>>(p, sib_pool, sib_off, m, status); ++g_gl_launches; }
}
void launch_merkle_verify_batch(const u64* leaves, u32 leaf_len, const u64* idx, const u64* paths, u32 path_len, const u64* cap,
                                u32 cap_height, u64 k, int* ok, cudaStream_t st) {
    if (k) { k_merkle_verify_batch<<<nblk(k, 128), 128, 0, st>>>(leaves, leaf_len, idx, paths, path_len, cap, cap_height, k, ok); ++g_gl_launches; }
}
void launch_pow_grind(const u64* state12, unsigned pos, unsigned out_pos, unsigned min_lz, u64 start, u64 count,
                      unsigned long long* best, cudaStream_t st) {
    if (count) { k_pow_grind<<<nblk(count, HASH_BLOCK), HASH_BLOCK, 0, st>>>(state12, pos, out_pos, min_lz, start, count, best); ++g_gl_launches; }
}

// Merkle tree over num_leaves = 2^lg leaves split in 2^cap_height subtrees.  digests: plonky2 layout.
void launch_leaf_hash_cols(const u64* lde, u64 ld, u32 c, unsigned lg_leaves, unsigned cap_height, u64* digests,
                           u64* cap, cudaStream_t st) {
    u64 n = (u64)1 << lg_leaves;
    unsigned sub_bits = lg_leaves - cap_height;
    { k_leaf_hash_cols<<<nblk(n, HASH_BLOCK), HASH_BLOCK, 0, st>>>(lde, ld, c, n, sub_bits, digests, cap); ++g_gl_launches; }
}
void launch_leaf_absorb_cols(const u64* lde, u64 ld, u32 col_begin, u32 col_end, unsigned lg_leaves, unsigned cap_height,
                             u64* state, bool first, bool last, u64* digests, u64* cap, cudaStream_t st) {
    u64 n = (u64)1 << lg_leaves;
    unsigned sub_bits = lg_leaves - cap_height;
    k_leaf_absorb_cols<<<nblk(n, HASH_BLOCK), HASH_BLOCK, 0, st>>>(lde, ld, col_begin, col_end, n, sub_bits, state, first ? 1 : 0,
                                                                    last ? 1 : 0, digests, cap);
    ++g_gl_launches;
}
void launch_merkle_levels(unsigned lg_leaves, unsigned cap_height, u64* digests, u64* cap, cudaStream_t st) {
    u64 n = (u64)1 << lg_leaves;
    unsigned sub_bits = lg_leaves - cap_height;
    for (unsigned layer = 1; layer <= sub_bits; layer++) {
        u64 nodes = n >> layer;
        { k_merkle_level<<<nblk(nodes, HASH_BLOCK), HASH_BLOCK, 0, st>>>(digests, cap, sub_bits, layer, nodes); ++g_gl_launches; }
    }
}
void launch_merkle_cols(const u64* lde, u64 ld, u32 c, unsigned lg_leaves, unsigned cap_height, u64* digests,
                        u64* cap, cudaStream_t st) {
    launch_leaf_hash_cols(lde, ld, c, lg_leaves, cap_height, digests, cap, st);
    launch_merkle_levels(lg_leaves, cap_height, digests, cap, st);
}
void launch_merkle_rows(const u64* leaves, u32 leaf_len, unsigned lg_leaves, unsigned cap_height, u64* digests,
                        u64* cap, cudaStream_t st) {
    u64 n = (u64)1 << lg_leaves;
    unsigned sub_bits = lg_leaves - cap_height;
    { k_leaf_hash_rows<<<nblk(n, HASH_BLOCK), HASH_BLOCK, 0, st>>>(leaves, leaf_len, n, sub_bits, digests, cap); ++g_gl_launches; }
    for (unsigned layer = 1; layer <= sub_bits; layer++) {
        u64 nodes = n >> layer;
        { k_merkle_level<<<nblk(nodes, HASH_BLOCK), HASH_BLOCK, 0, st>>>(digests, cap, sub_bits, layer, nodes); ++g_gl_launches; }
    }
}

// Blinding salt: `count` uniform field elements (plonky2's F::rand_vec = rng.gen_range(0..ORDER) per element).  Counter
// mode: element i = mix(seed, stream, i) through two rounds of splitmix64, redrawn with a bumped counter while it falls
// in [p, 2^64) (probability 2^-32 per draw).
__device__ __forceinline__ u64 salt_mix(u64 x) {
    x += 0x9E3779B97F4A7C15ULL;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ULL;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBULL;
    return x ^ (x >> 31);
}
__global__ void __launch_bounds__(256) k_salt_fill(u64* __restrict__ out, u64 count, u64 seed, u64 stream) {
    const u64 key = salt_mix(seed ^ salt_mix(stream));
    for (u64 i = blockIdx.x * (u64)256 + threadIdx.x; i < count; i += (u64)gridDim.x * 256) {
        u64 v, redraw = 0;
        do {
            v = salt_mix(salt_mix(key + i) ^ (redraw++ << 56) ^ key);
        } while (v >= GL_P);
        out[i] = v;
    }
}
void launch_salt_fill(u64* out, u64 count, u64 seed, u64 stream, cudaStream_t st) {
    if (!count) return;
    u64 blocks = (count + 255) / 256;
    if (blocks > 4096) blocks = 4096;
    k_salt_fill<<<(unsigned)blocks, 256, 0, st>>>(out, count, seed, stream);
    ++g_gl_launches;
}

// N2: SMT bulk build (shares this translation unit's Poseidon constants)
#include "smt_kernels.cu"
#include "smt_proofs.cu"
