/*
 * gl_b200.h -- C ABI of libgl_b200.so: the B200-native Goldilocks NTT/LDE + Poseidon Merkle commit
 * core that sits underneath every `data.prove(pw)` / `builder.build::<C>()` / `PoseidonHash::*`
 * call of Orbiter-Finance/Plonky2-lib.
 *
 * The reference itself has no FFI: the path lives in its un-vendored dependency plonky2 0.1.4
 * (ZeroKPunk fork, /root/reference/Cargo.toml:10-11,32-34).  Each entry point below names the
 * upstream Rust interface it replaces AND the reference call sites (paths relative to
 * /root/reference) that reach it; INTEGRATION.md shows the Rust `extern "C"` shim a maintainer of
 * the fork would add.
 *
 * Conventions
 *  - field elements are u64, little-endian host order; inputs may be any u64 (taken mod p),
 *    outputs are canonical (< p = 2^64 - 2^32 + 1), so byte-compare with HashOut::to_bytes works.
 *  - `space` says where the caller's buffers live: GL_HOST (pageable or pinned host memory; the
 *    library stages the copies) or GL_DEVICE (device pointers on the ctx's device; used by callers
 *    that keep data resident, e.g. bench.py's `value` leg).
 *  - every function returns 0 on success or a GL_E_* code; gl_last_error() gives the text.  The
 *    upstream functions are infallible and panic on contract violation (log2_strict on a
 *    non-power-of-two, `cap_height <= log2(leaves.len())`, inconsistent polynomial degrees): those
 *    violations return GL_E_ARG and the Rust shim turns any non-zero code into panic!.
 *  - a gl_ctx owns one device, one stream and its scratch; calls on one ctx are stream-ordered and
 *    blocking at return.  One ctx per GPU; multi-GPU sharding is set with gl_ctx_set_shard().
 *  - no CPU fallback exists: without a CUDA device gl_ctx_create fails with GL_E_CUDA.
 */
#ifndef GL_B200_H
#define GL_B200_H
#include <stddef.h>
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define GL_OK 0
#define GL_E_ARG 1   /* upstream would panic: bad sizes / non power of two / cap_height too large */
#define GL_E_CUDA 2  /* CUDA runtime error (no device, launch failure, ...) */
#define GL_E_OOM 3   /* device or pinned host allocation failed */
#define GL_E_STATE 4 /* handle used on the wrong ctx / after free */
#define GL_E_NCCL 5  /* NCCL missing or a collective failed (gl_group_* only) */

#define GL_HOST 0
#define GL_DEVICE 1

typedef struct gl_ctx gl_ctx;
typedef struct gl_commit gl_commit;

/* ---- context --------------------------------------------------------------------------------- */
int gl_ctx_create(int device, gl_ctx **out);
void gl_ctx_destroy(gl_ctx *ctx);
const char *gl_last_error(const gl_ctx *ctx); /* ctx may be NULL: error of the last failed create */
void *gl_ctx_stream(gl_ctx *ctx);             /* the ctx's cudaStream_t, for CUDA-event timing */
int gl_ctx_sync(gl_ctx *ctx);
/* Multi-GPU: this ctx computes only leaf block [index*N/count, (index+1)*N/count) of every commit
 * (= LDE cosets k with bitrev_r(k) in that range = whole top-level Merkle subtrees, SURVEY 8e).
 * count must divide 2^rate_bits and 2^cap_height.  Default (0, 1). */
int gl_ctx_set_shard(gl_ctx *ctx, uint32_t index, uint32_t count);
uint64_t gl_ctx_kernel_launches(const gl_ctx *ctx); /* kernels launched so far by this process */
/* Device time of the phases of the last gl_commit_from_* call on this ctx, in ms (CUDA events on the
 * ctx stream): [0] copy-in, [1] IFFT, [2] coefficients out, [3] LDE NTT, [4] leaf hashing, [5] tree levels. */
int gl_ctx_commit_phase_ms(const gl_ctx *ctx, float *out6);
/* Return pooled device memory (freed commits keep their blocks for the next commit) to the driver. */
int gl_ctx_trim(gl_ctx *ctx);
/* Device memory owned by the caller (host mirrors keep the FRI polynomial and the layer values resident between
 * calls with it) and a copy between any two spaces, ordered on the ctx stream and blocking at return. */
int gl_dev_alloc(gl_ctx *ctx, size_t bytes, void **out);
void gl_dev_free(gl_ctx *ctx, void *p);
int gl_copy(gl_ctx *ctx, void *dst, int dst_space, const void *src, int src_space, size_t bytes);
/* Page-locked host memory for callers that want full-speed PCIe copies of their GL_HOST buffers
 * (the Rust shim backs the Vec<F> of a PolynomialBatch with it); plain malloc memory also works. */
int gl_host_alloc(size_t bytes, void **out);
void gl_host_free(void *p);

/* ---- P5/P6: PoseidonHash (plonky2::hash::poseidon) ------------------------------------------- */
/* Poseidon::poseidon over m states [m][12], in place. */
int gl_poseidon_permute_batch(gl_ctx *ctx, uint64_t *states, uint64_t m, int space);
/* m consecutive Challenger::duplexing steps with a full input buffer (plonky2::iop::challenger, overwrite mode):
 * for each chunk of 8 elements, state[0..8] = chunk, then permute.  One launch for the whole chain, so observing
 * a Merkle cap (64 elements) costs 8 dependent permutations and ONE host round trip.  state: 12 elements, in and
 * out; chunks: [m][8].  Host pointers. */
int gl_poseidon_duplex_chain(gl_ctx *ctx, uint64_t *state, const uint64_t *chunks, uint64_t m);
/* PoseidonHash::two_to_one (src/smt/goldilocks_poseidon/mod.rs:165, src/zkdsa/account.rs:165,
 * src/zkdsa/circuits/mod.rs:66-67): l, r, out are [m][4]. */
int gl_poseidon_two_to_one_batch(gl_ctx *ctx, const uint64_t *l, const uint64_t *r, uint64_t *out,
                                 uint64_t m, int space);
/* PoseidonHash::hash_no_pad over m inputs of len_each elements, in [m][len_each], out [m][4]. */
int gl_poseidon_hash_no_pad_batch(gl_ctx *ctx, const uint64_t *in, uint32_t len_each, uint64_t m,
                                  uint64_t *out, int space);
/* PoseidonNodeHash::calc_node_hash(Node::Leaf(k, v)) = hash_pad([k, v, 1])
 * (src/smt/goldilocks_poseidon/mod.rs:167-181): keys, values, out are [m][4]. */
int gl_smt_leaf_hash_batch(gl_ctx *ctx, const uint64_t *keys, const uint64_t *values, uint64_t *out,
                           uint64_t m, int space);

/* ---- P7: SparseMerkleProcessProof::check over a batch (src/smt/proof/process.rs:47-51,153-337) -- */
typedef struct {
    uint64_t old_root[4], old_key[4], old_value[4];
    uint64_t new_root[4], new_key[4], new_value[4];
    uint32_t is_old0;
    uint32_t fnc; /* ProcessMerkleProofRole: 0 NoOp, 1 Update, 2 Insert, 3 Delete */
} gl_smt_proof_hdr;
/* proofs [m]; siblings of proof t are sib_pool[sib_off[t] .. sib_off[t+1]) (each 4 x u64), top level
 * first, exactly `proof.siblings`; status[t] = 0 when every assert of verify_smt_process_proof
 * holds, else the ordinal of the first assert that would panic (1..8, see DESIGN.md). */
int gl_smt_verify_process_batch(gl_ctx *ctx, const gl_smt_proof_hdr *proofs, const uint64_t *sib_pool,
                                const uint64_t *sib_off, uint64_t m, int32_t *status, int space);

/* ---- N2: bulk build of the sparse Merkle tree (src/smt/tree.rs) ------------------------------------------------- */
/* The root (and optionally every internal node) of the compact sparse Merkle tree holding m DISTINCT keys with
 * non-default values: what m successive SparseMerkleTree::set calls (src/smt/tree.rs:143-155; insert :255-387) on an
 * empty PoseidonSparseMerkleTreeMemory leave behind, in any order (insert-only batches are order independent).
 * keys, values [m][4]; root_out [4]; nodes_out [nodes_cap][12] = (hash, left, right) of every Node::Internal the
 * NodeData store would hold, unordered (may be NULL); leaf_hashes_out [m][4] in input order (may be NULL);
 * *num_nodes_out = internal nodes produced (can exceed nodes_cap: only the first nodes_cap are stored).
 * Duplicate keys return GL_E_ARG ("given key already exists"). */
int gl_smt_build(gl_ctx *ctx, const uint64_t *keys, const uint64_t *values, uint64_t m, uint64_t *root_out,
                 uint64_t *nodes_out, uint64_t nodes_cap, uint64_t *num_nodes_out, uint64_t *leaf_hashes_out,
                 int space);

/* The m SparseMerkleProcessProofs that m successive `tree.set(keys[t], values[t])` calls return, in call order, when they
 * start from an EMPTY tree (src/smt/tree.rs:143-155; find :588-676, update :174-253, insert :255-387, remove :389-586).
 * Keys may repeat and values may be zero, exactly as with `set`: a non-zero value inserts the key or updates it, a zero
 * value removes it (ProcessDelete) or does nothing when it is not there (ProcessNoOp); proof t is against the tree the
 * first t calls left.  proofs_out [m]; the siblings of proof t are sib_pool_out[sib_off_out[t] .. sib_off_out[t+1])
 * exactly as `proof.siblings`: the three arrays are what gl_smt_verify_process_batch takes.  *num_siblings_out = total
 * number of siblings; when it exceeds sib_cap (or sib_pool_out is NULL) the pool is not written: call again with a
 * larger pool.  proofs_out[m-1].new_root is the root of the final tree.  A batch on a NON-empty tree: put the existing
 * entries first (any order) and drop their proofs. */
int gl_smt_set_proofs(gl_ctx *ctx, const uint64_t *keys, const uint64_t *values, uint64_t m,
                         gl_smt_proof_hdr *proofs_out, uint64_t *sib_pool_out, uint64_t sib_cap,
                         uint64_t *sib_off_out, uint64_t *num_siblings_out, int space);

/* SparseMerkleInclusionProof (src/smt/proof/inclusion.rs:5-33) without its siblings */
typedef struct gl_smt_inclusion_hdr {
    uint64_t root[4], key[4], value[4], not_found_key[4], not_found_value[4];
    uint32_t found;   /* the key is in the tree: `value` is its value */
    uint32_t is_old0; /* not found and the search ended in an empty slot (else, when not found: not_found_key / _value) */
} gl_smt_inclusion_hdr;
/* `tree.find(queries[i])` (src/smt/tree.rs:588-676) for nq keys against the tree that the m `set` calls of
 * (keys, values) leave when they start from an empty tree (same rules as gl_smt_set_proofs: keys may repeat, a zero
 * value removes).  proofs_out [nq]; siblings of proof i = sib_pool_out[sib_off_out[i] .. sib_off_out[i+1]), top level
 * first, every level down to where the search stops.  Pool sizing as in gl_smt_set_proofs. */
int gl_smt_find_batch(gl_ctx *ctx, const uint64_t *keys, const uint64_t *values, uint64_t m, const uint64_t *queries,
                      uint64_t nq, gl_smt_inclusion_hdr *proofs_out, uint64_t *sib_pool_out, uint64_t sib_cap,
                      uint64_t *sib_off_out, uint64_t *num_siblings_out, int space);

/* ---- P4: MerkleTree::new(leaves: Vec<Vec<F>>, cap_height) (plonky2::hash::merkle_tree) --------- */
/* leaves [num_leaves][leaf_len] row-major; digests_out [2*(num_leaves - 2^cap_height)][4] in
 * plonky2's recursive in-order layout (what MerkleTree::prove indexes); cap_out [2^cap_height][4].
 * digests_out may be NULL. */
int gl_merkle_build(gl_ctx *ctx, const uint64_t *leaves, uint64_t num_leaves, uint32_t leaf_len,
                    uint32_t cap_height, uint64_t *digests_out, uint64_t *cap_out, int space);

/* verify_merkle_proof_to_cap (plonky2::hash::merkle_proofs, the verifier's side of MerkleTree::prove) for k proofs against
 * one cap: leaves [k][leaf_len] (hash_or_noop applies), leaf_indices [k], paths [k][path_len][4] (siblings, leaf level
 * first), cap [2^cap_height][4]; ok[i] = 1 when the path leads to cap[leaf_index >> path_len], else 0.  rows / paths are
 * laid out as gl_commit_open writes them. */
int gl_merkle_verify_batch(gl_ctx *ctx, const uint64_t *leaves, uint32_t leaf_len, const uint64_t *leaf_indices,
                           const uint64_t *paths, uint32_t path_len, const uint64_t *cap, uint32_t cap_height,
                           uint64_t k, int32_t *ok, int space);

/* ---- P1/P2/P9: plonky2_field::fft on batches of columns ----------------------------------------- */
/* In place on [c][2^log_n] (column after column), natural order in and out.
 * gl_fft_batch      = PolynomialCoeffs::fft            (coeffs -> values on <w_n>)
 * gl_ifft_batch     = PolynomialValues::ifft           ("IFFT" stage of from_values)
 * gl_coset_fft_batch / gl_coset_ifft_batch = coset_fft(shift) / coset_ifft(shift) */
int gl_fft_batch(gl_ctx *ctx, uint64_t *data, uint32_t log_n, uint32_t c, int space);
int gl_ifft_batch(gl_ctx *ctx, uint64_t *data, uint32_t log_n, uint32_t c, int space);
int gl_coset_fft_batch(gl_ctx *ctx, uint64_t *data, uint32_t log_n, uint32_t c, uint64_t shift, int space);
int gl_coset_ifft_batch(gl_ctx *ctx, uint64_t *data, uint32_t log_n, uint32_t c, uint64_t shift, int space);

/* ---- P*: PolynomialBatch::from_values / from_coeffs (plonky2::fri::oracle) --------------------- */
/* Reached from data.prove(pw) (44 sites, e.g. src/ecdsa/gadgets/ecdsa.rs:349,
 * src/hash/keccak256.rs:248, src/smt/gadgets/process/mod.rs:82, src/zkdsa/circuits/mod.rs:326) and
 * builder.build::<C>() (41 sites, e.g. src/ecdsa/gadgets/ecdsa.rs:298).
 * values / coeffs: [c][2^log_n], one contiguous column after another (Vec<PolynomialValues<F>>).
 * These two entry points are the blinding = false form (every config of the reference: zero_knowledge: false); the _ex
 * forms below take upstream's `blinding` argument.
 * coeffs_out [c][2^log_n] (PolynomialBatch.polynomials; may be NULL), cap_out [2^cap_height][4]
 * (with a shard set: only this shard's 2^cap_height/count entries, written at their global index).
 * The LDE leaves and the digests stay on the device behind *handle ("resident mode"). */
int gl_commit_from_values(gl_ctx *ctx, const uint64_t *values, uint32_t log_n, uint32_t c,
                          uint32_t rate_bits, uint32_t cap_height, uint64_t *coeffs_out,
                          uint64_t *cap_out, gl_commit **handle, int space);
int gl_commit_from_coeffs(gl_ctx *ctx, const uint64_t *coeffs, uint32_t log_n, uint32_t c,
                          uint32_t rate_bits, uint32_t cap_height, uint64_t *cap_out,
                          gl_commit **handle, int space);
/* The same two commits with the polynomials where the reference keeps them: one host array per polynomial
 * (`values: Vec<PolynomialValues<F>>`, each a Vec<F> of 2^log_n elements -- plonky2::fri::oracle from_values /
 * from_coeffs; result `polynomials: Vec<PolynomialCoeffs<F>>`), so the binding passes `c` pointers and never
 * flattens.  Host memory only; the arrays may be page-able: helper threads pack them into page-locked rings
 * while the DMA engine and the transforms run (GL_B200_HOST_THREADS, default min(8, cores / 2)).
 * coeffs_out: `c` pointers to arrays of 2^log_n (or NULL). */
int gl_commit_from_values_cols(gl_ctx *ctx, const uint64_t *const *values, uint32_t log_n, uint32_t c,
                               uint32_t rate_bits, uint32_t cap_height, uint64_t *const *coeffs_out,
                               uint64_t *cap_out, gl_commit **handle);
int gl_commit_from_coeffs_cols(gl_ctx *ctx, const uint64_t *const *coeffs, uint32_t log_n, uint32_t c,
                               uint32_t rate_bits, uint32_t cap_height, uint64_t *cap_out,
                               gl_commit **handle);
/* Upstream's full signatures, `blinding` included (plonky2::fri::oracle::PolynomialBatch::from_values(values, rate_bits,
 * blinding, cap_height, ..) / from_coeffs): with blinding != 0 every leaf carries SALT_SIZE = 4 uniform random field
 * elements after its c polynomial values (lde_values(): `.chain((0..salt_size).map(|_| F::rand_vec(n << rate_bits)))`), so
 * MerkleTree.leaves[i].len() = c + 4 -- gl_commit_open, gl_commit_download, gl_group_commit_open and the rows of
 * gl_fri_prove have that width (gl_commit_leaf_len) -- while gl_commit_get_lde_values strips the salt as upstream does
 * and the polynomials stay c.  Pass the polynomials either as one array (values / coeffs, `space` memory) or as one host
 * array each (values_cols / coeffs_cols; the other pointer NULL).  The salt comes from a counter-mode generator on the
 * device seeded from the OS entropy source at gl_ctx_create; gl_ctx_set_salt_seed makes it reproducible (tests). */
#define GL_SALT_SIZE 4u
int gl_commit_from_values_ex(gl_ctx *ctx, const uint64_t *values, const uint64_t *const *values_cols, uint32_t log_n,
                             uint32_t c, uint32_t rate_bits, uint32_t blinding, uint32_t cap_height, uint64_t *coeffs_out,
                             uint64_t *const *coeffs_out_cols, uint64_t *cap_out, gl_commit **handle, int space);
int gl_commit_from_coeffs_ex(gl_ctx *ctx, const uint64_t *coeffs, const uint64_t *const *coeffs_cols, uint32_t log_n,
                             uint32_t c, uint32_t rate_bits, uint32_t blinding, uint32_t cap_height, uint64_t *cap_out,
                             gl_commit **handle, int space);
int gl_ctx_set_salt_seed(gl_ctx *ctx, uint64_t seed);
int gl_commit_leaf_len(const gl_commit *h, uint32_t *len);   /* c, or c + GL_SALT_SIZE for a blinded commit */
/* The same commit fed column block by column block (from_coeffs as a stream): begin allocates the resident buffers,
 * add_coeffs copies the coefficients of polynomials [col0, col0 + ncols) ([ncols][2^log_n]) behind the handle and runs
 * their LDE, finish hashes the leaves and builds the tree once every column has arrived.  Lets a caller overlap the
 * arrival of coefficients (PCIe, or an NCCL all-gather in the multi-GPU plan) with the transforms of earlier blocks. */
int gl_commit_begin(gl_ctx *ctx, uint32_t log_n, uint32_t c, uint32_t rate_bits, uint32_t cap_height, gl_commit **handle);
/* flags: GL_COMMIT_STREAM_HASH -- when the blocks are added in polynomial order, every complete group of 8 polynomials
 * (the sponge rate) is absorbed into the per-leaf Poseidon state as soon as its LDE exists, so the leaf hashing of the
 * blocks that have arrived overlaps the arrival (PCIe, NCCL) of the next ones instead of starting after the last;
 * costs 96 B of state per leaf until finish.  Same digests either way. */
#define GL_COMMIT_STREAM_HASH 1u
#define GL_COMMIT_BLINDING 2u   /* salted leaves, as gl_commit_from_coeffs_ex(blinding = 1); also taken by gl_group_commit_* */
int gl_commit_begin_ex(gl_ctx *ctx, uint32_t log_n, uint32_t c, uint32_t rate_bits, uint32_t cap_height, uint32_t flags,
                       gl_commit **handle);
int gl_commit_add_coeffs(gl_commit *h, uint32_t col0, uint32_t ncols, const uint64_t *coeffs, int space);
int gl_commit_finish(gl_commit *h, uint64_t *cap_out, int space);
/* PolynomialBatch.polynomials: the coefficients [c][2^log_n] kept on the device behind the handle. */
int gl_commit_coeffs(gl_commit *h, uint64_t *coeffs_out, int space);
/* OpeningSet::new (plonky2::plonk::proof; PolynomialCoeffs::eval at an extension-field point) for every polynomial of
 * the commit: values_out [c][2] = polynomial j evaluated at point = (a0, a1) of F[X]/(X^2 - 7), from the resident
 * coefficients (nothing but c x 16 bytes crosses PCIe). */
int gl_commit_eval(gl_commit *h, const uint64_t point[2], uint64_t *values_out, int space);
/* "mirror mode": fill the upstream structs.  leaves_out [N_local][c] row-major in leaf order
 * (= MerkleTree.leaves after transpose + reverse_index_bits), digests_out [2*(N_local - caps_local)][4]
 * (= MerkleTree.digests).  Either may be NULL. */
int gl_commit_download(gl_commit *h, uint64_t *leaves_out, uint64_t *digests_out, int space);
/* MerkleTree::get(i) + MerkleTree::prove(i) for k leaf indices (global indices; must be owned by
 * this shard): rows_out [k][c], paths_out [k][log2(N) - cap_height][4] (siblings, leaf level first). */
int gl_commit_open(gl_commit *h, const uint64_t *leaf_indices, uint32_t k, uint64_t *rows_out,
                   uint64_t *paths_out, int space);
/* PolynomialBatch::get_lde_values(index, step) = leaves[reverse_bits(index*step, log2 N)] for k indices. */
int gl_commit_get_lde_values(gl_commit *h, const uint64_t *indices, uint32_t k, uint64_t step,
                             uint64_t *rows_out, int space);
/* geometry of a handle */
int gl_commit_info(const gl_commit *h, uint32_t *log_n, uint32_t *c, uint32_t *rate_bits,
                   uint32_t *cap_height, uint64_t *leaf_begin, uint64_t *leaf_end);
/* device pointers of the resident data (column-major leaves [c][ld], digests), for device callers */
int gl_commit_device_ptrs(const gl_commit *h, const uint64_t **lde_cols, uint64_t *ld,
                          const uint64_t **digests);
void gl_commit_free(gl_commit *h);

/* ---- (e) multi-GPU: one commit sharded over the GPUs of a box, NCCL behind this ABI (SURVEY 8b, 8e) -----------------------
 * One rank = one gl_ctx = one GPU.  Rank r owns leaf block r of nranks (LDE cosets = whole top-level Merkle subtrees and
 * their cap entries); the IFFT is sharded by polynomial and the coefficients are exchanged round by round while the
 * previous round is extended -- by ncclAllGather when the inputs are resident, by the ranks' own pull kernels over peer
 * memory (NVLink; exchange buffers mapped with CUDA IPC across processes) when they are host buffers; the cap is
 * all-gathered; query openings are exchanged by gl_group_commit_open.  A process
 * may hold all ranks (the Rust prover: one process, 8 GPUs, id = NULL) or some of them (one rank per process under a
 * torchrun-style launcher: rank 0 calls gl_group_unique_id and hands the 128 bytes to the others out of band).
 * NCCL is bound at run time (dlopen): nothing else in this header needs it.  Replaces the rayon data parallelism of
 * plonky2_maybe_rayon 0.1.1 (Cargo.lock:993-998) inside from_values / from_coeffs, reached from data.prove(pw)
 * (e.g. src/zkdsa/circuits/mod.rs:326, src/ecdsa/gadgets/ecdsa.rs:349). */
typedef struct gl_group gl_group;
#define GL_GROUP_ID_BYTES 128
int gl_group_unique_id(uint8_t *id_out /* [GL_GROUP_ID_BYTES] */);
/* ctxs [nlocal]: this process's ranks rank0 .. rank0 + nlocal - 1 of nranks (a power of two dividing 2^rate_bits and
 * 2^cap_height of every commit made with the group).  Sets each ctx's shard to (rank, nranks).  Collective. */
int gl_group_create(gl_ctx *const *ctxs, uint32_t nlocal, uint32_t rank0, uint32_t nranks, const uint8_t *id, gl_group **out);
void gl_group_destroy(gl_group *g);
const char *gl_group_last_error(const gl_group *g);
int gl_group_info(const gl_group *g, uint32_t *nlocal, uint32_t *rank0, uint32_t *nranks, int *nccl_version);
int gl_group_commit_phase_ms(const gl_group *g, float *out6); /* first local rank, as gl_ctx_commit_phase_ms */
/* PolynomialBatch::from_values / from_coeffs, sharded.  Collective: every rank calls it with the same geometry.
 * values [nlocal]: per local rank the WHOLE batch [c][2^log_n] in `space` memory of that rank (GL_DEVICE: on its GPU;
 * GL_HOST: host memory, the pointers may be equal); a rank reads only the polynomials it inverse-transforms.
 * coeffs_out [nlocal] or NULL: GL_DEVICE: every rank receives all c coefficient vectors; GL_HOST: a rank writes only ITS
 * polynomials into coeffs_out[i] (one shared array is complete when the process holds every rank).
 * cap_out [nlocal] or NULL: the WHOLE cap [2^cap_height][4] on every rank.  handles [nlocal]: this rank's shard
 * (gl_commit_open serves its own leaves, gl_group_commit_open any leaf).  flags: GL_COMMIT_STREAM_HASH, GL_COMMIT_BLINDING
 * (every rank salts its own leaves). */
int gl_group_commit_from_values(gl_group *g, const uint64_t *const *values, uint32_t log_n, uint32_t c, uint32_t rate_bits,
                                uint32_t cap_height, uint64_t *const *coeffs_out, uint64_t *const *cap_out,
                                gl_commit **handles, int space, uint32_t flags);
int gl_group_commit_from_coeffs(gl_group *g, const uint64_t *const *coeffs, uint32_t log_n, uint32_t c, uint32_t rate_bits,
                                uint32_t cap_height, uint64_t *const *cap_out, gl_commit **handles, int space, uint32_t flags);
/* MerkleTree::get(i) + MerkleTree::prove(i) for k GLOBAL leaf indices of a sharded commit (fri_prover_query_round's
 * initial-tree openings): each index is served by the rank that owns the leaf and the rows / paths are exchanged over
 * NCCL; every rank ends with rows_out[i] [k][c] and paths_out[i] [k][log2(N) - cap_height][4].  Collective; host buffers. */
int gl_group_commit_open(gl_group *g, gl_commit *const *handles, const uint64_t *leaf_indices, uint32_t k,
                         uint64_t *const *rows_out, uint64_t *const *paths_out, int space);
/* Pins the calling thread to the CPUs next to the ctx's GPU (sysfs local_cpulist), so that page-locked buffers it
 * allocates afterwards and the staging threads' copies stay on the GPU's NUMA node. */
int gl_ctx_bind_host_numa(gl_ctx *ctx);

/* ---- P8: one reduction layer of fri_committed_trees (plonky2::fri::prover) ---------------------- */
/* values_ext: len extension elements [len][2] in natural order of their coset.  Builds the layer
 * tree: reverse_index_bits(values), leaves = chunks of 2^arity_bits ext elements flattened,
 * MerkleTree::new(leaves, cap_height).  digests_out may be NULL. */
int gl_fri_layer_tree(gl_ctx *ctx, const uint64_t *values_ext, uint64_t len, uint32_t arity_bits,
                      uint32_t cap_height, uint64_t *digests_out, uint64_t *cap_out, int space);
/* The same layer tree, kept RESIDENT for the query phase (fri_prover_query_round reads tree.get(x >> arity_bits)
 * and tree.prove(x >> arity_bits) from every layer): *handle behaves like a commit of 2 * 2^arity_bits columns
 * over len >> arity_bits leaves (gl_commit_open returns the flattened evals and the sibling path). */
int gl_fri_layer_commit(gl_ctx *ctx, const uint64_t *values_ext, uint64_t len, uint32_t arity_bits,
                        uint32_t cap_height, uint64_t *cap_out, gl_commit **handle, int space);
/* coeffs.chunks_exact(2^arity_bits).map(|c| reduce_with_powers(c, beta)) then coset_fft(shift) over
 * F::Extension: coeffs_ext [len][2] -> folded_coeffs_out [len >> arity_bits][2] and
 * next_values_out [len >> arity_bits][2] (either may be NULL). */
int gl_fri_fold(gl_ctx *ctx, const uint64_t *coeffs_ext, uint64_t len, uint32_t arity_bits,
                const uint64_t beta[2], uint64_t shift, uint64_t *folded_coeffs_out,
                uint64_t *next_values_out, int space);

/* ---- N1: PolynomialBatch::prove_openings up to the FRI polynomial (plonky2::fri::oracle) ----------------- */
/* One FriBatchInfo: the polynomials polys[first_poly .. first_poly + num_polys) are opened at `point`
 * (an extension element); a polynomial is (oracle_index, polynomial_index) into the resident commits. */
typedef struct {
    uint64_t point[2];
    uint32_t first_poly, num_polys;
} gl_fri_batch;
typedef struct {
    uint32_t oracle_index, polynomial_index;
} gl_fri_poly;
/* final_poly = sum_i alpha^(k_i) (F_i(X) - F_i(z_i)) / (X - z_i), F_i = sum_j alpha^j f_ij  (reduce_polys_base,
 * divide_by_linear, shift_poly), then final_poly.lde(rate_bits) and its coset_fft(7) over the extension.
 * Every oracle must be a commit of this ctx with the same degree.  Outputs: lde_coeffs_out and lde_values_out,
 * both [n << rate_bits][2] (natural order) -- the two arguments fri_proof takes.  Either may be NULL. */
int gl_fri_final_poly(gl_ctx *ctx, gl_commit *const *oracles, uint32_t num_oracles, const gl_fri_batch *batches,
                      uint32_t num_batches, const gl_fri_poly *polys, const uint64_t alpha[2], uint32_t rate_bits,
                      uint64_t *lde_coeffs_out, uint64_t *lde_values_out, int space);

/* Fork-version switches, all in one place (SURVEY 8c "residual risk": the plonky2 fork is not vendored, so every choice
 * that differs between upstream revisions is isolated here and can be flipped when the fork's source is at hand):
 *   GL_COMPAT_FRI_FINAL_POLY_TIMES_X  prove_openings multiplies the FRI polynomial by X (`final_poly.coeffs.insert(0, ZERO)`,
 *       upstream PR #436) and the verifier's fri_combine_initial returns `sum * subgroup_x`.  Upstream later removed this
 *       ("pad back to power of two" instead); the default (flag clear) is the later form.
 * Other revision-dependent points and where they live: proof-of-work = duplex-state form, output lane 7
 * (gl_pow_grind; csrc k_pow_grind takes the output lane as a parameter); hash_pad pads to SPONGE_WIDTH = 12 (forced by the
 * reference itself, src/smt/gadgets/common.rs:87-101); Challenger = overwrite-mode duplex, outputs popped from the back. */
#define GL_COMPAT_FRI_FINAL_POLY_TIMES_X 1u
int gl_ctx_set_compat(gl_ctx *ctx, uint32_t flags);

/* ---- N1 in one call: PolynomialBatch::prove_openings + fri_proof (plonky2::fri::oracle, fri::prover) ----------------------
 * The Fiat-Shamir sponge (plonky2::iop::challenger::Challenger, overwrite-mode duplex) as plain data: */
typedef struct {
    uint64_t sponge_state[12];
    uint64_t input_buffer[8];
    uint64_t output_buffer[8];   /* popped from the back: output_buffer[output_len - 1] is the next challenge */
    uint32_t input_len, output_len;
} gl_challenger;
#define GL_FRI_MAX_LAYERS 16
typedef struct {
    uint32_t rate_bits, cap_height, proof_of_work_bits, num_query_rounds;   /* FriConfig */
    uint32_t num_reduction_layers;
    uint32_t reduction_arity_bits[GL_FRI_MAX_LAYERS];                        /* FriParams.reduction_arity_bits */
    uint32_t flags;                                                          /* GL_COMPAT_FRI_* (or'ed with the ctx's) */
} gl_fri_params;
/* Size of the proof in u64 words for oracles of oracle_columns[i] polynomials of degree 2^degree_bits. */
int gl_fri_proof_words(const gl_fri_params *prm, const uint32_t *oracle_columns, uint32_t num_oracles, uint32_t degree_bits,
                       uint64_t *words_out);
/* `challenger`: in = the transcript state when prove_openings is entered (openings already observed), out = its state after
 * the proof (what the caller's Challenger continues from).  The FRI polynomial, every layer tree, the sponge, the
 * proof-of-work search (smallest witness) and the query openings stay on the device; ONE copy brings the proof back:
 *   for each reduction layer: cap [2^cap_height][4]
 *   final_poly [len][2]; pow_witness
 *   for each query round: x_index; for each oracle: leaf row [c], Merkle path [lg N - cap_height][4];
 *                         for each layer: evals [2^arity][2], Merkle path
 * (FriProof { commit_phase_merkle_caps, final_poly, pow_witness, query_round_proofs } field by field, in declaration
 * order of use).  proof_out: host buffer of proof_cap_words words; *proof_words_out = words needed / written. */
int gl_fri_prove(gl_ctx *ctx, gl_commit *const *oracles, uint32_t num_oracles, const gl_fri_batch *batches, uint32_t num_batches,
                 const gl_fri_poly *polys, const gl_fri_params *prm, gl_challenger *challenger, uint64_t *proof_out,
                 uint64_t proof_cap_words, uint64_t *proof_words_out);

/* ---- N3: compute_quotient_polys (plonky2::plonk::prover, vanishing_poly::eval_vanishing_poly_base_batch) ------------------
 * The last prover stage that reads every LDE row (SURVEY 3.2 step 8): with it the three prove-time oracles never leave HBM.
 * Reached from every data.prove(pw); the gate evaluators cover upstream's NoopGate / ConstantGate / PublicInputGate and
 * the three gates whose source is in the reference: U32InterleaveGate (src/u32/gates/interleave_u32.rs:89-126),
 * UninterleaveToU32Gate (uninterleave_to_u32.rs:98-145), UninterleaveToB32Gate (uninterleave_to_b32.rs:101-149) -- the
 * circuits of src/hash/keccak256.rs:248 are built from them plus plonky2_u32's gates (not covered yet). */
#define GL_GATE_NOOP 0
#define GL_GATE_CONSTANT 1            /* ConstantGate { num_consts = num_ops } */
#define GL_GATE_PUBLIC_INPUT 2
#define GL_GATE_U32_INTERLEAVE 3
#define GL_GATE_UNINTERLEAVE_TO_U32 4
#define GL_GATE_UNINTERLEAVE_TO_B32 5
typedef struct {
    uint32_t kind, num_ops;
    uint32_t selector_index;          /* selectors_info.selector_indices[gate]: its selector column among the constants */
    uint32_t group_start, group_end;  /* selectors_info.groups[selector_index]; the gate's own index is its position in gates[] */
    uint32_t reserved;
} gl_gate;
typedef struct {
    uint32_t degree_bits, num_wires, num_routed_wires;
    uint32_t num_constants;           /* constant columns INCLUDING the num_selectors selector columns, which come first */
    uint32_t num_selectors, num_challenges;
    uint32_t quotient_degree_factor;  /* a power of two <= 2^rate_bits (8 for every preset the reference uses) */
    uint32_t num_gates;               /* <= 16 */
} gl_circuit;
/* constants_sigmas: commit of [num_constants constants | num_routed_wires sigmas]; wires: num_wires columns;
 * zs_partial_products: [Z_0 .. Z_{nch-1} | partial products of challenge 0, 1, ..] (num_challenges * ceil(routed / qdf)
 * columns).  All three resident on ctx with the same degree and rate_bits, unsharded.  k_is [num_routed_wires],
 * public_inputs_hash [4], betas / gammas / alphas [num_challenges]: host.  chunks_out [num_challenges *
 * quotient_degree_factor][2^degree_bits] = quotient_polys.flat_map(|p| p.chunks(degree)): the coefficient vectors the
 * prover commits next (gl_commit_from_coeffs takes them as they are, also with space = GL_DEVICE). */
int gl_quotient_polys(gl_ctx *ctx, const gl_circuit *circuit, const gl_gate *gates, const uint64_t *k_is,
                      gl_commit *constants_sigmas, gl_commit *wires, gl_commit *zs_partial_products,
                      const uint64_t *public_inputs_hash, const uint64_t *betas, const uint64_t *gammas,
                      const uint64_t *alphas, uint64_t *chunks_out, int space);

/* ---- plonky2::plonk::prover all_wires_permutation_partial_products / wires_permutation_partial_products_and_zs ----------
 * (SURVEY 3.2 step 5), on the resident oracles; reached from every data.prove(pw).  Reads degree_bits, num_wires,
 * num_routed_wires (R), num_constants, num_challenges (nch <= 4) and quotient_degree_factor (deg, a power of two) of
 * `circuit`.  The routed wire values (columns [0, R) of `wires`) and the sigma values (columns [num_constants,
 * num_constants + R) of `constants_sigmas`) are recovered on the device from the coefficients the two commits hold (commits
 * of from_values or from_coeffs, blinded or not; unsharded, same degree, nch * ceil(R / deg) <= 64).  k_is [R], betas /
 * gammas [nch]: host.
 * zs_partial_products_out [nch * ceil(R / deg)][2^degree_bits] in `space`: values on the subgroup, canonical, laid out as
 * the prover commits them (Z_0 .. Z_{nch-1}, then the ceil(R / deg) - 1 partial products of challenge 0, 1, ..) -- what
 * gl_quotient_polys reads; a GL_DEVICE buffer goes straight into gl_commit_from_values(.., GL_DEVICE).
 * grand_products_out [nch] (host, may be NULL): per challenge the product of the row ratios over all rows, 1 exactly when
 * the witness satisfies every copy constraint.  A product other than 1 is not an error: the call returns GL_OK with every
 * column written, as the prover does not panic there (the proof is simply invalid).  This is the one deliberate
 * difference from the CPU restatement glo_permutation_zs (oracle/gl_oracle.c), which stops at the first challenge whose
 * product is not 1 and fails.  A zero denominator
 * wire + beta * sigma + gamma at some row returns GL_E_ARG (upstream's batch_multiplicative_inverse panics). */
int gl_permutation_zs(gl_ctx *ctx, const gl_circuit *circuit, const uint64_t *k_is, gl_commit *constants_sigmas,
                      gl_commit *wires, const uint64_t *betas, const uint64_t *gammas, uint64_t *zs_partial_products_out,
                      int space, uint64_t *grand_products_out);

/* ---- N3 in one call: plonky2::plonk::prover::prove from the point where the witness exists ------------------------------
 * Reached from every data.prove(pw) (44 sites, e.g. src/ecdsa/gadgets/ecdsa.rs:349, src/hash/keccak256.rs:248,
 * src/smt/gadgets/process/mod.rs:82, src/zkdsa/circuits/mod.rs:326), for circuits built from the gates gl_quotient_polys
 * evaluates.  Upstream's order, with the Fiat-Shamir sponge on the device:
 *   public_inputs_hash = hash_no_pad(public_inputs) ([0, 0, 0, 0] without public inputs); wires commit (from_values,
 *   blinding = false); Challenger::new(), observe circuit_digest, public_inputs_hash, wires cap; betas, gammas
 *   (get_n_challenges(num_challenges) each); Z and partial products (gl_permutation_zs) and their commit; observe the cap,
 *   alphas; quotient (gl_quotient_polys) and its commit (from_coeffs); observe the cap, zeta = get_extension_challenge()
 *   (GL_E_STATE when zeta^(2^degree_bits) == 1, upstream's ensure!); OpeningSet at zeta, plonk_zs_next at g * zeta;
 *   observe_openings(to_fri_openings()); prove_openings (gl_fri_prove) over the oracles [constants_sigmas, wires,
 *   zs_partial_products, quotient]: every polynomial at zeta, polynomials 0 .. num_challenges of oracle 2 at g * zeta.
 * constants_sigmas: the caller's resident prover-data commit ([num_constants | num_routed_wires sigmas], unblinded, unsharded,
 *   this ctx, degree 2^degree_bits; prm's rate_bits and cap_height); it is read, never modified.  circuit_digest [4]:
 *   prover_data.circuit_digest (its derivation differs between fork revisions, so it is an input).  Witness: `wires`
 *   [num_wires][2^degree_bits] in `space` memory, or `wires_cols`, num_wires host arrays (the other pointer NULL), as in
 *   gl_commit_from_values_ex.  prm->flags and the ctx's compat flags apply as in gl_fri_prove.  public_inputs: host.
 * proof_out (host, ONE copy at the end), in u64 words: wires cap, zs_partial_products cap, quotient cap ([2^cap_height][4]
 *   each); the OpeningSet in declaration order, [k][2] per field: constants (num_constants), plonk_sigmas (num_routed_wires),
 *   wires (num_wires), plonk_zs (nch), plonk_zs_next (nch), partial_products (nch * (ceil(routed / qdf) - 1)),
 *   quotient_polys (nch * qdf); then the FRI proof word for word as gl_fri_prove writes it.  *proof_words_out is always
 *   set; a NULL or too small proof_out returns GL_E_ARG.  A witness that breaks a gate or copy constraint still returns
 *   GL_OK and a proof, as upstream's prover does: the verifier rejects it.  The three commits are internal and freed
 *   before return. */
int gl_prove(gl_ctx *ctx, const gl_circuit *circuit, const gl_gate *gates, const uint64_t *k_is, gl_commit *constants_sigmas,
             const uint64_t circuit_digest[4], const gl_fri_params *prm, const uint64_t *wires, const uint64_t *const *wires_cols,
             int space, const uint64_t *public_inputs, uint32_t num_public_inputs, uint64_t *proof_out, uint64_t proof_cap_words,
             uint64_t *proof_words_out);

/* ---- P10: fri_proof_of_work ------------------------------------------------------------------- */
/* Smallest w >= 0 such that permute(state with state[input_pos] = w)[7] (the last rate lane, as
 * `duplex_state.squeeze().last()`) has >= min_leading_zeros leading zero bits.  Upstream's rayon
 * find_any returns an arbitrary satisfying w; "smallest" makes the proof deterministic. */
int gl_pow_grind(gl_ctx *ctx, const uint64_t state[12], uint32_t input_pos, uint32_t min_leading_zeros,
                 uint64_t *witness_out);

#ifdef __cplusplus
}
#endif
#endif
