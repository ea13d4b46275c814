//! Raw bindings of include/gl_b200.h (link with `cargo:rustc-link-lib=dylib=gl_b200`).
#![allow(non_camel_case_types)]
use std::os::raw::{c_char, c_int, c_void};

pub enum gl_ctx {}
pub enum gl_commit {}
pub const GL_HOST: c_int = 0;
pub const GL_DEVICE: c_int = 1;
pub const GL_COMMIT_STREAM_HASH: u32 = 1;   // gl_commit_begin_ex: absorb the leaves block by block as they arrive

#[repr(C)]
pub struct gl_smt_proof_hdr {
    pub old_root: [u64; 4], pub old_key: [u64; 4], pub old_value: [u64; 4],
    pub new_root: [u64; 4], pub new_key: [u64; 4], pub new_value: [u64; 4],
    pub is_old0: u32,
    pub fnc: u32, // ProcessMerkleProofRole: 0 NoOp, 1 Update, 2 Insert, 3 Delete
}

extern "C" {
    pub fn gl_ctx_create(device: c_int, out: *mut *mut gl_ctx) -> c_int;
    pub fn gl_ctx_destroy(ctx: *mut gl_ctx);
    pub fn gl_last_error(ctx: *const gl_ctx) -> *const c_char;
    pub fn gl_ctx_set_shard(ctx: *mut gl_ctx, index: u32, count: u32) -> c_int;
    pub fn gl_host_alloc(bytes: usize, out: *mut *mut c_void) -> c_int;
    pub fn gl_host_free(p: *mut c_void);

    pub fn gl_poseidon_permute_batch(ctx: *mut gl_ctx, states: *mut u64, m: u64, space: c_int) -> c_int;
    pub fn gl_poseidon_duplex_chain(ctx: *mut gl_ctx, state: *mut u64, chunks: *const u64, m: u64) -> c_int;
    pub fn gl_poseidon_two_to_one_batch(ctx: *mut gl_ctx, l: *const u64, r: *const u64, out: *mut u64, m: u64, space: c_int) -> c_int;
    pub fn gl_poseidon_hash_no_pad_batch(ctx: *mut gl_ctx, input: *const u64, len_each: u32, m: u64, out: *mut u64, space: c_int) -> c_int;
    pub fn gl_smt_leaf_hash_batch(ctx: *mut gl_ctx, keys: *const u64, values: *const u64, out: *mut u64, m: u64, space: c_int) -> c_int;
    pub fn gl_smt_verify_process_batch(ctx: *mut gl_ctx, proofs: *const gl_smt_proof_hdr, sib_pool: *const u64,
                                       sib_off: *const u64, m: u64, status: *mut i32, space: c_int) -> c_int;

    pub fn gl_merkle_build(ctx: *mut gl_ctx, leaves: *const u64, num_leaves: u64, leaf_len: u32, cap_height: u32,
                           digests_out: *mut u64, cap_out: *mut u64, space: c_int) -> c_int;

    pub fn gl_merkle_verify_batch(ctx: *mut gl_ctx, leaves: *const u64, leaf_len: u32, leaf_indices: *const u64, paths: *const u64,
                                  path_len: u32, cap: *const u64, cap_height: u32, k: u64, ok: *mut i32, space: c_int) -> c_int;

    pub fn gl_commit_from_values(ctx: *mut gl_ctx, values: *const u64, log_n: u32, c: u32, rate_bits: u32, cap_height: u32,
                                 coeffs_out: *mut u64, cap_out: *mut u64, handle: *mut *mut gl_commit, space: c_int) -> c_int;
    pub fn gl_commit_from_coeffs(ctx: *mut gl_ctx, coeffs: *const u64, log_n: u32, c: u32, rate_bits: u32, cap_height: u32,
                                 cap_out: *mut u64, handle: *mut *mut gl_commit, space: c_int) -> c_int;
    pub fn gl_commit_from_values_cols(ctx: *mut gl_ctx, values: *const *const u64, log_n: u32, c: u32, rate_bits: u32, cap_height: u32,
                                      coeffs_out: *const *mut u64, cap_out: *mut u64, handle: *mut *mut gl_commit) -> c_int;
    pub fn gl_commit_from_coeffs_cols(ctx: *mut gl_ctx, coeffs: *const *const u64, log_n: u32, c: u32, rate_bits: u32, cap_height: u32,
                                      cap_out: *mut u64, handle: *mut *mut gl_commit) -> c_int;
    // upstream's full signatures (`blinding` taken): SALT_SIZE = 4 random elements appended to every leaf when blinding != 0
    pub fn gl_commit_from_values_ex(ctx: *mut gl_ctx, values: *const u64, values_cols: *const *const u64, log_n: u32, c: u32,
                                    rate_bits: u32, blinding: u32, cap_height: u32, coeffs_out: *mut u64,
                                    coeffs_out_cols: *const *mut u64, cap_out: *mut u64, handle: *mut *mut gl_commit,
                                    space: c_int) -> c_int;
    pub fn gl_commit_from_coeffs_ex(ctx: *mut gl_ctx, coeffs: *const u64, coeffs_cols: *const *const u64, log_n: u32, c: u32,
                                    rate_bits: u32, blinding: u32, cap_height: u32, cap_out: *mut u64,
                                    handle: *mut *mut gl_commit, space: c_int) -> c_int;
    pub fn gl_ctx_set_salt_seed(ctx: *mut gl_ctx, seed: u64) -> c_int;
    pub fn gl_commit_leaf_len(h: *const gl_commit, len: *mut u32) -> c_int;
    // plonky2_field::fft on batches of columns, in place on [c][2^log_n] (PolynomialCoeffs::fft, PolynomialValues::ifft, coset_*)
    pub fn gl_fft_batch(ctx: *mut gl_ctx, data: *mut u64, log_n: u32, c: u32, space: c_int) -> c_int;
    pub fn gl_ifft_batch(ctx: *mut gl_ctx, data: *mut u64, log_n: u32, c: u32, space: c_int) -> c_int;
    pub fn gl_coset_fft_batch(ctx: *mut gl_ctx, data: *mut u64, log_n: u32, c: u32, shift: u64, space: c_int) -> c_int;
    pub fn gl_coset_ifft_batch(ctx: *mut gl_ctx, data: *mut u64, log_n: u32, c: u32, shift: u64, space: c_int) -> c_int;
    pub fn gl_commit_begin(ctx: *mut gl_ctx, log_n: u32, c: u32, rate_bits: u32, cap_height: u32, handle: *mut *mut gl_commit) -> c_int;
    pub fn gl_commit_coeffs(h: *mut gl_commit, coeffs_out: *mut u64, space: c_int) -> c_int;
    pub fn gl_commit_info(h: *const gl_commit, log_n: *mut u32, c: *mut u32, rate_bits: *mut u32, cap_height: *mut u32,
                          leaf_begin: *mut u64, leaf_end: *mut u64) -> c_int;
    pub fn gl_ctx_sync(ctx: *mut gl_ctx) -> c_int;
    pub fn gl_ctx_trim(ctx: *mut gl_ctx) -> c_int;      // give pooled device memory back
    // instrumentation for benchmarks
    pub fn gl_ctx_stream(ctx: *mut gl_ctx) -> *mut c_void;
    pub fn gl_ctx_kernel_launches(ctx: *const gl_ctx) -> u64;
    pub fn gl_ctx_commit_phase_ms(ctx: *const gl_ctx, out6: *mut f32) -> c_int;
    pub fn gl_commit_device_ptrs(h: *const gl_commit, lde_cols: *mut *const u64, ld: *mut u64, digests: *mut *const u64) -> c_int;
    pub fn gl_commit_begin_ex(ctx: *mut gl_ctx, log_n: u32, c: u32, rate_bits: u32, cap_height: u32, flags: u32, handle: *mut *mut gl_commit) -> c_int;
    pub fn gl_commit_add_coeffs(h: *mut gl_commit, col0: u32, ncols: u32, coeffs: *const u64, space: c_int) -> c_int;
    pub fn gl_commit_finish(h: *mut gl_commit, cap_out: *mut u64, space: c_int) -> c_int;
    pub fn gl_commit_eval(h: *mut gl_commit, point: *const u64, values_out: *mut u64, space: c_int) -> c_int;   // OpeningSet::new
    pub fn gl_commit_download(h: *mut gl_commit, leaves_out: *mut u64, digests_out: *mut u64, space: c_int) -> c_int;
    pub fn gl_commit_open(h: *mut gl_commit, leaf_indices: *const u64, k: u32, rows_out: *mut u64, paths_out: *mut u64, space: c_int) -> c_int;
    pub fn gl_commit_get_lde_values(h: *mut gl_commit, indices: *const u64, k: u32, step: u64, rows_out: *mut u64, space: c_int) -> c_int;
    pub fn gl_commit_free(h: *mut gl_commit);

    pub fn gl_fri_layer_tree(ctx: *mut gl_ctx, values_ext: *const u64, len: u64, arity_bits: u32, cap_height: u32,
                             digests_out: *mut u64, cap_out: *mut u64, space: c_int) -> c_int;
    pub fn gl_fri_fold(ctx: *mut gl_ctx, coeffs_ext: *const u64, len: u64, arity_bits: u32, beta: *const u64, shift: u64,
                       folded_coeffs_out: *mut u64, next_values_out: *mut u64, space: c_int) -> c_int;
    pub fn gl_pow_grind(ctx: *mut gl_ctx, state: *const u64, input_pos: u32, min_leading_zeros: u32, witness_out: *mut u64) -> c_int;

    // N1: prove_openings / fri_proof with the FRI polynomial resident in HBM
    pub fn gl_dev_alloc(ctx: *mut gl_ctx, bytes: usize, out: *mut *mut c_void) -> c_int;
    pub fn gl_dev_free(ctx: *mut gl_ctx, p: *mut c_void);
    pub fn gl_copy(ctx: *mut gl_ctx, dst: *mut c_void, dst_space: c_int, src: *const c_void, src_space: c_int, bytes: usize) -> c_int;
    pub fn gl_fri_final_poly(ctx: *mut gl_ctx, oracles: *const *mut gl_commit, num_oracles: u32, batches: *const gl_fri_batch,
                             num_batches: u32, polys: *const gl_fri_poly, alpha: *const u64, rate_bits: u32,
                             lde_coeffs_out: *mut u64, lde_values_out: *mut u64, space: c_int) -> c_int;
    pub fn gl_fri_layer_commit(ctx: *mut gl_ctx, values_ext: *const u64, len: u64, arity_bits: u32, cap_height: u32,
                               cap_out: *mut u64, handle: *mut *mut gl_commit, space: c_int) -> c_int;
    // N2: bulk build of the sparse Merkle tree, the process proofs of a batch of `set` calls, `find` for a batch of queries
    pub fn gl_smt_find_batch(ctx: *mut gl_ctx, keys: *const u64, values: *const u64, m: u64, queries: *const u64, nq: u64,
                             proofs_out: *mut gl_smt_inclusion_hdr, sib_pool_out: *mut u64, sib_cap: u64, sib_off_out: *mut u64,
                             num_siblings_out: *mut u64, space: c_int) -> c_int;
    pub fn gl_smt_set_proofs(ctx: *mut gl_ctx, keys: *const u64, values: *const u64, m: u64, proofs_out: *mut gl_smt_proof_hdr,
                                sib_pool_out: *mut u64, sib_cap: u64, sib_off_out: *mut u64, num_siblings_out: *mut u64, space: c_int) -> c_int;
    pub fn gl_smt_build(ctx: *mut gl_ctx, keys: *const u64, values: *const u64, m: u64, root_out: *mut u64, nodes_out: *mut u64,
                        nodes_cap: u64, num_nodes_out: *mut u64, leaf_hashes_out: *mut u64, space: c_int) -> c_int;
    // N3: compute_quotient_polys on the resident oracles (plonk/prover.rs step 8)
    pub fn gl_quotient_polys(ctx: *mut gl_ctx, circuit: *const gl_circuit, gates: *const gl_gate, k_is: *const u64,
                             constants_sigmas: *mut gl_commit, wires: *mut gl_commit, zs_partial_products: *mut gl_commit,
                             public_inputs_hash: *const u64, betas: *const u64, gammas: *const u64, alphas: *const u64,
                             chunks_out: *mut u64, space: c_int) -> c_int;
    // all_wires_permutation_partial_products on the resident oracles (plonk/prover.rs, before the Z commit)
    pub fn gl_permutation_zs(ctx: *mut gl_ctx, circuit: *const gl_circuit, k_is: *const u64, constants_sigmas: *mut gl_commit,
                             wires: *mut gl_commit, betas: *const u64, gammas: *const u64, zs_partial_products_out: *mut u64,
                             space: c_int, grand_products_out: *mut u64) -> c_int;
    // plonk/prover.rs::prove from the witness on: every stage above chained by the transcript, one proof stream back
    pub fn gl_prove(ctx: *mut gl_ctx, circuit: *const gl_circuit, gates: *const gl_gate, k_is: *const u64,
                    constants_sigmas: *mut gl_commit, circuit_digest: *const u64, prm: *const gl_fri_params, wires: *const u64,
                    wires_cols: *const *const u64, space: c_int, public_inputs: *const u64, num_public_inputs: u32,
                    proof_out: *mut u64, proof_cap_words: u64, proof_words_out: *mut u64) -> c_int;
    // N1 in one call: prove_openings + fri_proof with the transcript on the device; fork-version switches
    pub fn gl_ctx_set_compat(ctx: *mut gl_ctx, flags: u32) -> c_int;
    pub fn gl_fri_proof_words(prm: *const gl_fri_params, oracle_columns: *const u32, num_oracles: u32, degree_bits: u32,
                              words_out: *mut u64) -> c_int;
    pub fn gl_fri_prove(ctx: *mut gl_ctx, oracles: *const *mut gl_commit, num_oracles: u32, batches: *const gl_fri_batch,
                        num_batches: u32, polys: *const gl_fri_poly, prm: *const gl_fri_params, challenger: *mut gl_challenger,
                        proof_out: *mut u64, proof_cap_words: u64, proof_words_out: *mut u64) -> c_int;
    // (e) multi-GPU: NCCL behind the ABI.  One process drives all GPUs of the box (id = null) or one rank per process.
    pub fn gl_group_unique_id(id_out: *mut u8) -> c_int;                                     // [GL_GROUP_ID_BYTES]
    pub fn gl_group_create(ctxs: *const *mut gl_ctx, nlocal: u32, rank0: u32, nranks: u32, id: *const u8, out: *mut *mut gl_group) -> c_int;
    pub fn gl_group_destroy(g: *mut gl_group);
    pub fn gl_group_last_error(g: *const gl_group) -> *const c_char;
    pub fn gl_group_info(g: *const gl_group, nlocal: *mut u32, rank0: *mut u32, nranks: *mut u32, nccl_version: *mut c_int) -> c_int;
    pub fn gl_group_commit_phase_ms(g: *const gl_group, out6: *mut f32) -> c_int;
    pub fn gl_group_commit_from_values(g: *mut gl_group, values: *const *const u64, log_n: u32, c: u32, rate_bits: u32, cap_height: u32,
                                       coeffs_out: *const *mut u64, cap_out: *const *mut u64, handles: *mut *mut gl_commit,
                                       space: c_int, flags: u32) -> c_int;
    pub fn gl_group_commit_from_coeffs(g: *mut gl_group, coeffs: *const *const u64, log_n: u32, c: u32, rate_bits: u32, cap_height: u32,
                                       cap_out: *const *mut u64, handles: *mut *mut gl_commit, space: c_int, flags: u32) -> c_int;
    pub fn gl_group_commit_open(g: *mut gl_group, handles: *const *mut gl_commit, leaf_indices: *const u64, k: u32,
                                rows_out: *const *mut u64, paths_out: *const *mut u64, space: c_int) -> c_int;
    pub fn gl_ctx_bind_host_numa(ctx: *mut gl_ctx) -> c_int;
}
#[repr(C)] pub struct gl_gate { pub kind: u32, pub num_ops: u32, pub selector_index: u32, pub group_start: u32, pub group_end: u32, pub reserved: u32 }
#[repr(C)] pub struct gl_circuit { pub degree_bits: u32, pub num_wires: u32, pub num_routed_wires: u32, pub num_constants: u32,
                                   pub num_selectors: u32, pub num_challenges: u32, pub quotient_degree_factor: u32, pub num_gates: u32 }
pub const GL_COMPAT_FRI_FINAL_POLY_TIMES_X: u32 = 1;
pub const GL_FRI_MAX_LAYERS: usize = 16;
#[repr(C)] pub struct gl_challenger { pub sponge_state: [u64; 12], pub input_buffer: [u64; 8], pub output_buffer: [u64; 8],
                                      pub input_len: u32, pub output_len: u32 }
#[repr(C)] pub struct gl_fri_params { pub rate_bits: u32, pub cap_height: u32, pub proof_of_work_bits: u32, pub num_query_rounds: u32,
                                      pub num_reduction_layers: u32, pub reduction_arity_bits: [u32; GL_FRI_MAX_LAYERS], pub flags: u32 }
pub enum gl_group {}
pub const GL_GROUP_ID_BYTES: usize = 128;
#[repr(C)] pub struct gl_smt_inclusion_hdr { pub root: [u64; 4], pub key: [u64; 4], pub value: [u64; 4], pub not_found_key: [u64; 4],
                                            pub not_found_value: [u64; 4], pub found: u32, pub is_old0: u32 }
#[repr(C)] pub struct gl_fri_batch { pub point: [u64; 2], pub first_poly: u32, pub num_polys: u32 }
#[repr(C)] pub struct gl_fri_poly { pub oracle_index: u32, pub polynomial_index: u32 }
