"""ctypes binding of libgl_b200.so (the C ABI of include/gl_b200.h).

The library is the product; this module only declares its signatures.  There is deliberately no
fallback: if the shared library is missing or no CUDA device is present, calls raise.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libgl_b200.so")

GL_OK, GL_E_ARG, GL_E_CUDA, GL_E_OOM, GL_E_STATE, GL_E_NCCL = 0, 1, 2, 3, 4, 5
GL_GROUP_ID_BYTES = 128
GL_HOST, GL_DEVICE = 0, 1
GL_COMMIT_STREAM_HASH = 1
GL_COMMIT_BLINDING = 2
GL_SALT_SIZE = 4

u64p = C.POINTER(C.c_uint64)
vp = C.c_void_p
u32 = C.c_uint32
u64 = C.c_uint64
cint = C.c_int


class SmtProofHdr(C.Structure):
    """gl_smt_proof_hdr == SparseMerkleProcessProof minus siblings (src/smt/proof/process.rs:12-23)."""

    _fields_ = [
        ("old_root", u64 * 4), ("old_key", u64 * 4), ("old_value", u64 * 4),
        ("new_root", u64 * 4), ("new_key", u64 * 4), ("new_value", u64 * 4),
        ("is_old0", u32), ("fnc", u32),
    ]


class SmtInclusionHdr(C.Structure):
    """gl_smt_inclusion_hdr == SparseMerkleInclusionProof minus siblings (src/smt/proof/inclusion.rs:5-33)."""

    _fields_ = [
        ("root", u64 * 4), ("key", u64 * 4), ("value", u64 * 4), ("not_found_key", u64 * 4), ("not_found_value", u64 * 4),
        ("found", u32), ("is_old0", u32),
    ]


class Gate(C.Structure):
    """gl_gate: one entry of CommonCircuitData.gates with its selector placement."""

    _fields_ = [("kind", u32), ("num_ops", u32), ("selector_index", u32), ("group_start", u32), ("group_end", u32), ("reserved", u32)]


class Circuit(C.Structure):
    """gl_circuit: the part of CommonCircuitData compute_quotient_polys reads."""

    _fields_ = [("degree_bits", u32), ("num_wires", u32), ("num_routed_wires", u32), ("num_constants", u32), ("num_selectors", u32),
                ("num_challenges", u32), ("quotient_degree_factor", u32), ("num_gates", u32)]


class Challenger(C.Structure):
    """gl_challenger: plonky2::iop::challenger::Challenger as plain data."""

    _fields_ = [("sponge_state", u64 * 12), ("input_buffer", u64 * 8), ("output_buffer", u64 * 8), ("input_len", u32), ("output_len", u32)]


GL_FRI_MAX_LAYERS = 16
GL_COMPAT_FRI_FINAL_POLY_TIMES_X = 1


class FriParams(C.Structure):
    """gl_fri_params: FriConfig + FriParams.reduction_arity_bits + compat flags."""

    _fields_ = [("rate_bits", u32), ("cap_height", u32), ("proof_of_work_bits", u32), ("num_query_rounds", u32),
                ("num_reduction_layers", u32), ("reduction_arity_bits", u32 * GL_FRI_MAX_LAYERS), ("flags", u32)]


class FriBatch(C.Structure):
    _fields_ = [("point", u64 * 2), ("first_poly", u32), ("num_polys", u32)]


class FriPoly(C.Structure):
    _fields_ = [("oracle_index", u32), ("polynomial_index", u32)]


# name -> (restype, argtypes); must list EVERY symbol include/gl_b200.h declares (tests check this)
SIGNATURES = {
    "gl_ctx_create": (cint, [cint, C.POINTER(vp)]),
    "gl_ctx_destroy": (None, [vp]),
    "gl_last_error": (C.c_char_p, [vp]),
    "gl_ctx_stream": (vp, [vp]),
    "gl_ctx_sync": (cint, [vp]),
    "gl_ctx_set_shard": (cint, [vp, u32, u32]),
    "gl_ctx_kernel_launches": (u64, [vp]),
    "gl_ctx_commit_phase_ms": (cint, [vp, C.POINTER(C.c_float)]),
    "gl_ctx_trim": (cint, [vp]),
    "gl_dev_alloc": (cint, [vp, C.c_size_t, C.POINTER(vp)]),
    "gl_dev_free": (None, [vp, vp]),
    "gl_copy": (cint, [vp, vp, cint, vp, cint, C.c_size_t]),
    "gl_host_alloc": (cint, [C.c_size_t, C.POINTER(vp)]),
    "gl_host_free": (None, [vp]),
    "gl_poseidon_permute_batch": (cint, [vp, vp, u64, cint]),
    "gl_poseidon_duplex_chain": (cint, [vp, vp, vp, u64]),
    "gl_poseidon_two_to_one_batch": (cint, [vp, vp, vp, vp, u64, cint]),
    "gl_poseidon_hash_no_pad_batch": (cint, [vp, vp, u32, u64, vp, cint]),
    "gl_smt_leaf_hash_batch": (cint, [vp, vp, vp, vp, u64, cint]),
    "gl_smt_verify_process_batch": (cint, [vp, vp, vp, vp, u64, vp, cint]),
    "gl_smt_build": (cint, [vp, vp, vp, u64, vp, vp, u64, u64p, vp, cint]),
    "gl_smt_find_batch": (cint, [vp, vp, vp, u64, vp, u64, vp, vp, u64, vp, C.POINTER(u64), cint]),
    "gl_smt_set_proofs": (cint, [vp, vp, vp, u64, vp, vp, u64, vp, C.POINTER(u64), cint]),
    "gl_merkle_verify_batch": (cint, [vp, vp, u32, vp, vp, u32, vp, u32, u64, vp, cint]),
    "gl_merkle_build": (cint, [vp, vp, u64, u32, u32, vp, vp, cint]),
    "gl_fft_batch": (cint, [vp, vp, u32, u32, cint]),
    "gl_ifft_batch": (cint, [vp, vp, u32, u32, cint]),
    "gl_coset_fft_batch": (cint, [vp, vp, u32, u32, u64, cint]),
    "gl_coset_ifft_batch": (cint, [vp, vp, u32, u32, u64, cint]),
    "gl_commit_from_values": (cint, [vp, vp, u32, u32, u32, u32, vp, vp, C.POINTER(vp), cint]),
    "gl_commit_from_coeffs": (cint, [vp, vp, u32, u32, u32, u32, vp, C.POINTER(vp), cint]),
    "gl_commit_from_values_cols": (cint, [vp, vp, u32, u32, u32, u32, vp, vp, C.POINTER(vp)]),
    "gl_commit_from_coeffs_cols": (cint, [vp, vp, u32, u32, u32, u32, vp, C.POINTER(vp)]),
    "gl_commit_from_values_ex": (cint, [vp, vp, vp, u32, u32, u32, u32, u32, vp, vp, vp, C.POINTER(vp), cint]),
    "gl_commit_from_coeffs_ex": (cint, [vp, vp, vp, u32, u32, u32, u32, u32, vp, C.POINTER(vp), cint]),
    "gl_ctx_set_salt_seed": (cint, [vp, u64]),
    "gl_commit_leaf_len": (cint, [vp, C.POINTER(u32)]),
    "gl_commit_begin": (cint, [vp, u32, u32, u32, u32, C.POINTER(vp)]),
    "gl_commit_begin_ex": (cint, [vp, u32, u32, u32, u32, u32, C.POINTER(vp)]),
    "gl_commit_add_coeffs": (cint, [vp, u32, u32, vp, cint]),
    "gl_commit_finish": (cint, [vp, vp, cint]),
    "gl_commit_eval": (cint, [vp, vp, vp, cint]),
    "gl_commit_coeffs": (cint, [vp, vp, cint]),
    "gl_commit_download": (cint, [vp, vp, vp, cint]),
    "gl_commit_open": (cint, [vp, vp, u32, vp, vp, cint]),
    "gl_commit_get_lde_values": (cint, [vp, vp, u32, u64, vp, cint]),
    "gl_commit_info": (cint, [vp, C.POINTER(u32), C.POINTER(u32), C.POINTER(u32), C.POINTER(u32), C.POINTER(u64), C.POINTER(u64)]),
    "gl_commit_device_ptrs": (cint, [vp, C.POINTER(vp), C.POINTER(u64), C.POINTER(vp)]),
    "gl_commit_free": (None, [vp]),
    "gl_fri_layer_tree": (cint, [vp, vp, u64, u32, u32, vp, vp, cint]),
    "gl_fri_layer_commit": (cint, [vp, vp, u64, u32, u32, vp, C.POINTER(vp), cint]),
    "gl_fri_fold": (cint, [vp, vp, u64, u32, u64p, u64, vp, vp, cint]),
    "gl_fri_final_poly": (cint, [vp, vp, u32, vp, u32, vp, u64p, u32, vp, vp, cint]),
    "gl_pow_grind": (cint, [vp, u64p, u32, u32, u64p]),
    "gl_ctx_set_compat": (cint, [vp, u32]),
    "gl_fri_proof_words": (cint, [vp, vp, u32, u32, C.POINTER(u64)]),
    "gl_fri_prove": (cint, [vp, vp, u32, vp, u32, vp, vp, vp, vp, u64, C.POINTER(u64)]),
    "gl_quotient_polys": (cint, [vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, cint]),
    "gl_permutation_zs": (cint, [vp, vp, vp, vp, vp, vp, vp, vp, cint, vp]),
    "gl_prove": (cint, [vp, vp, vp, vp, vp, vp, vp, vp, vp, cint, vp, u32, vp, u64, C.POINTER(u64)]),
    "gl_group_unique_id": (cint, [vp]),
    "gl_group_create": (cint, [vp, u32, u32, u32, vp, C.POINTER(vp)]),
    "gl_group_destroy": (None, [vp]),
    "gl_group_last_error": (C.c_char_p, [vp]),
    "gl_group_info": (cint, [vp, C.POINTER(u32), C.POINTER(u32), C.POINTER(u32), C.POINTER(cint)]),
    "gl_group_commit_phase_ms": (cint, [vp, C.POINTER(C.c_float)]),
    "gl_group_commit_from_values": (cint, [vp, vp, u32, u32, u32, u32, vp, vp, vp, cint, u32]),
    "gl_group_commit_from_coeffs": (cint, [vp, vp, u32, u32, u32, u32, vp, vp, cint, u32]),
    "gl_group_commit_open": (cint, [vp, vp, vp, u32, vp, vp, cint]),
    "gl_ctx_bind_host_numa": (cint, [vp]),
}

_lib = None


def load() -> C.CDLL:
    """dlopen the in-tree library (build it first with plonky2-lib_b200/build.py or __graft_entry__.build())."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: run `python plonky2-lib_b200/build.py` (nvcc, sm_100a). "
                "There is no CPU or PyTorch fallback for this path."
            )
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib
