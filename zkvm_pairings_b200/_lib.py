"""ctypes loader for libzkpair.so -- the C ABI of include/zkpair.h.

There is no CPU fallback: a missing library or missing CUDA device raises.
"""
from __future__ import annotations

import ctypes
import os

HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.environ.get("ZKPAIR_LIB", os.path.join(HERE, "libzkpair.so"))

c_u64p = ctypes.c_void_p
c_u8p = ctypes.c_void_p

# name -> (restype, argtypes); every symbol include/zkpair.h declares
SYMBOLS = {
    "zkp_device_count": (ctypes.c_int32, []),
    "zkp_ctx_create": (ctypes.c_int32, [ctypes.c_void_p, ctypes.c_int, ctypes.POINTER(ctypes.c_void_p)]),
    "zkp_ctx_destroy": (None, [ctypes.c_void_p]),
    "zkp_ctx_num_devices": (ctypes.c_int32, [ctypes.c_void_p]),
    "zkp_last_error": (ctypes.c_char_p, []),
    "zkp_version": (ctypes.c_char_p, []),
    "zkp_tower_op_batch": (ctypes.c_int32, [ctypes.c_void_p, ctypes.c_int32, c_u64p, c_u64p, c_u64p, c_u8p, ctypes.c_size_t]),
    "zkp_fp_mul_batch": (ctypes.c_int32, [ctypes.c_void_p, c_u64p, c_u64p, c_u64p, ctypes.c_size_t]),
    "zkp_sys_bigint": (ctypes.c_int32, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint32, ctypes.c_void_p, ctypes.c_void_p]),
    "zkp_syscall_fp_mulmod": (ctypes.c_int32, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]),
    "zkp_fp12_mul_batch": (ctypes.c_int32, [ctypes.c_void_p, c_u64p, c_u64p, c_u64p, ctypes.c_size_t]),
    "zkp_fp12_mul_by_014_batch": (ctypes.c_int32, [ctypes.c_void_p, c_u64p, c_u64p, c_u64p, ctypes.c_size_t]),
    "zkp_miller_loop_batch": (ctypes.c_int32, [ctypes.c_void_p, c_u64p, c_u8p, c_u64p, c_u8p, ctypes.c_size_t, c_u64p]),
    "zkp_final_exp_batch": (ctypes.c_int32, [ctypes.c_void_p, c_u64p, ctypes.c_size_t, c_u64p]),
    "zkp_pairing_batch": (ctypes.c_int32, [ctypes.c_void_p, c_u64p, c_u8p, c_u64p, c_u8p, ctypes.c_size_t, c_u64p]),
    "zkp_multi_miller_loop_batch": (ctypes.c_int32, [ctypes.c_void_p, c_u64p, c_u8p, c_u64p, c_u8p, ctypes.c_size_t, ctypes.c_int32, c_u64p]),
    "zkp_multi_pairing_batch": (ctypes.c_int32, [ctypes.c_void_p, c_u64p, c_u8p, c_u64p, c_u8p, ctypes.c_size_t, ctypes.c_int32, c_u64p, c_u8p]),
    "zkp_multi_miller_product": (ctypes.c_int32, [ctypes.c_void_p, c_u64p, c_u8p, c_u64p, c_u8p, ctypes.c_size_t, c_u64p, c_u64p]),
    "zkp_pairing_dev": (ctypes.c_int32, [ctypes.c_void_p, ctypes.c_int32, ctypes.c_int32, c_u64p, c_u8p, c_u64p, c_u8p, ctypes.c_size_t,
                                         ctypes.c_int32, c_u64p, c_u64p, c_u8p, ctypes.c_void_p, ctypes.c_void_p]),
    "zkp_tower_op_dev": (ctypes.c_int32, [ctypes.c_void_p, ctypes.c_int32, ctypes.c_int32, c_u64p, c_u64p, c_u64p, c_u8p, ctypes.c_void_p,
                                          ctypes.c_size_t, ctypes.c_void_p]),
    "zkp_product_scratch_elems": (ctypes.c_size_t, [ctypes.c_size_t]),
    "zkp_fp12_product_dev": (ctypes.c_int32, [ctypes.c_void_p, ctypes.c_int32, c_u64p, ctypes.c_size_t, c_u64p, c_u64p, ctypes.c_void_p, ctypes.c_void_p]),
    "zkp_gen_points_dev": (ctypes.c_int32, [ctypes.c_void_p, ctypes.c_int32, ctypes.c_uint64, ctypes.c_uint64, ctypes.c_size_t,
                                            c_u64p, c_u8p, c_u64p, c_u8p, ctypes.c_void_p]),
    "zkp_gen_points": (ctypes.c_int32, [ctypes.c_void_p, ctypes.c_uint64, ctypes.c_uint64, ctypes.c_size_t, c_u64p, c_u8p, c_u64p, c_u8p]),
    "zkp_g2_prepare_batch": (ctypes.c_int32, [ctypes.c_void_p, c_u64p, ctypes.c_size_t, c_u64p]),
    "zkp_g2_prepare_dev": (ctypes.c_int32, [ctypes.c_void_p, ctypes.c_int32, c_u64p, ctypes.c_size_t, c_u64p, ctypes.c_void_p, ctypes.c_void_p]),
    "zkp_multi_pairing_prepared_batch": (ctypes.c_int32, [ctypes.c_void_p, c_u64p, c_u8p, c_u64p, c_u8p, ctypes.c_size_t, ctypes.c_int32,
                                                          c_u64p, c_u8p, ctypes.c_int32, c_u64p, c_u8p]),
    "zkp_multi_pairing_prepared_dev": (ctypes.c_int32, [ctypes.c_void_p, ctypes.c_int32, c_u64p, c_u8p, c_u64p, c_u8p, ctypes.c_size_t,
                                                        ctypes.c_int32, c_u64p, c_u8p, ctypes.c_int32, c_u64p, c_u8p, ctypes.c_void_p,
                                                        ctypes.c_void_p]),
    "zkp_fp_from_bytes_batch": (ctypes.c_int32, [ctypes.c_void_p, c_u8p, ctypes.c_size_t, c_u64p, c_u8p]),
    "zkp_fp_to_bytes_batch": (ctypes.c_int32, [ctypes.c_void_p, c_u64p, ctypes.c_size_t, c_u8p]),
    "zkp_fp_bytes_dev": (ctypes.c_int32, [ctypes.c_void_p, ctypes.c_int32, ctypes.c_int32, ctypes.c_void_p, ctypes.c_void_p, c_u8p,
                                          ctypes.c_size_t, ctypes.c_void_p]),
    "zkp_g1_check_batch": (ctypes.c_int32, [ctypes.c_void_p, c_u64p, c_u8p, ctypes.c_size_t, c_u8p]),
    "zkp_g2_check_batch": (ctypes.c_int32, [ctypes.c_void_p, c_u64p, c_u8p, ctypes.c_size_t, c_u8p]),
    "zkp_g1_mul_batch": (ctypes.c_int32, [ctypes.c_void_p, c_u64p, c_u8p, c_u64p, ctypes.c_size_t, c_u64p, c_u8p]),
    "zkp_g2_mul_batch": (ctypes.c_int32, [ctypes.c_void_p, c_u64p, c_u8p, c_u64p, ctypes.c_size_t, c_u64p, c_u8p]),
    "zkp_g1_add_batch": (ctypes.c_int32, [ctypes.c_void_p, c_u64p, c_u8p, c_u64p, c_u8p, ctypes.c_size_t, c_u64p, c_u8p]),
    "zkp_g2_add_batch": (ctypes.c_int32, [ctypes.c_void_p, c_u64p, c_u8p, c_u64p, c_u8p, ctypes.c_size_t, c_u64p, c_u8p]),
    "zkp_g1_msm": (ctypes.c_int32, [ctypes.c_void_p, c_u64p, c_u8p, c_u64p, ctypes.c_size_t, c_u64p, c_u8p, c_u8p]),
    "zkp_g2_msm": (ctypes.c_int32, [ctypes.c_void_p, c_u64p, c_u8p, c_u64p, ctypes.c_size_t, c_u64p, c_u8p, c_u8p]),
    "zkp_g1_msm_scratch_bytes": (ctypes.c_size_t, [ctypes.c_size_t]),
    "zkp_g2_msm_scratch_bytes": (ctypes.c_size_t, [ctypes.c_size_t]),
    "zkp_g1_msm_dev": (ctypes.c_int32, [ctypes.c_void_p, ctypes.c_int32, c_u64p, c_u8p, c_u64p, ctypes.c_size_t, c_u64p, c_u8p, c_u8p,
                                        ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]),
    "zkp_g2_msm_dev": (ctypes.c_int32, [ctypes.c_void_p, ctypes.c_int32, c_u64p, c_u8p, c_u64p, ctypes.c_size_t, c_u64p, c_u8p, c_u8p,
                                        ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]),
    "zkp_groth16_vk_create": (ctypes.c_int32, [ctypes.c_void_p, c_u64p, c_u64p, c_u64p, c_u64p, c_u64p, c_u8p, ctypes.c_int32,
                                               ctypes.POINTER(ctypes.c_void_p)]),
    "zkp_groth16_vk_destroy": (None, [ctypes.c_void_p]),
    "zkp_groth16_verify_batch": (ctypes.c_int32, [ctypes.c_void_p, ctypes.c_void_p, c_u64p, c_u8p, c_u64p, ctypes.c_size_t, c_u8p]),
    "zkp_groth16_scratch_bytes": (ctypes.c_size_t, [ctypes.c_size_t]),
    "zkp_groth16_verify_dev": (ctypes.c_int32, [ctypes.c_void_p, ctypes.c_int32, ctypes.c_void_p, c_u64p, c_u8p, c_u64p, ctypes.c_size_t,
                                                c_u8p, ctypes.c_void_p, ctypes.c_void_p]),
    "zkp_kzg_setup_create": (ctypes.c_int32, [ctypes.c_void_p, c_u64p, ctypes.POINTER(ctypes.c_void_p)]),
    "zkp_kzg_setup_destroy": (None, [ctypes.c_void_p]),
    "zkp_kzg_verify_batch": (ctypes.c_int32, [ctypes.c_void_p, ctypes.c_void_p, c_u64p, c_u8p, c_u64p, ctypes.c_size_t, c_u8p]),
    "zkp_kzg_scratch_bytes": (ctypes.c_size_t, [ctypes.c_size_t]),
    "zkp_kzg_verify_dev": (ctypes.c_int32, [ctypes.c_void_p, ctypes.c_int32, ctypes.c_void_p, c_u64p, c_u8p, c_u64p, ctypes.c_size_t, c_u8p,
                                            ctypes.c_void_p, ctypes.c_void_p]),
    "zkp_kzg_verify_blob_batch": (ctypes.c_int32, [ctypes.c_void_p, ctypes.c_void_p, c_u8p, c_u64p, c_u8p, ctypes.c_size_t, c_u8p, c_u64p]),
    "zkp_kzg_blob_scratch_bytes": (ctypes.c_size_t, [ctypes.c_size_t]),
    "zkp_kzg_verify_blob_dev": (ctypes.c_int32, [ctypes.c_void_p, ctypes.c_int32, ctypes.c_void_p, c_u8p, c_u64p, c_u8p, ctypes.c_size_t,
                                                 c_u8p, c_u64p, ctypes.c_void_p, ctypes.c_void_p]),
    "zkp_kzg_setup_create_prover": (ctypes.c_int32, [ctypes.c_void_p, c_u64p, c_u64p, ctypes.POINTER(ctypes.c_void_p)]),
    "zkp_kzg_blob_to_commitment_batch": (ctypes.c_int32, [ctypes.c_void_p, ctypes.c_void_p, c_u8p, ctypes.c_size_t, c_u64p, c_u8p, c_u8p]),
    "zkp_kzg_compute_proof_batch": (ctypes.c_int32, [ctypes.c_void_p, ctypes.c_void_p, c_u8p, c_u64p, ctypes.c_size_t, c_u64p, c_u8p, c_u64p,
                                                     c_u8p]),
    "zkp_kzg_compute_blob_proof_batch": (ctypes.c_int32, [ctypes.c_void_p, ctypes.c_void_p, c_u8p, c_u64p, c_u8p, ctypes.c_size_t, c_u64p,
                                                          c_u8p, c_u8p, c_u64p]),
    "zkp_kzg_prover_scratch_bytes": (ctypes.c_size_t, [ctypes.c_size_t]),
    "zkp_kzg_blob_to_commitment_dev": (ctypes.c_int32, [ctypes.c_void_p, ctypes.c_int32, ctypes.c_void_p, c_u8p, ctypes.c_size_t, c_u64p, c_u8p,
                                                        c_u8p, ctypes.c_void_p]),
    "zkp_kzg_compute_proof_dev": (ctypes.c_int32, [ctypes.c_void_p, ctypes.c_int32, ctypes.c_void_p, c_u8p, c_u64p, ctypes.c_size_t, c_u64p,
                                                   c_u8p, c_u64p, c_u8p, ctypes.c_void_p, ctypes.c_void_p]),
    "zkp_kzg_compute_blob_proof_dev": (ctypes.c_int32, [ctypes.c_void_p, ctypes.c_int32, ctypes.c_void_p, c_u8p, c_u64p, c_u8p, ctypes.c_size_t,
                                                        c_u64p, c_u8p, c_u8p, c_u64p, ctypes.c_void_p, ctypes.c_void_p]),
    "zkp_kzg_setup_create_cells": (ctypes.c_int32, [ctypes.c_void_p, c_u64p, c_u64p, c_u64p, ctypes.POINTER(ctypes.c_void_p)]),
    "zkp_kzg_compute_cells_batch": (ctypes.c_int32, [ctypes.c_void_p, ctypes.c_void_p, c_u8p, ctypes.c_size_t, c_u8p, c_u8p]),
    "zkp_kzg_compute_cells_and_proofs_batch": (ctypes.c_int32, [ctypes.c_void_p, ctypes.c_void_p, c_u8p, ctypes.c_size_t, c_u8p, c_u64p, c_u8p,
                                                                c_u8p]),
    "zkp_kzg_verify_cell_batch": (ctypes.c_int32, [ctypes.c_void_p, ctypes.c_void_p, c_u64p, c_u8p, c_u64p, c_u8p, c_u64p, c_u8p, ctypes.c_size_t,
                                                   c_u8p]),
    "zkp_kzg_cells_proofs_scratch_bytes": (ctypes.c_size_t, [ctypes.c_size_t]),
    "zkp_kzg_verify_cell_scratch_bytes": (ctypes.c_size_t, [ctypes.c_size_t]),
    "zkp_kzg_compute_cells_dev": (ctypes.c_int32, [ctypes.c_void_p, ctypes.c_int32, ctypes.c_void_p, c_u8p, ctypes.c_size_t, c_u8p, c_u8p,
                                                   ctypes.c_void_p]),
    "zkp_kzg_compute_cells_and_proofs_dev": (ctypes.c_int32, [ctypes.c_void_p, ctypes.c_int32, ctypes.c_void_p, c_u8p, ctypes.c_size_t, c_u8p,
                                                              c_u64p, c_u8p, c_u8p, ctypes.c_void_p, ctypes.c_void_p]),
    "zkp_kzg_verify_cell_dev": (ctypes.c_int32, [ctypes.c_void_p, ctypes.c_int32, ctypes.c_void_p, c_u64p, c_u8p, c_u64p, c_u8p, c_u64p, c_u8p,
                                                 ctypes.c_size_t, c_u8p, ctypes.c_void_p, ctypes.c_void_p]),
    "zkp_kzg_recover_cells_batch": (ctypes.c_int32, [ctypes.c_void_p, ctypes.c_void_p, c_u64p, c_u8p, c_u64p, ctypes.c_size_t, c_u8p, c_u8p]),
    "zkp_kzg_recover_cells_and_proofs_batch": (ctypes.c_int32, [ctypes.c_void_p, ctypes.c_void_p, c_u64p, c_u8p, c_u64p, ctypes.c_size_t, c_u8p,
                                                                c_u64p, c_u8p, c_u8p]),
    "zkp_kzg_recover_cells_dev": (ctypes.c_int32, [ctypes.c_void_p, ctypes.c_int32, ctypes.c_void_p, c_u64p, c_u8p, c_u64p, ctypes.c_size_t, c_u8p,
                                                   c_u8p, ctypes.c_void_p]),
    "zkp_kzg_recover_cells_and_proofs_dev": (ctypes.c_int32, [ctypes.c_void_p, ctypes.c_int32, ctypes.c_void_p, c_u64p, c_u8p, c_u64p,
                                                              ctypes.c_size_t, c_u8p, c_u64p, c_u8p, c_u8p, ctypes.c_void_p, ctypes.c_void_p]),
    "zkp_imad_peak": (ctypes.c_int32, [ctypes.c_void_p, ctypes.c_int32, ctypes.c_int32, ctypes.POINTER(ctypes.c_double)]),
    "zkp_launch_count": (ctypes.c_uint64, [ctypes.c_void_p]),
    "zkp_set_kernel_timing": (ctypes.c_int32, [ctypes.c_void_p, ctypes.c_int32]),
    "zkp_last_kernel_ms": (ctypes.c_int32, [ctypes.c_void_p, ctypes.c_int32, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_uint64)]),
}

ZKP_OK = 0
ZKP_ERR_INVALID_ARG = -1
ZKP_ERR_CUDA = -2
ZKP_ERR_NONCANONICAL = -3
ZKP_ERR_NO_DEVICE = -4
ZKP_ERR_TOO_MANY_PAIRS = -5

_lib = None


def lib_path() -> str:
    return _SO


def load():
    """Loads libzkpair.so and binds every declared symbol.  Raises if the library is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(_SO):
        raise RuntimeError(
            "libzkpair.so not found at %s -- build it with `python -m zkvm_pairings_b200.build` "
            "(there is no CPU fallback)" % _SO)
    lib = ctypes.CDLL(_SO)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)   # AttributeError if the library does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib
