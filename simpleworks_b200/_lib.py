"""ctypes loader for libswb200.so (the C ABI declared in include/swb200.h).

There is no CPU fallback: if the CUDA library is missing or fails to load, importing the
operators raises.  The library is built in-tree by `python -m simpleworks_b200.build`
(nvcc -gencode arch=compute_100a,code=sm_100a).
"""
from __future__ import annotations

import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# SWB_LIB points the loader at another build of the same library (A/B measurements of kernel variants)
LIB_PATH = os.environ.get("SWB_LIB") or os.path.join(_HERE, "libswb200.so")

# every symbol include/swb200.h declares; tests/test_abi.py checks the header against this list
# and that the built library exports each one.
SYMBOLS = [
    "swb_init", "swb_destroy", "swb_last_error", "swb_trim", "swb_set_stream", "swb_reset_stream", "swb_sync", "swb_device_info",
    "swb_launch_count", "swb_dev_alloc", "swb_dev_free", "swb_h2d", "swb_d2h",
    "swb_fr_mul_vec_dev", "swb_fr_add_vec_dev", "swb_fr_sub_vec_dev",
    "swb_fq_mul_vec_dev", "swb_fq_add_vec_dev", "swb_fq_sub_vec_dev",
    "swb_fr_batch_inverse_dev", "swb_measure_mul_peak", "swb_measure_imad_peak",
    "swb_profile_enable", "swb_profile_last",
    "swb_bases_load", "swb_bases_load_dev", "swb_bases_from_powers", "swb_bases_export", "swb_bases_precompute", "swb_bases_table_info",
    "swb_bases_len", "swb_bases_free",
    "swb_msm_g1", "swb_msm_g1_dev", "swb_msm_g1_fr_dev", "swb_msm_g1_fr", "swb_msm_g1_batch_dev", "swb_set_msm_shard", "swb_set_msm_peers", "swb_peer_copy_bytes", "swb_comm_unique_id", "swb_comm_init", "swb_comm_info", "swb_comm_sum_g1", "swb_comm_destroy", "swb_msm_plan", "swb_msm_set_window_bits", "swb_msm_set_table_policy", "swb_msm_set_pair_sums", "swb_msm_set_bucket_shard", "swb_g1_sum_jacobian",
    "swb_fixed_base_powers",
    "swb_ntt_fr", "swb_ntt_fr_dev", "swb_ntt_fr_batch_dev",
    "swb_rng_test_rng", "swb_rng_from_seed", "swb_rng_from_entropy", "swb_rng_next_u64", "swb_rng_free",
    "swb_r1cs_new", "swb_r1cs_builtin", "swb_r1cs_add_constraint", "swb_r1cs_set_assignment", "swb_r1cs_is_satisfied",
    "swb_r1cs_free",
    "swb_marlin_profile_enable", "swb_marlin_last_phases", "swb_marlin_universal_setup", "swb_srs_max_degree", "swb_srs_set_tune_after", "swb_srs_table_info", "swb_srs_free", "swb_marlin_index", "swb_pk_free", "swb_vk_free",
    "swb_marlin_prove", "swb_marlin_verify", "swb_marlin_verify_batch", "swb_bytes_free",
    "swb_vk_serialize", "swb_vk_deserialize", "swb_proof_deserialize", "swb_proof_serialize", "swb_proof_free", "swb_marlin_verify_proof", "swb_pk_serialize", "swb_pk_deserialize", "swb_r1cs_read", "swb_r1cs_write",
]

_lib = None


class SwbError(RuntimeError):
    pass


def load() -> ctypes.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise SwbError(
            f"{LIB_PATH} not found: build it with `python -m simpleworks_b200.build` "
            "(there is no CPU fallback for the Marlin hot path)")
    lib = ctypes.CDLL(LIB_PATH)
    vp, sz, i32, u32 = ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int, ctypes.c_uint32
    pvp = ctypes.POINTER(ctypes.c_void_p)
    sig = {
        "swb_init": (i32, [i32, pvp]),
        "swb_destroy": (None, [vp]),
        "swb_last_error": (ctypes.c_char_p, [vp]),
        "swb_trim": (i32, [vp]),
        "swb_set_stream": (i32, [vp, vp]),
        "swb_reset_stream": (i32, [vp]),
        "swb_sync": (i32, [vp]),
        "swb_device_info": (i32, [vp, ctypes.POINTER(i32), ctypes.POINTER(i32), ctypes.POINTER(i32), ctypes.POINTER(sz)]),
        "swb_launch_count": (ctypes.c_uint64, [vp]),
        "swb_dev_alloc": (i32, [vp, sz, pvp]),
        "swb_dev_free": (i32, [vp, vp]),
        "swb_h2d": (i32, [vp, vp, vp, sz]),
        "swb_d2h": (i32, [vp, vp, vp, sz]),
        "swb_fr_batch_inverse_dev": (i32, [vp, vp, sz]),
        "swb_measure_mul_peak": (i32, [vp, i32, i32, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_double)]),
        "swb_measure_imad_peak": (i32, [vp, i32, i32, ctypes.POINTER(ctypes.c_double)]),
        "swb_profile_enable": (i32, [vp, i32]),
        "swb_profile_last": (i32, [vp, ctypes.POINTER(ctypes.c_char_p), ctypes.POINTER(ctypes.c_double), i32, ctypes.POINTER(i32)]),
        "swb_bases_from_powers": (i32, [vp, vp, vp, sz, pvp]),
        "swb_bases_export": (i32, [vp, vp, sz, sz, vp]),
        "swb_bases_load": (i32, [vp, vp, sz, pvp]),
        "swb_bases_load_dev": (i32, [vp, vp, sz, pvp]),
        "swb_srs_set_tune_after": (i32, [vp, ctypes.c_long]),
        "swb_srs_table_info": (i32, [vp, ctypes.POINTER(i32), ctypes.POINTER(i32)]),
        "swb_marlin_profile_enable": (i32, [i32]),
        "swb_marlin_last_phases": (sz, [ctypes.c_char_p, sz]),
        "swb_bases_precompute": (i32, [vp, vp, i32]),
        "swb_bases_table_info": (i32, [vp, ctypes.POINTER(i32), ctypes.POINTER(i32)]),
        "swb_bases_len": (sz, [vp]),
        "swb_bases_free": (None, [vp]),
        "swb_msm_g1_batch_dev": (i32, [vp, vp, vp, vp, vp, sz, i32, vp]),
        "swb_set_msm_shard": (i32, [vp, i32, i32, vp, vp]),
        "swb_set_msm_peers": (i32, [vp, pvp, i32]),
        "swb_peer_copy_bytes": (ctypes.c_uint64, [vp]),
        "swb_comm_unique_id": (i32, [ctypes.c_char_p]),
        "swb_comm_init": (i32, [vp, ctypes.c_char_p, i32, i32]),
        "swb_comm_info": (i32, [vp, ctypes.POINTER(i32), ctypes.POINTER(i32)]),
        "swb_comm_sum_g1": (i32, [vp, vp, sz, vp]),
        "swb_comm_destroy": (i32, [vp]),
        "swb_msm_g1": (i32, [vp, vp, sz, vp, sz, vp]),
        "swb_msm_g1_dev": (i32, [vp, vp, sz, vp, sz, vp]),
        "swb_msm_g1_fr_dev": (i32, [vp, vp, sz, vp, sz, vp]),
        "swb_msm_g1_fr": (i32, [vp, vp, sz, vp, sz, vp]),
        "swb_rng_test_rng": (vp, []),
        "swb_rng_from_seed": (vp, [ctypes.c_char_p]),
        "swb_rng_from_entropy": (vp, []),
        "swb_rng_next_u64": (ctypes.c_uint64, [vp]),
        "swb_rng_free": (None, [vp]),
        "swb_r1cs_new": (vp, [sz, sz]),
        "swb_r1cs_builtin": (vp, [i32, sz, ctypes.c_uint64, ctypes.c_uint64]),
        "swb_r1cs_add_constraint": (i32, [vp, vp, vp, sz, vp, vp, sz, vp, vp, sz]),
        "swb_r1cs_set_assignment": (i32, [vp, vp, sz, vp, sz]),
        "swb_r1cs_is_satisfied": (i32, [vp]),
        "swb_r1cs_free": (None, [vp]),
        "swb_marlin_universal_setup": (i32, [vp, sz, sz, sz, vp, pvp]),
        "swb_srs_max_degree": (sz, [vp]),
        "swb_srs_free": (None, [vp]),
        "swb_marlin_index": (i32, [vp, vp, vp, pvp, pvp]),
        "swb_pk_free": (None, [vp]),
        "swb_vk_free": (None, [vp]),
        "swb_marlin_prove": (i32, [vp, vp, vp, vp, ctypes.POINTER(ctypes.POINTER(ctypes.c_uint8)), ctypes.POINTER(sz)]),
        "swb_marlin_verify": (i32, [vp, vp, vp, sz, ctypes.c_char_p, sz, vp, ctypes.POINTER(i32)]),
        "swb_marlin_verify_batch": (i32, [vp, sz, vp, vp, vp, vp, vp, vp, ctypes.POINTER(i32)]),
        "swb_bytes_free": (None, [ctypes.POINTER(ctypes.c_uint8)]),
        "swb_vk_serialize": (i32, [vp, ctypes.POINTER(ctypes.POINTER(ctypes.c_uint8)), ctypes.POINTER(sz)]),
        "swb_vk_deserialize": (vp, [ctypes.c_char_p, sz]),
        "swb_proof_deserialize": (vp, [ctypes.c_char_p, sz]),
        "swb_proof_serialize": (i32, [vp, ctypes.POINTER(ctypes.POINTER(ctypes.c_uint8)), ctypes.POINTER(sz)]),
        "swb_proof_free": (None, [vp]),
        "swb_marlin_verify_proof": (i32, [vp, vp, vp, sz, vp, vp, ctypes.POINTER(i32)]),
        "swb_pk_serialize": (i32, [vp, vp, vp, ctypes.POINTER(ctypes.POINTER(ctypes.c_uint8)), ctypes.POINTER(sz)]),
        "swb_pk_deserialize": (i32, [vp, ctypes.c_char_p, sz, pvp, pvp]),
        "swb_r1cs_read": (vp, [ctypes.c_char_p, sz]),
        "swb_r1cs_write": (i32, [vp, ctypes.POINTER(ctypes.POINTER(ctypes.c_uint8)), ctypes.POINTER(sz)]),
        "swb_msm_plan": (i32, [vp, sz, ctypes.POINTER(i32), ctypes.POINTER(i32)]),
        "swb_msm_set_window_bits": (i32, [vp, i32]),
        "swb_msm_set_table_policy": (i32, [vp, i32]),
        "swb_msm_set_pair_sums": (i32, [vp, i32]),
        "swb_msm_set_bucket_shard": (i32, [vp, i32, i32]),
        "swb_g1_sum_jacobian": (i32, [vp, vp, sz, vp]),
        "swb_fixed_base_powers": (i32, [vp, vp, vp, sz, vp]),
        "swb_ntt_fr": (i32, [vp, vp, u32, i32, i32]),
        "swb_ntt_fr_dev": (i32, [vp, vp, u32, i32, i32]),
        "swb_ntt_fr_batch_dev": (i32, [vp, vp, u32, sz, i32, i32]),
    }
    for name in ("swb_fr_mul_vec_dev", "swb_fr_add_vec_dev", "swb_fr_sub_vec_dev",
                 "swb_fq_mul_vec_dev", "swb_fq_add_vec_dev", "swb_fq_sub_vec_dev"):
        sig[name] = (i32, [vp, vp, vp, vp, sz])
    for name in SYMBOLS:
        fn = getattr(lib, name)          # AttributeError here = library/headers out of sync
        fn.restype, fn.argtypes = sig[name]
    _lib = lib
    return lib
