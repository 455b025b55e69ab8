"""ctypes loader of libaccmsm.so.  There is no CPU fallback: a missing library is an ImportError-grade
failure and a missing GPU makes `Context()` raise."""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.environ.get("ACCMSM_SO") or os.path.join(HERE, "libaccmsm.so")   # ACCMSM_SO: development builds (tuning sweeps)

# every symbol include/accmsm.h declares (tests/test_abi.py checks the header against this list)
SYMBOLS = [
    "accmsm_init", "accmsm_init_multi", "accmsm_device_count", "accmsm_device_ctx", "accmsm_set_min_shard", "accmsm_destroy", "accmsm_host_alloc", "accmsm_host_free", "accmsm_strerror", "accmsm_last_error", "accmsm_set_window_bits", "accmsm_set_ipa_fold",
    "accmsm_kernel_launches", "accmsm_last_timings", "accmsm_stage_name",
    "accmsm_register_bases", "accmsm_release_bases", "accmsm_register_synthetic_bases", "accmsm_download_bases", "accmsm_precompute_bases", "accmsm_register_bases_compressed", "accmsm_serialize_bases",
    "accmsm_msm", "accmsm_msm_oneshot", "accmsm_msm_oneshot_batch", "accmsm_msm_batch", "accmsm_commit", "accmsm_msm_dev", "accmsm_msm_partial_dev", "accmsm_msm_partial", "accmsm_combine_partials_dev", "accmsm_combine_partials_batch_dev",
    "accmsm_ipa_final_key", "accmsm_ipa_check_final_key", "accmsm_ipa_final_key_partial_dev",
    "accmsm_ipa_open_begin", "accmsm_ipa_open_begin_combined", "accmsm_ipa_open_use_hiding_generator", "accmsm_ipa_open_round", "accmsm_ipa_open_fold", "accmsm_ipa_open_fold_round", "accmsm_ipa_open_finish", "accmsm_ipa_open_begin_shard", "accmsm_ipa_open_round_partial_dev", "accmsm_ipa_open_hide", "accmsm_ipa_open_hiding_challenge",
    "accmsm_compute_coeffs", "accmsm_combine_check_polys", "accmsm_poly_evaluate",
    "accmsm_hp_decide", "accmsm_hp_decide_partial_dev", "accmsm_hp_product_poly_comm", "accmsm_hp_product_poly_comm_partial_dev", "accmsm_csr_matvec_commit_partial_dev", "accmsm_register_csr", "accmsm_release_csr", "accmsm_csr_matvec_commit",
    "accmsm_nark_prove_zk", "accmsm_nark_verify", "accmsm_nark_as_decide",
    "accmsm_hp_prove_begin", "accmsm_hp_prove_product_poly_comm", "accmsm_hp_prove_finish", "accmsm_hp_prove_abort",
    "accmsm_vec_hadamard", "accmsm_vec_scale", "accmsm_vec_lincomb", "accmsm_vec_tvecs", "accmsm_csr_matvec",
]

_lib = None


class AccmsmError(RuntimeError):
    pass


def load() -> C.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(SO_PATH):
        raise AccmsmError(
            f"{SO_PATH} is missing: build the CUDA extension first (python -m accumulation_b200.build). "
            "accumulation_b200 has no CPU path.")
    lib = C.CDLL(SO_PATH)
    for name in SYMBOLS:
        getattr(lib, name)  # raises AttributeError if the ABI and the header diverge
    lib.accmsm_strerror.restype = C.c_char_p
    lib.accmsm_last_error.restype = C.c_char_p
    lib.accmsm_stage_name.restype = C.c_char_p
    lib.accmsm_kernel_launches.restype = C.c_uint64
    lib.accmsm_last_error.argtypes = [C.c_void_p]
    lib.accmsm_kernel_launches.argtypes = [C.c_void_p]
    lib.accmsm_destroy.argtypes = [C.c_void_p]
    lib.accmsm_destroy.restype = None
    lib.accmsm_device_ctx.restype = C.c_void_p
    lib.accmsm_device_ctx.argtypes = [C.c_void_p, C.c_int]
    lib.accmsm_device_count.argtypes = [C.c_void_p]
    lib.accmsm_host_alloc.restype = C.c_void_p
    lib.accmsm_host_alloc.argtypes = [C.c_size_t]
    lib.accmsm_host_free.argtypes = [C.c_void_p]
    lib.accmsm_host_free.restype = None
    _lib = lib
    return lib
