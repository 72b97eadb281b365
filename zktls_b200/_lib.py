"""ctypes loader for libzkb200.so (the C-ABI declared in include/zkb200.h).

There is no CPU fallback: if the shared library is missing or no CUDA device is present, loading / zkb_init
raises.  Nothing in this package imports the CPU oracle.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.path.join(_HERE, "libzkb200.so")
_lib = None


class ZkbError(RuntimeError):
    pass


# every symbol include/zkb200.h declares (tests/test_abi_symbols.py checks the header against this list and the .so)
SYMBOLS = [
    "zkb_version", "zkb_free_error", "zkb_init", "zkb_init_on_stream", "zkb_destroy", "zkb_sync", "zkb_device_info", "zkb_device_count",
    "zkb_kernel_launches", "zkb_timer_start", "zkb_timer_stop",
    "zkb_alloc", "zkb_free", "zkb_host_alloc", "zkb_host_free", "zkb_memset0", "zkb_fill_u32", "zkb_h2d", "zkb_d2h", "zkb_d2d",
    "zkb_batch_interpolate_ntt", "zkb_zk_shift", "zkb_batch_interpolate_ntt_zk_shift", "zkb_batch_expand", "zkb_batch_evaluate_ntt",
    "zkb_batch_expand_into_evaluate_ntt", "zkb_batch_bit_reverse",
    "zkb_poseidon2_hash_rows", "zkb_poseidon2_hash_fold", "zkb_poseidon2_merkle_build",
    "zkb_batch_evaluate_any", "zkb_mix_poly_coeffs", "zkb_poly_divide", "zkb_combos_divide", "zkb_eltwise_sum_extelem", "zkb_fri_fold",
    "zkb_eltwise_add_elem", "zkb_eltwise_copy_elem", "zkb_eltwise_zeroize_elem", "zkb_gather_sample", "zkb_gather_rows", "zkb_prefix_products", "zkb_scatter",
    "zkb_eval_check", "zkb_eval_check_source", "zkb_eval_check_precompile", "zkb_accumulate",
    "zkb_prover_new", "zkb_prover_free", "zkb_prover_segment_begin", "zkb_prover_segment_finish", "zkb_prover_seal_words",
    "zkb_prover_seal_copy", "zkb_prover_root_count", "zkb_prover_roots_copy", "zkb_prove_segment", "zkb_prover_stage_traces",
    "zkb_prove_staged", "zkb_prover_stage_wait", "zkb_verify_segment",
    "zkb_program_new", "zkb_program_commit", "zkb_program_control_ids", "zkb_program_free", "zkb_prover_set_program",
    "zkb_session_new", "zkb_session_commit", "zkb_session_control_ids", "zkb_session_submit", "zkb_session_wait", "zkb_session_free",
    "zkb_poseidon254_hash_rows", "zkb_poseidon254_hash_fold", "zkb_poseidon254_merkle_build", "zkb_poseidon254_permute_host",
]


def lib():
    """Loads libzkb200.so; raises if it has not been built (python -m zktls_b200.build / __graft_entry__.build())."""
    global _lib
    if _lib is None:
        if not os.path.exists(SO_PATH):
            raise ZkbError(f"{SO_PATH} is missing: build it with `python zktls_b200/build.py` (there is no CPU fallback)")
        L = C.CDLL(SO_PATH)
        for name in SYMBOLS:
            fn = getattr(L, name)          # AttributeError if the .so does not export a declared symbol
            fn.restype = C.c_void_p        # const char* error (NULL == ok); kept as an address so it can be freed
        L.zkb_version.restype = C.c_char_p
        L.zkb_free_error.restype = None
        _lib = L
    return _lib


def check(err):
    if err:
        msg = C.cast(err, C.c_char_p).value.decode(errors="replace")
        lib().zkb_free_error(C.c_void_p(err))
        raise ZkbError(msg)
