"""ctypes loader for the C-ABI library (pir_b200/lib/libpirb200.so, built by `make` / __graft_entry__.build()).

There is no CPU fallback: if the library is missing the import fails loudly, and every compute entry point
returns status 13 (Internal) when no CUDA device is present.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libpirb200.so")

u64p = C.POINTER(C.c_uint64)
u32p = C.POINTER(C.c_uint32)

PIRB_MAX_MODULI = 9
PIRB_MAX_DIMS = 8
PIRB_N_STAGES = 6
STAGE_NAMES = ("expand", "sv_ntt", "scan", "row_intt", "upper_dims", "total")
DIST_STAGE_NAMES = ("expand", "exchange_tail", "first_subbatch_arrived", "multiply", "reduce", "total",
                    "x_ntt", "x_head_push", "x_repack", "x_row_push")


class pirb_params(C.Structure):
    _fields_ = [
        ("poly_modulus_degree", C.c_uint32),
        ("n_moduli", C.c_uint32),
        ("coeff_modulus", C.c_uint64 * PIRB_MAX_MODULI),
        ("plain_modulus", C.c_uint64),
        ("n_dims", C.c_uint32),
        ("dims", C.c_uint32 * PIRB_MAX_DIMS),
        ("num_pt", C.c_uint64),
        ("device", C.c_int32),
        ("shard_index", C.c_uint32),
        ("shard_count", C.c_uint32),
        ("use_ciphertext_multiplication", C.c_uint32),
    ]


# every symbol include/pir_b200.h declares: name -> (restype, argtypes)
SYMBOLS = {
    "pirb_last_error": (C.c_char_p, []),
    "pirb_ctx_create": (C.c_int, [C.POINTER(pirb_params), C.POINTER(C.c_void_p)]),
    "pirb_ctx_destroy": (None, [C.c_void_p]),
    "pirb_ct_limbs": (C.c_uint64, [C.c_void_p]),
    "pirb_pt_limbs": (C.c_uint64, [C.c_void_p]),
    "pirb_key_limbs": (C.c_uint64, [C.c_void_p]),
    "pirb_expansion_ratio": (C.c_uint32, [C.c_void_p]),
    "pirb_reply_cts": (C.c_uint64, [C.c_void_p]),
    "pirb_dim_sum": (C.c_uint64, [C.c_void_p]),
    "pirb_query_cts": (C.c_uint64, [C.c_void_p]),
    "pirb_shard_pt_begin": (C.c_uint64, [C.c_void_p]),
    "pirb_shard_pt_count": (C.c_uint64, [C.c_void_p]),
    "pirb_db_size": (C.c_uint64, [C.c_void_p]),
    "pirb_db_load_coeff": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64]),
    "pirb_db_load_items": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32]),
    "pirb_db_load_ntt": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64]),
    "pirb_db_read_ntt": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64]),
    "pirb_db_fill_random": (C.c_int, [C.c_void_p, C.c_uint64]),
    "pirb_keys_load": (C.c_int, [C.c_void_p, u32p, C.c_uint32, C.c_void_p, C.POINTER(C.c_void_p)]),
    "pirb_keys_destroy": (None, [C.c_void_p]),
    "pirb_substitute": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32]),
    "pirb_mul_inv_pow_x": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p]),
    "pirb_expand": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_int, C.c_void_p]),
    "pirb_db_multiply": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, u64p]),
    "pirb_answer": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint64, C.c_void_p]),
    "pirb_answer_multi": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), C.c_void_p, C.c_uint32, C.c_uint64, C.c_void_p]),
    "pirb_answer_multi_dev": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), C.c_void_p, C.c_uint32, C.c_uint64, C.c_void_p,
                                        C.c_void_p]),
    "pirb_relin_keys_load": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(C.c_void_p)]),
    "pirb_reply_polys": (C.c_uint32, [C.c_void_p, C.c_int]),
    "pirb_db_multiply_ct": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_uint64, u32p]),
    "pirb_answer_ct": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint64, C.c_void_p]),
    "pirb_answer_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint64, C.c_void_p, C.c_void_p]),
    "pirb_answer_partial_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint64, C.c_void_p,
                                          C.c_void_p]),
    "pirb_expand_ntt_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint64, C.c_void_p, C.c_void_p]),
    "pirb_multiply_partial_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p]),
    "pirb_reduce_finish_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint64, C.c_uint32, C.c_void_p,
                                         C.c_void_p]),
    "pirb_dist_create": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p, C.POINTER(C.c_void_p)]),
    "pirb_dist_open_ipc": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32]),
    "pirb_dist_attach": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), C.c_uint32, C.c_uint32]),
    "pirb_dist_prepare": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32]),
    "pirb_dist_answer_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint64, C.c_void_p, C.c_void_p]),
    "pirb_dist_answer": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint64, C.c_void_p]),
    "pirb_dist_status": (C.c_int, [C.c_void_p]),
    "pirb_dist_stage_ms": (C.c_int, [C.c_void_p, C.POINTER(C.c_float)]),
    "pirb_scan_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p]),
    "pirb_sync": (C.c_int, [C.c_void_p]),
    "pirb_debug_stamps": (C.c_int, [C.c_void_p, u64p, C.c_uint64]),
    "pirb_set_profiling": (C.c_int, [C.c_void_p, C.c_int]),
    "pirb_get_stage_ms": (C.c_int, [C.c_void_p, C.POINTER(C.c_float)]),
    "pirb_last_scan_ms": (C.c_int, [C.c_void_p, C.POINTER(C.c_float)]),
    "pirb_last_launch_count": (C.c_uint64, [C.c_void_p]),
    "pirb_scan_bytes": (C.c_uint64, [C.c_void_p, C.c_uint32]),
    "pirb_host_alloc": (C.c_int, [C.c_uint64, C.POINTER(C.c_void_p)]),
    "pirb_host_free": (None, [C.c_void_p]),
    "pirb_calculate_dimensions": (None, [C.c_uint32, C.c_uint32, u32p]),
    "pirb_next_power_two": (C.c_uint64, [C.c_uint64]),
    "pirb_ceil_log2": (C.c_uint32, [C.c_uint32]),
    "pirb_log2": (C.c_uint32, [C.c_uint32]),
    "pirb_plain_modulus_batching": (C.c_uint64, [C.c_uint32, C.c_uint32]),
    "pirb_bfv_default_coeff_modulus": (C.c_int, [C.c_uint32, u64p, C.c_uint32]),
}

_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                "pir_b200: %s not found. Build it with `make` (or __graft_entry__.build()). "
                "There is no CPU fallback." % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(L, name)  # AttributeError if the library does not export a declared symbol
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def last_error():
    return lib().pirb_last_error().decode("utf-8", "replace")
