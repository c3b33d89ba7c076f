"""ctypes binding of libb200pir.so (include/b200pir.h).  There is no CPU fallback: if the CUDA
library is missing or cannot be loaded, importing this module raises."""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.path.join(_HERE, "libb200pir.so")


class B200PirError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("b200pir error %d: %s" % (code, msg))
        self.code = code


class CParams(C.Structure):
    _fields_ = [(k, C.c_uint64) for k in ("n", "nu_1", "nu_2", "p", "q2_bits", "t_gsw", "t_conv", "t_exp_left",
                                           "t_exp_right", "instances", "db_item_size", "version")] + \
               [("expand_queries", C.c_int32)]


def _load():
    if not os.path.exists(SO_PATH):
        raise ImportError("sdk_b200: %s not found — build it with `python -m sdk_b200.build` "
                          "(the product has no CPU path)" % SO_PATH)
    lib = C.CDLL(SO_PATH)
    vp, u64p, u32p, u8p, szp = C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_size_t)
    sig = {
        "b200pir_last_error": (C.c_char_p, []),
        "b200pir_device_count": (C.c_int, []),
        "b200pir_ctx_create": (C.c_int, [C.POINTER(CParams), C.c_int, C.POINTER(vp)]),
        "b200pir_ctx_destroy": (None, [vp]),
        "b200pir_ctx_set_stream": (C.c_int, [vp, vp]),
        "b200pir_ctx_synchronize": (C.c_int, [vp]),
        "b200pir_ctx_set_option": (C.c_int, [vp, C.c_char_p, C.c_int64]),
        "b200pir_ctx_reserve": (C.c_int, [vp, C.c_size_t, C.c_size_t]),
        "b200pir_ctx_sizes": (C.c_int, [vp, C.POINTER(C.c_uint64)] + [C.POINTER(C.c_uint64)] * 2),
        "b200pir_db_create": (C.c_int, [vp, C.c_uint64, C.c_uint64, C.POINTER(vp)]),
        "b200pir_db_destroy": (None, [vp]),
        "b200pir_db_upload_slice": (C.c_int, [vp, vp, C.c_uint64, u64p, C.c_size_t]),
        "b200pir_db_upload": (C.c_int, [vp, vp, u64p, C.c_size_t]),
        "b200pir_db_load_file": (C.c_int, [vp, vp, C.c_char_p]),
        "b200pir_db_load_raw_file": (C.c_int, [vp, vp, C.c_char_p]),
        "b200pir_db_upsert_item": (C.c_int, [vp, vp, C.c_uint64, C.c_uint64, u64p]),
        "b200pir_db_update_item_raw": (C.c_int, [vp, vp, C.c_uint64, u8p, C.c_size_t]),
        "b200pir_db_update_many_items": (C.c_int, [vp, vp, u8p, C.c_size_t, C.POINTER(C.c_uint64)]),
        "b200pir_db_fill_synthetic": (C.c_int, [vp, vp, C.c_uint64]),
        "b200pir_db_info": (C.c_int, [vp, C.POINTER(C.c_int), C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
        "b200pir_db_present_items": (C.c_int, [vp, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
        "b200pir_pp_create": (C.c_int, [vp, u64p, u64p, u64p, u64p, C.POINTER(vp)]),
        "b200pir_pp_create_from_bytes": (C.c_int, [vp, u8p, C.c_size_t, C.POINTER(vp)]),
        "b200pir_query_from_bytes": (C.c_int, [vp, u8p, C.c_size_t, u64p]),
        "b200pir_process_query_bytes": (C.c_int, [vp, vp, vp, u8p, C.c_size_t, C.c_size_t, u8p, szp]),
        "b200pir_pp_destroy": (None, [vp]),
        "b200pir_ntt_forward": (C.c_int, [vp, u64p, C.c_size_t]),
        "b200pir_ntt_inverse": (C.c_int, [vp, u64p, C.c_size_t]),
        "b200pir_ntt32_dev": (C.c_int, [vp, u32p, C.c_size_t, C.c_int]),
        "b200pir_ntt4096_dev": (C.c_int, [vp, u32p, C.c_size_t, C.c_int]),
        "b200pir_ntt4096": (C.c_int, [vp, u64p, C.c_size_t, C.c_int]),
        "b200pir_to_ntt": (C.c_int, [vp, u64p, u64p, C.c_size_t]),
        "b200pir_from_ntt": (C.c_int, [vp, u64p, u64p, C.c_size_t]),
        "b200pir_multiply_reg_by_database": (C.c_int, [vp, vp, C.c_uint64, u64p, u64p]),
        "b200pir_fold_ciphertexts": (C.c_int, [vp, u64p, C.c_size_t, u64p, u64p]),
        "b200pir_get_v_folding_neg": (C.c_int, [vp, u64p, u64p]),
        "b200pir_coefficient_expansion": (C.c_int, [vp, vp, u64p]),
        "b200pir_expand_query": (C.c_int, [vp, vp, u64p, u64p, u64p]),
        "b200pir_pack": (C.c_int, [vp, vp, u64p, u64p]),
        "b200pir_encode": (C.c_int, [vp, u64p, u8p, szp]),
        "b200pir_process_query": (C.c_int, [vp, vp, vp, u64p, u64p, u64p, u8p, szp]),
        "b200pir_process_query_batch": (C.c_int, [vp, vp, vp, u64p, C.c_size_t, u8p, szp]),
        "b200pir_process_queries": (C.c_int, [vp, vp, C.POINTER(vp), C.POINTER(vp), C.c_size_t, C.POINTER(vp)]),
        "b200pir_coalesce_stats": (C.c_int, [vp, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
        "b200pir_process_query_batch_dev": (C.c_int, [vp, vp, vp, u64p, C.c_size_t, u8p]),
        "b200pir_query_stage_a_dev": (C.c_int, [vp, vp, vp, u64p, C.c_size_t, u64p]),
        "b200pir_query_stage_b_dev": (C.c_int, [vp, vp, u64p, C.c_size_t, C.c_size_t, u8p]),
        "b200pir_expand_queries_dev": (C.c_int, [vp, vp, u64p, C.c_size_t, vp, u32p]),
        "b200pir_first_dim_fold_dev": (C.c_int, [vp, vp, vp, u32p, C.c_size_t, u32p]),
        "b200pir_query_image_bytes": (C.c_size_t, [vp]),
        "b200pir_expand_queries_images_dev": (C.c_int, [vp, vp, u64p, C.c_size_t, vp, u32p]),
        "b200pir_first_dim_fold_images_dev": (C.c_int, [vp, vp, vp, C.c_size_t, C.c_size_t, u32p, u32p]),
        "b200pir_finish_queries_dev": (C.c_int, [vp, vp, u32p, C.c_size_t, C.c_size_t, C.c_size_t, C.c_size_t, u32p, u8p]),
        "b200pir_last_stage_ms": (C.c_int, [vp, C.POINTER(C.c_double)]),
        "b200pir_kernel_launches": (C.c_ulonglong, []),
        "b200pir_peer_alloc": (C.c_int, [C.c_int, C.c_size_t, C.POINTER(vp), C.c_char_p]),
        "b200pir_peer_open": (C.c_int, [C.c_int, C.c_char_p, C.POINTER(vp)]),
        "b200pir_peer_close": (C.c_int, [C.c_int, vp]),
        "b200pir_peer_free": (C.c_int, [C.c_int, vp]),
        "b200pir_peer_copy_async": (C.c_int, [vp, vp, C.c_size_t, vp]),
        "b200pir_dpir_create": (C.c_int, [C.c_int, u32p, C.c_uint64, C.c_uint64, C.POINTER(vp)]),
        "b200pir_dpir_create_synthetic": (C.c_int, [C.c_int, C.c_uint64, C.c_uint64, C.c_uint64, C.POINTER(vp)]),
        "b200pir_dpir_destroy": (None, [vp]),
        "b200pir_dpir_setup": (C.c_int, [C.c_int, u32p, C.c_uint64, C.c_uint64, u32p, C.c_uint64, u32p, C.c_uint32, C.c_uint64,
                                         C.c_uint64, u32p, u32p, u32p, u32p]),
        "b200pir_dpir_matmul": (C.c_int, [C.c_int, u32p, C.c_uint64, C.c_uint64, u32p, C.c_uint64, u32p]),
        "b200pir_dpir_set_stream": (C.c_int, [vp, vp]),
        "b200pir_dpir_matvec_packed": (C.c_int, [vp, u32p, u32p]),
        "b200pir_dpir_matvec_packed_dev": (C.c_int, [vp, u32p, u32p, C.c_int]),
        "b200pir_dpir_matvec_packed_rows": (C.c_int, [vp, C.c_uint64, C.c_uint64, u32p, u32p]),
        "b200pir_dpir_matrix_mul_transposed_packed": (C.c_int, [C.c_int, u32p, C.c_uint64, C.c_uint64, u32p, C.c_uint64,
                                                                 C.c_uint64, u32p]),
        "b200pir_dpir_transpose_expand_concat_cols_squish": (C.c_int, [C.c_int, u32p, C.c_uint64, C.c_uint64, C.c_uint64,
                                                                        C.c_uint64, C.c_uint64, u32p, C.POINTER(C.c_uint64),
                                                                        C.POINTER(C.c_uint64)]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(lib, name)          # raises AttributeError if the .so does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    return lib, sorted(sig)


LIB, EXPORTED = _load()


def check(rc):
    if rc != 0:
        raise B200PirError(rc, LIB.b200pir_last_error().decode())
