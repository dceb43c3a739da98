"""ctypes binding of liblime_b200.so (the C ABI declared in include/lime_b200.h).

There is deliberately no fallback: if the shared library is missing, or no CUDA device is visible
when a compute entry point is called, the error is raised to the caller.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("LIME_B200_LIB") or os.path.join(_HERE, "liblime_b200.so")   # the override selects an experiment build

c_float_p = C.c_void_p      # device pointers travel as integers (tensor.data_ptr())
c_int_p = C.c_void_p


class LimeNewsCache(C.Structure):
    _fields_ = [
        ("hist_rows", C.c_void_p), ("cand_rows", C.c_void_p), ("hist_tab", C.c_void_p),
        ("cand_tab", C.c_void_p), ("gate_bias", C.c_void_p), ("un_prefix", C.c_void_p),
        ("topic_table", C.c_void_p), ("cand16", C.c_void_p), ("ctab16", C.c_void_p), ("news_meta", C.c_void_p),
        ("hist_vg", C.c_void_p), ("htab_vg", C.c_void_p),
        ("news_num", C.c_int32), ("num_buckets", C.c_int32), ("user_nodes", C.c_int32), ("num_topics", C.c_int32),
        ("tab_gw_absmax", C.c_float), ("sigmoid_alpha", C.c_float), ("penalty_beta", C.c_float),
        ("use_lifetime_weighting", C.c_int32), ("use_expired_penalty", C.c_int32),
        ("topic_logit_absmax", C.c_float), ("tc_tables_ok", C.c_int32), ("tab_replicas", C.c_int32),
    ]


class LimeImpressions(C.Structure):
    _fields_ = [
        ("hist_news", C.c_void_p), ("hist_mask", C.c_void_p), ("hist_fresh", C.c_void_p),
        ("hist_life", C.c_void_p), ("cand_news", C.c_void_p), ("cand_fresh", C.c_void_p),
        ("cand_life", C.c_void_p), ("cand_remaining", C.c_void_p), ("unit_imp", C.c_void_p), ("unit_pair0", C.c_void_p),
        ("unit_count", C.c_void_p), ("num_units", C.c_int32), ("max_history", C.c_int32),
        ("tile_c", C.c_int32),
    ]


# name -> (restype, argtypes); every symbol include/lime_b200.h declares
P, I64, I32, F32 = C.c_void_p, C.c_int64, C.c_int32, C.c_float
_LINEAR = [P, I64, P, I64, P, P, I64, P, I64, I64, C.c_int, C.c_int, C.c_int, P]
PROTOTYPES = {
    "lime_abi_version": (C.c_int, []),
    "lime_last_error": (C.c_char_p, []),
    "lime_device_count": (C.c_int, []),
    "lime_launch_count": (I64, []),
    "lime_launch_count_reset": (None, []),
    "lime_bucketize": (C.c_int, [P, I64, C.c_int, P, P]),
    "lime_linear": (C.c_int, _LINEAR),
    "lime_linear_bf16": (C.c_int, _LINEAR),
    "lime_gemm_strided": (C.c_int, [P, I64, I64, P, I64, I64, P, I64, C.c_int, C.c_int, C.c_int, F32, P]),
    "lime_linear_x3_tma": (C.c_int, [P, P, I64, P, P, I64, P, P, I64, P, I64, I64, I32, I32, I32, F32, I32, P]),
    "lime_linear_x3_pairs_tma": (C.c_int, [P, P, I64, P, P, I64, P, P, P, I64, F32, I64, I32, I32, I32, F32, I32, P]),
    "lime_linear_bf16_tma": (C.c_int, [P, I64, P, I64, P, P, I64, P, I64, I32, I64, I32, I32, I32, F32, I32, P]),
    "lime_split_bf16_pairs": (C.c_int, [P, I64, I64, I32, P, P, I32, F32, I32, P]),
    "lime_cast_bf16_colsum": (C.c_int, [P, I64, I64, I32, P, I32, P, P]),
    "lime_embed_pe_bf16": (C.c_int, [P, I64, P, I64, C.c_int, C.c_int, P, P, P, I32, P]),
    "lime_mha_bf16": (C.c_int, [P, I64, P, I64, I64, C.c_int, C.c_int, C.c_int, P]),
    "lime_embed_pe_pairs": (C.c_int, [P, I64, P, I64, C.c_int, C.c_int, P, P, P, P, I32, F32, P]),
    "lime_layernorm_pairs": (C.c_int, [P, I64, P, P, P, I64, P, P, I32, F32, I64, C.c_int, F32, P]),
    "lime_layernorm_bf16": (C.c_int, [P, I64, P, P, P, I64, P, I32, I64, C.c_int, F32, P]),
    "lime_embed_pe": (C.c_int, [P, I64, P, I64, C.c_int, C.c_int, P, P, P]),
    "lime_mha": (C.c_int, [P, P, I64, C.c_int, C.c_int, C.c_int, F32, C.c_uint64, I64, P]),
    "lime_layernorm": (C.c_int, [P, I64, P, P, P, I64, I64, C.c_int, F32, P]),
    "lime_layernorm_meanpool": (C.c_int, [P, P, P, P, I64, I64, C.c_int, C.c_int, F32, P]),
    "lime_topic_rep": (C.c_int, [P, P, P, P, P, P, I64, P, I64, C.c_int, P]),
    "lime_intent_pool": (C.c_int, [P, P, P, P, I64, I64, C.c_int, C.c_int, P]),
    "lime_content_fuse": (C.c_int, [P, P, P, P, P, P, I64, C.c_int, C.c_int, C.c_int, P, I64, P]),
    "lime_bucket_pairs": (C.c_int, [P, P, C.c_int, C.c_int, P, P]),
    "lime_scale_rows": (C.c_int, [P, I64, P, F32, C.c_int, C.c_int, P]),
    "lime_prefix_rows": (C.c_int, [P, I64, C.c_int, C.c_int, P]),
    "lime_row_absmax": (C.c_int, [P, I64, I64, C.c_int, P, I64, P]),
    "lime_score_impressions": (C.c_int, [C.POINTER(LimeNewsCache), C.POINTER(LimeImpressions), I64, I32,
                                         I64, I32, P, P, P]),
    "lime_score_long_scratch_ints": (I64, [I32, I32]),
    "lime_score_long_work_floats": (I64, [I64, I32, I32]),
    "lime_score_impressions_long": (C.c_int, [C.POINTER(LimeNewsCache), C.POINTER(LimeImpressions), C.POINTER(LimeImpressions), I32, I64,
                                              I32, I64, I32, I64, I32, P, P, P, P]),
    "lime_split_f16_pairs": (C.c_int, [P, I64, I64, I32, F32, P, P, I64, P]),
    "lime_cache_write_rows": (C.c_int, [P, P, I64, P, P, P, P, P, P, I64, P]),
    "lime_score_phase_clocks": (C.c_int, [P]),
    "lime_score_smem_bytes": (I64, [I32, I32]),
    "lime_score_configure": (C.c_int, [I32, F32]),
    "lime_explain_pairs": (C.c_int, [C.POINTER(LimeNewsCache), C.POINTER(LimeImpressions), I32, P, P, P, P, P, P, P, P]),
    "lime_score_scratch_ints": (I64, [I32]),
    "lime_score_tile_c": (I32, [I32]),
    "lime_sizeof_news_cache": (I64, []),
    "lime_sizeof_impressions": (I64, []),
    "lime_topic_pair_table": (C.c_int, [P, I64, P, I64, I32, P, P]),
    "lime_rank_metrics": (C.c_int, [P, P, P, I64, P, P, P]),
    "lime_metrics_reduce": (C.c_int, [P, I64, P, P]),
    "lime_pool_topk_scratch_bytes": (I64, [I32, I64, I32]),
    "lime_pool_topk": (C.c_int, [P, I32, I64, P, P, P, P, P, I32, I32, P, P, P, P, P]),
    "lime_pool_rank_scratch_bytes": (I64, [I32, I32]),
    "lime_pool_rank_metrics": (C.c_int, [P, I32, I64, P, P, P, P, P, I32, P, I32, P, I32, P, P, P, P, P, P]),
    "lime_gemm": (C.c_int, [P, I64, C.c_int, P, I64, C.c_int, P, I64, I64, C.c_int, I64, F32, C.c_int, P]),
    "lime_gemm_bf16": (C.c_int, [P, I64, C.c_int, P, I64, C.c_int, P, I64, I64, C.c_int, I64, F32, C.c_int, P]),
    "lime_gemm_bf16_tn_tma": (C.c_int, [P, I64, P, I64, P, I64, I32, I32, I64, F32, I32, P]),
    "lime_act_bwd": (C.c_int, [P, I64, P, I64, P, I64, I64, C.c_int, C.c_int, P]),
    "lime_col_sum": (C.c_int, [P, I64, I64, C.c_int, P, P]),
    "lime_layernorm_bwd": (C.c_int, [P, I64, P, P, I64, C.c_int, P, I64, P, P, I64, C.c_int, F32, P]),
    "lime_gather_rows": (C.c_int, [P, I64, I64, P, I64, C.c_int, P, I64, P]),
    "lime_scatter_add_rows": (C.c_int, [P, I64, P, I64, C.c_int, P, I64, I64, P]),
    "lime_scatter_add_rows_sorted": (C.c_int, [P, I64, P, P, I64, C.c_int, P, I64, I64, P]),
    "lime_mha_bwd": (C.c_int, [P, P, P, I64, C.c_int, C.c_int, C.c_int, F32, C.c_uint64, I64, P]),
    "lime_mha_fwd_bf16": (C.c_int, [P, P, I64, C.c_int, C.c_int, C.c_int, F32, C.c_uint64, I64, P]),
    "lime_mha_x3": (C.c_int, [P, P, P, P, I32, F32, I64, C.c_int, C.c_int, C.c_int, F32, C.c_uint64, I64, P]),
    "lime_mha_bwd_bf16": (C.c_int, [P, P, P, I64, C.c_int, C.c_int, C.c_int, F32, C.c_uint64, I64, P]),
    "lime_intent_pool_bwd": (C.c_int, [P, P, P, P, I64, P, P, P, I64, C.c_int, C.c_int, P]),
    "lime_content_fuse_bwd": (C.c_int, [P, P, P, I64, I64, C.c_int, P, P, P]),
    "lime_dropout": (C.c_int, [P, I64, P, I64, I64, C.c_int, F32, C.c_uint64, P]),
    "lime_dropout_fused": (C.c_int, [P, I64, P, I64, P, I64, I64, C.c_int, F32, C.c_uint64, C.c_uint64, C.c_int, P]),
    "lime_embed_pe_dropout": (C.c_int, [P, I64, P, I64, C.c_int, C.c_int, P, F32, C.c_uint64, C.c_uint64, P, P]),
    "lime_ca_attention_fwd": (C.c_int, [P, P, P, I32, I32, I32, F32, C.c_uint64, P, P]),
    "lime_ca_attention_bwd": (C.c_int, [P, P, P, I32, I32, I32, F32, C.c_uint64, P, P, P, P]),
    "lime_row_scale_fwd": (C.c_int, [P, P, I64, C.c_int, P, P]),
    "lime_row_scale_bwd": (C.c_int, [P, P, P, I64, C.c_int, P, P, P]),
    "lime_gate_mix_fwd": (C.c_int, [P, P, P, I64, P, P]),
    "lime_gate_mix_bwd": (C.c_int, [P, P, P, P, I64, P, P, P, P]),
    "lime_sage_mean_fwd": (C.c_int, [P, P, I32, I32, I32, I32, P, P]),
    "lime_sage_mean_bwd": (C.c_int, [P, I32, I32, I32, I32, P, P, P]),
    "lime_add_row_bcast": (C.c_int, [P, P, I64, I32, C.c_int, P, P]),
    "lime_sum_over_h": (C.c_int, [P, I32, I32, C.c_int, P, P]),
    "lime_pool_fwd": (C.c_int, [P, P, P, I32, I32, I32, P, P, P]),
    "lime_pool_bwd": (C.c_int, [P, P, P, P, P, I32, I32, I32, P, P, P, P]),
    "lime_click_score_fwd": (C.c_int, [P, P, P, I64, F32, F32, I32, I32, P, P, P]),
    "lime_click_score_bwd": (C.c_int, [P, P, P, P, I64, P, P, P]),
}

ABI_VERSION = 8
_lib = None


class LimeError(RuntimeError):
    pass


def load():
    """Load the library once.  Raises if it has not been built (run __graft_entry__.build())."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise LimeError("liblime_b200.so not found at %s — build it with "
                        "`python -c 'import __graft_entry__ as g; g.build()'` "
                        "(there is no CPU fallback)" % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(lib, name)          # AttributeError here == header/library mismatch
        fn.restype = res
        fn.argtypes = args
    if (lib.lime_sizeof_news_cache() != C.sizeof(LimeNewsCache)
            or lib.lime_sizeof_impressions() != C.sizeof(LimeImpressions)):
        raise LimeError("ctypes struct layout does not match include/lime_b200.h")
    if lib.lime_abi_version() != ABI_VERSION:
        raise LimeError("liblime_b200.so ABI %d != binding ABI %d" % (lib.lime_abi_version(), ABI_VERSION))
    _lib = lib
    return lib


def check(code, what):
    if code != 0:
        msg = load().lime_last_error().decode("utf-8", "replace")
        raise LimeError("%s failed (code %d): %s" % (what, code, msg))


def require_device():
    lib = load()
    if lib.lime_device_count() <= 0:
        raise LimeError("no CUDA device visible: the LIME B200 path has no CPU fallback")
    return lib
