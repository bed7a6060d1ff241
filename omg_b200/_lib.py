"""ctypes binding of include/omg_b200.h.  The product path has no CPU fallback: if the CUDA library is
missing or a call fails this raises."""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("OMG_B200_LIB") or os.path.join(_HERE, "lib", "libomg_b200.so")  # override: A/B builds

OMG_MAX_A = 4
OMG_MAX_SEGS = 12
OMG_ATTN_MAX_ITEMS = 16
OMG_MAX_CONCEPTS = 8
EPI_NONE, EPI_GEGLU, EPI_SILU, EPI_QUICK_GELU, EPI_GELU, EPI_GELU_TANH = 0, 1, 2, 3, 4, 5
DTYPE_F16, DTYPE_BF16 = 0, 1


class View4(C.Structure):
    _fields_ = [("ptr", C.c_void_p), ("C", C.c_int32), ("W", C.c_int32), ("H", C.c_int32), ("B", C.c_int32),
                ("sw", C.c_int64), ("sh", C.c_int64), ("sb", C.c_int64)]


class Seg(C.Structure):
    _fields_ = [("a_idx", C.c_int32), ("dx", C.c_int32), ("dy", C.c_int32), ("a_c0", C.c_int32),
                ("k_len", C.c_int32), ("b_k0", C.c_int32), ("b_idx", C.c_int32)]


class GemmDesc(C.Structure):
    _fields_ = [("a", View4 * OMG_MAX_A), ("n_a", C.c_int32), ("segs", Seg * OMG_MAX_SEGS), ("n_segs", C.c_int32),
                ("w", C.c_void_p), ("N", C.c_int32), ("Ktot", C.c_int32), ("w2", C.c_void_p), ("K2tot", C.c_int32),
                ("d", View4), ("bias", C.c_void_p),
                ("rowvec", C.c_void_p), ("rowvec_ld", C.c_int32), ("residual", C.c_void_p),
                ("residual_ld", C.c_int32), ("epilogue", C.c_int32), ("block_n", C.c_int32),
                ("row_stats_out", C.c_void_p), ("row_stats_in", C.c_void_p), ("row_stats_parts", C.c_int32),
                ("row_stats_stride", C.c_int64), ("ln_dim", C.c_int32), ("ln_eps", C.c_float), ("col_c1", C.c_void_p), ("col_c2", C.c_void_p),
                ("n_col_groups", C.c_int32), ("col_group_end", C.c_int64 * 8), ("w_group_planes", C.c_int32), ("cta_pair", C.c_int32),
                ("col_stats_out", C.c_void_p), ("col_stats_rb0", C.c_int32), ("col_stats_rb_total", C.c_int32),
                ("residual_f32", C.c_void_p), ("residual_f32_ld", C.c_int64), ("out_f32", C.c_void_p), ("out_f32_ld", C.c_int64),
                ("dtype", C.c_int32)]


class AttnDesc(C.Structure):
    _fields_ = [("q", C.c_void_p), ("q_ld", C.c_int32), ("q_bs", C.c_int64), ("q_col0", C.c_int32),
                ("k", C.c_void_p), ("k_ld", C.c_int32), ("k_bs", C.c_int64), ("k_col0", C.c_int32),
                ("v", C.c_void_p), ("v_ld", C.c_int32), ("v_bs", C.c_int64), ("v_col0", C.c_int32),
                ("out", C.c_void_p), ("out_ld", C.c_int32), ("out_bs", C.c_int64), ("out_col0", C.c_int32),
                ("n_q", C.c_int32), ("n_kv", C.c_int32), ("heads", C.c_int32), ("head_dim", C.c_int32),
                ("n_items", C.c_int32),
                ("out_b", C.c_int32 * OMG_ATTN_MAX_ITEMS), ("q_b", C.c_int32 * OMG_ATTN_MAX_ITEMS),
                ("k_b", C.c_int32 * OMG_ATTN_MAX_ITEMS), ("v_b", C.c_int32 * OMG_ATTN_MAX_ITEMS),
                ("scale", C.c_float), ("out_weight", C.c_float), ("accumulate", C.c_int32), ("causal", C.c_int32)]


class FuseDesc(C.Structure):
    _fields_ = [("noise_main", C.c_void_p), ("noise_concept", C.c_void_p * OMG_MAX_CONCEPTS),
                ("mask", C.c_void_p * OMG_MAX_CONCEPTS), ("n_concepts", C.c_int32), ("guidance", C.c_float),
                ("sigma", C.c_float), ("sigma_next", C.c_float), ("latents", C.c_void_p),
                ("next_main_in", C.c_void_p), ("next_concept_in", C.c_void_p), ("latents_f16", C.c_void_p),
                ("HW", C.c_int32)]


# every symbol include/omg_b200.h declares: (restype, argtypes)
SYMBOLS = {
    "omg_gemm": (C.c_int, [C.POINTER(GemmDesc), C.c_void_p]),
    "omg_gemm_plan": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "omg_gemm_colstats_blocks": (C.c_int, [C.c_int, C.c_int]),
    "omg_colstats": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "omg_groupnorm_apply": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int,
                                      C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_float, C.c_int, C.c_void_p, C.c_void_p,
                                      C.c_void_p]),
    "omg_attention": (C.c_int, [C.POINTER(AttnDesc), C.c_void_p]),
    "omg_groupnorm": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                C.c_float, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "omg_groupnorm_bf16": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                     C.c_float, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "omg_layernorm": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_longlong, C.c_int, C.c_float,
                                C.c_void_p]),
    "omg_fuse_step": (C.c_int, [C.POINTER(FuseDesc), C.c_void_p]),
    "omg_ctx_mix": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "omg_axpy": (C.c_int, [C.c_void_p, C.c_void_p, C.c_float, C.c_void_p, C.c_longlong, C.c_void_p]),
    "omg_softmax_rows": (C.c_int, [C.c_void_p, C.c_longlong, C.c_int, C.c_longlong, C.c_float, C.c_void_p]),
    "omg_softmax_rows_bf16": (C.c_int, [C.c_void_p, C.c_longlong, C.c_int, C.c_longlong, C.c_float, C.c_void_p]),
    "omg_dwconv": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                             C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "omg_group1x1": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_longlong, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "omg_relu_linear_attention": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, C.c_void_p]),
    "omg_resize_bicubic": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "omg_plan_create": (C.c_void_p, []),
    "omg_plan_destroy": (None, [C.c_void_p]),
    "omg_plan_record_begin": (C.c_int, [C.c_void_p]),
    "omg_plan_record_end": (C.c_int, [C.c_void_p]),
    "omg_plan_length": (C.c_int, [C.c_void_p]),
    "omg_plan_clear": (C.c_int, [C.c_void_p]),
    "omg_plan_run": (C.c_int, [C.c_void_p, C.c_void_p]),
    "omg_last_error": (C.c_char_p, []),
    "omg_version": (C.c_char_p, []),
    "omg_launch_count": (C.c_uint64, []),
}

_lib = None


def load():
    """Load the C-ABI library (building is __graft_entry__.build()'s job).  Raises if it is missing."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(f"{LIB_PATH} not found: run `python -c 'import __graft_entry__ as g; g.build()'` "
                               "(there is no CPU fallback)")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SYMBOLS.items():
            if not hasattr(lib, name) and os.environ.get("OMG_B200_LIB"):
                continue   # A/B against an older build of the library: entry points added since are simply absent
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def check(status: int, what: str):
    if status != 0:
        raise RuntimeError(f"{what}: {load().omg_last_error().decode()}")


def launch_count() -> int:
    return int(load().omg_launch_count())
