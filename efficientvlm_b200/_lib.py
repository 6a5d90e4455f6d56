"""ctypes binding of libevlm_b200.so (C ABI declared in include/evlm.h).

There is deliberately NO fallback: if the shared library is missing, or a kernel is asked to run without a CUDA
device, this module raises.  Return codes follow include/evlm.h: <0 -> ValueError, >0 -> RuntimeError(cudaError).
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libevlm_b200.so")

BF16, F32 = 0, 1
ACT_NONE, ACT_QUICK_GELU, ACT_GELU_ERF = 0, 1, 2
GATE_NONE, GATE_PRE_ACT, GATE_POST_ACT = 0, 1, 2
EPI_FORWARD, EPI_ACT_BACKWARD = 0, 1

c_i32, c_i64, c_u32, c_u64, c_f, c_p = C.c_int32, C.c_int64, C.c_uint32, C.c_uint64, C.c_float, C.c_void_p


class GemmArgs(C.Structure):
    _fields_ = [
        ("M", c_i32), ("N", c_i32), ("K", c_i32),
        ("A", c_p), ("lda", c_i64), ("a_mn", c_i32),
        ("B", c_p), ("ldb", c_i64), ("b_mn", c_i32),
        ("D", c_p), ("ldd", c_i64), ("d_dtype", c_i32),
        ("epi_mode", c_i32),
        ("bias", c_p),
        ("alpha", c_f), ("alpha_cols", c_i32),
        ("act", c_i32),
        ("gate", c_p), ("gate_mode", c_i32),
        ("aux_out", c_p), ("ld_aux_out", c_i64),
        ("aux_in", c_p), ("ld_aux_in", c_i64),
        ("residual", c_p), ("ldr", c_i64), ("res_dtype", c_i32),
        ("dropout_p", c_f), ("dropout_seed", c_u64), ("dropout_stream", c_u32),
        ("splits", c_i32), ("accumulate", c_i32), ("max_ctas", c_i32),
        ("m_limit", c_p), ("n_limit", c_p), ("k_limit", c_p),
    ]


class AttnArgs(C.Structure):
    _fields_ = [
        ("B", c_i32), ("H", c_i32), ("Lq", c_i32), ("Lk", c_i32),
        ("q", c_p), ("ldq", c_i64), ("k", c_p), ("ldk", c_i64), ("v", c_p), ("ldv", c_i64),
        ("ctx", c_p), ("ldc", c_i64),
        ("probs", c_p), ("lse", c_p), ("key_mask", c_p), ("full_mask", c_p),
        ("causal", c_i32), ("causal_offset", c_i32), ("scale", c_f),
        ("head_z", c_p),
        ("dropout_p", c_f), ("dropout_seed", c_u64), ("dropout_stream", c_u32),
        ("dctx", c_p), ("lddc", c_i64), ("dprobs_ext", c_p),
        ("dq", c_p), ("lddq", c_i64), ("dk", c_p), ("lddk", c_i64), ("dv", c_p), ("lddv", c_i64),
        ("dhead_z", c_p), ("dkv_accum", c_p),
        ("kv_index", c_p), ("kv_batches", c_i32),
        ("pack_items", c_p), ("pack_groups", c_i32), ("pack_width", c_i32), ("pack_own_kv", c_i32),
        ("ldp", c_i64), ("dp_rowdot", c_p), ("kv_item_rows", c_i64), ("dp_kd_coef", c_p),
    ]


class MsePair(C.Structure):
    _fields_ = [("s", c_p), ("t", c_p), ("ds", c_p), ("n", c_i64), ("scale", c_f), ("s_dtype", c_i32), ("t_dtype", c_i32),
                ("pad", c_i32), ("rowdot", c_p), ("row_len", c_i64)]


class CastEntry(C.Structure):
    _fields_ = [("src", c_p), ("dst", c_p), ("rows", c_i64), ("cols", c_i64), ("ldd", c_i64)]


class AdamWGroup(C.Structure):
    _fields_ = [("p", c_p), ("g", c_p), ("m", c_p), ("v", c_p), ("p_bf16", c_p), ("n", c_i64), ("lr", c_f), ("beta1", c_f),
                ("beta2", c_f), ("eps", c_f), ("weight_decay", c_f), ("step", c_i32), ("pad", c_i32)]


# name -> (restype, argtypes).  Every symbol include/evlm.h declares is listed (tests check the export table).
PROTOTYPES = {
    "evlm_abi_version": (c_i32, []),
    "evlm_launch_count": (C.c_ulonglong, []),
    "evlm_reset_launch_count": (None, []),
    "evlm_gemm_bf16": (c_i32, [C.POINTER(GemmArgs), c_p]),
    "evlm_gemm_fp8": (c_i32, [C.POINTER(GemmArgs), c_p, c_p, c_p]),
    "evlm_quant_rows_e4m3": (c_i32, [c_p, c_i32, c_i64, c_i64, c_i64, c_p, c_i64, c_p, c_p]),
    "evlm_sgemm": (c_i32, [c_i32, c_i32, c_i32, c_f, c_p, c_i64, c_i32, c_p, c_i64, c_i32, c_f, c_p, c_i64, c_p, c_i32, c_p]),
    "evlm_dot": (c_i32, [c_p, c_p, c_i64, c_f, c_p, c_i32, c_p]),
    "evlm_cast_f32_to_bf16": (c_i32, [c_p, c_i64, c_p, c_i64, c_i64, c_i64, c_f, c_u64, c_u32, c_p]),
    "evlm_cast_table": (c_i32, [c_p, c_i32, c_p]),
    "evlm_greedy_select": (c_i32, [c_p, c_i64, c_i32, c_i32, c_p, c_i64, c_p, c_i32, c_p, c_p, c_p, c_p, c_p]),
    "evlm_cast_bf16_to_f32": (c_i32, [c_p, c_i64, c_p, c_i64, c_i64, c_i64, c_p]),
    "evlm_colsum": (c_i32, [c_p, c_i32, c_i64, c_i64, c_i64, c_p, c_i32, c_p]),
    "evlm_coldot": (c_i32, [c_p, c_p, c_i64, c_i64, c_i64, c_p, c_p]),
    "evlm_compact_index": (c_i32, [c_p, c_i32, c_p, c_p, c_p]),
    "evlm_gather_rows": (c_i32, [c_p, c_i64, c_i32, c_p, c_p, c_p, c_i64, c_i64, c_i64, c_p]),
    "evlm_gather_cols_bf16": (c_i32, [c_p, c_i64, c_p, c_p, c_p, c_i64, c_i64, c_i64, c_p]),
    "evlm_scatter_rows_add": (c_i32, [c_p, c_i64, c_p, c_p, c_p, c_i64, c_i64, c_i64, c_i32, c_p]),
    "evlm_scatter_cols_add": (c_i32, [c_p, c_i64, c_p, c_p, c_p, c_i64, c_i64, c_i64, c_i32, c_p]),
    "evlm_act_fwd": (c_i32, [c_p, c_i32, c_p, c_i32, c_i64, c_i32, c_p]),
    "evlm_act_bwd": (c_i32, [c_p, c_i32, c_p, c_i32, c_p, c_i32, c_i64, c_i32, c_p]),
    "evlm_im2col_patch": (c_i32, [c_p, c_p, c_i32, c_i32, c_i32, c_i32, c_p]),
    "evlm_vit_assemble_fwd": (c_i32, [c_p, c_p, c_p, c_p, c_i32, c_i32, c_i32, c_p]),
    "evlm_vit_assemble_bwd": (c_i32, [c_p, c_p, c_p, c_p, c_i32, c_i32, c_i32, c_p]),
    "evlm_bert_embed_fwd": (c_i32, [c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_i64, c_i32, c_i32, c_i32, c_i64, c_p]),
    "evlm_bert_embed_bwd": (c_i32, [c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_i64, c_i32, c_i32, c_i32, c_i64, c_p]),
    "evlm_layernorm_fwd": (c_i32, [c_p, c_i32, c_p, c_p, c_f, c_p, c_p, c_p, c_p, c_i64, c_i32, c_f, c_u64, c_u32, c_p]),
    "evlm_layernorm_bwd": (c_i32, [c_p, c_i32, c_p, c_i32, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_i64, c_i32, c_f, c_u64,
                                   c_u32, c_p]),
    "evlm_layernorm_bwd_ex": (c_i32, [c_p, c_i32, c_p, c_i32, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_i64, c_i32, c_f, c_u64,
                                      c_u32, c_f, c_u32, c_p, c_p]),
    "evlm_attention_fwd": (c_i32, [C.POINTER(AttnArgs), c_p]),
    "evlm_attention_bwd": (c_i32, [C.POINTER(AttnArgs), c_p]),
    "evlm_attention_bwd_workspace": (C.c_size_t, [C.POINTER(AttnArgs)]),
    "evlm_mse_pairs_fwd": (c_i32, [c_p, c_i32, c_p, c_p]),
    "evlm_mse_pairs_bwd": (c_i32, [c_p, c_i32, c_p, c_p]),
    "evlm_xent_fwd": (c_i32, [c_p, c_i64, c_i64, c_i32, c_p, c_i64, c_f, c_p, c_p, c_p]),
    "evlm_xent_bwd": (c_i32, [c_p, c_i64, c_i64, c_i32, c_p, c_i64, c_f, c_p, c_p, c_p, c_i64, c_i32, c_p]),
    "evlm_kl_fwd": (c_i32, [c_p, c_p, c_i64, c_i64, c_i64, c_i32, c_f, c_p, c_p, c_p, c_p]),
    "evlm_kl_bwd": (c_i32, [c_p, c_p, c_i64, c_i64, c_i64, c_i32, c_f, c_p, c_p, c_p, c_p, c_i64, c_i32, c_p]),
    "evlm_soft_xent_fwd": (c_i32, [c_p, c_i64, c_p, c_i64, c_i64, c_i32, c_p, c_p, c_p]),
    "evlm_soft_xent_bwd": (c_i32, [c_p, c_i64, c_p, c_i64, c_i64, c_i32, c_p, c_p, c_p, c_i64, c_i32, c_p]),
    "evlm_reduce_sum": (c_i32, [c_p, c_i64, c_f, c_p, c_i32, c_p]),
    "evlm_l2norm_fwd": (c_i32, [c_p, c_p, c_p, c_i64, c_i32, c_p]),
    "evlm_l2norm_bwd": (c_i32, [c_p, c_p, c_p, c_p, c_i64, c_i32, c_p]),
    "evlm_itm_sample_neg": (c_i32, [c_p, c_i64, c_p, c_p, c_p, c_i32, c_p]),
    "evlm_l0_sample_fwd": (c_i32, [c_p, c_p, c_p, c_i64, c_f, c_p]),
    "evlm_l0_sample_bwd": (c_i32, [c_p, c_p, c_p, c_p, c_i64, c_f, c_p]),
    "evlm_l0_expected_fwd": (c_i32, [c_p, c_i64, c_f, c_f, c_p, c_i32, c_p]),
    "evlm_l0_expected_bwd": (c_i32, [c_p, c_i64, c_f, c_f, c_p, c_p, c_p]),
    "evlm_l0_deterministic": (c_i32, [c_p, c_p, c_p, c_i32, c_i32, c_f, c_f, c_p]),
    "evlm_clamp_": (c_i32, [c_p, c_i64, c_f, c_f, c_p]),
    "evlm_sumsq": (c_i32, [c_p, c_i64, c_p, c_p]),
    "evlm_adamw_step": (c_i32, [C.POINTER(AdamWGroup), c_i32, c_p, c_p]),
    "evlm_clip_coef": (c_i32, [c_p, c_f, c_p, c_p]),
    "evlm_adamw_step_dev": (c_i32, [C.POINTER(AdamWGroup), c_i32, c_p, c_p, c_p]),
    "evlm_store_f32": (c_i32, [c_p, C.POINTER(C.c_float), c_i32, c_p]),
    "evlm_rng_bind": (c_i32, [c_p]),
    "evlm_index_add_rows": (c_i32, [c_p, c_p, c_p, c_i64, c_i64, c_p]),
    "evlm_index_fold_rows": (c_i32, [c_p, c_p, c_i64, c_i64, c_i64, c_p, c_p, c_p]),
    "evlm_rng_advance": (c_i32, [c_p, C.c_uint64, c_i32, c_p]),
    "evlm_beam_step": (c_i32, [c_p, c_i64, c_i32, c_i32, c_i32, c_i32, c_i32, c_f, C.c_double, c_i32, c_i64, c_i64, c_p, c_i64, c_p, c_p, c_p,
                               c_p, c_p, c_p, c_p, c_p, c_p]),
    "evlm_beam_finalize": (c_i32, [c_p, c_i64, c_p, c_p, c_i32, c_i32, c_i32, c_i32, C.c_double, c_i64, c_i64, c_p, c_p, c_p, c_p, c_p, c_p,
                                   c_p, c_p]),
    "evlm_kv_beam_reorder": (c_i32, [C.POINTER(c_p), c_i32, c_i32, c_i32, c_i64, c_i64, c_i32, c_p, c_p]),
}

ABI_VERSION = 9   # must equal EVLM_ABI_VERSION in include/evlm.h
_lib = None


def load():
    """Load the kernel library (idempotent).  Raises if it has not been built: there is no CPU path."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            "efficientvlm_b200: %s not found. Build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(or `make -C efficientvlm_b200/csrc`). There is no CPU / eager fallback." % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(lib, name)  # AttributeError here == ABI mismatch: fail loudly
        fn.restype = res
        fn.argtypes = args
    if lib.evlm_abi_version() != ABI_VERSION:
        raise RuntimeError("efficientvlm_b200: ABI version mismatch")
    _lib = lib
    return lib


def check(rc, what):
    if rc == 0:
        return
    if rc < 0:
        raise ValueError("%s: invalid argument / unsupported shape (evlm rc=%d)" % (what, rc))
    raise RuntimeError("%s: CUDA error %d" % (what, rc))
