"""ctypes loader for libmacaw_b200.so (the C ABI declared in include/macaw_b200.h).

There is deliberately no fallback: if the library is missing it is built with nvcc, and if that fails the import
raises — the product path never silently routes through torch or the CPU oracle.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libmacaw_b200.so")

c_i32, c_i64, c_f32, c_vp, c_u32 = C.c_int32, C.c_int64, C.c_float, C.c_void_p, C.c_uint32


class GemmArgs(C.Structure):
    """Mirror of `mm_gemm_args` (include/macaw_b200.h)."""

    _fields_ = [
        ("M", c_i32), ("N", c_i32), ("K", c_i32), ("batch", c_i32), ("batch2", c_i32),
        ("A", c_vp), ("lda", c_i64), ("a_bs", c_i64), ("a_bs2", c_i64),
        ("B", c_vp), ("ldb", c_i64), ("b_bs", c_i64), ("b_bs2", c_i64), ("b_mn_major", c_i32),
        ("C", c_vp), ("ldc", c_i64), ("c_bs", c_i64), ("c_bs2", c_i64), ("c_fp32", c_i32),
        ("epi", c_i32), ("act", c_i32), ("alpha", c_f32),
        ("bias", c_vp), ("bias_bs", c_i64),
        ("row_scale", c_vp),
        ("residual", c_vp), ("ldr", c_i64), ("r_bs", c_i64), ("r_bs2", c_i64), ("res_row_mod", c_i32),
        ("rope_cos", c_vp), ("rope_sin", c_vp), ("rope_T", c_i32), ("rope_cols", c_i32), ("rope_pos", c_vp), ("c_trans", c_i32),
        ("a_fp16", c_i32), ("b_fp16", c_i32), ("c_fp16", c_i32),
        ("bias_rs", c_vp), ("bias2", c_vp), ("bias2_rs", c_vp), ("a_mn_major", c_i32),
        ("sumsq_out", c_vp), ("rs_sumsq", c_vp), ("rs_parts", c_i32), ("rs_eps", c_f32),
        ("sk_workspace", c_vp), ("sk_workspace_bytes", c_i64),
    ]


class GemmPlan(C.Structure):
    """Mirror of `mm_gemm_schedule` (include/macaw_b200.h), filled by mm_gemm_plan()."""

    _fields_ = [("block_n", c_i32), ("pairs", c_i32), ("m_tiles", c_i32), ("n_tiles", c_i32), ("k_blocks", c_i32),
                ("units", c_i64), ("workers", c_i32), ("grid", c_i32), ("waves", c_i32), ("group_m", c_i32),
                ("streamk_tiles", c_i32), ("smem_bytes", c_i32), ("vectorised_epilogue", c_i32)]


class ThinArgs(C.Structure):
    """mirror of mm_thin_args"""
    _fields_ = [("part", c_vp), ("splits", c_i32), ("N", c_i32), ("M", c_i32), ("ldp", c_i32), ("mode", c_i32),
                ("row_scale", c_vp), ("rs_sumsq", c_vp), ("rs_parts", c_i32), ("rs_K", c_i32), ("rs_eps", c_f32),
                ("residual", c_vp), ("ldr", c_i64), ("out", c_vp), ("ldo", c_i64), ("sumsq_out", c_vp),
                ("rope_cos", c_vp), ("rope_sin", c_vp), ("pos_dev", c_vp), ("E", c_i32), ("cache", c_vp),
                ("Tmax", c_i32), ("t0", c_i32), ("t0_dev", c_vp)]


class AttnArgs(C.Structure):
    """Mirror of `mm_attn_args` (include/macaw_b200.h)."""

    _fields_ = [
        ("q", c_vp), ("k", c_vp), ("v", c_vp), ("out", c_vp),
        ("B", c_i32), ("H", c_i32), ("Tq", c_i32), ("Tk", c_i32), ("head_dim", c_i32),
        ("q_bs", c_i64), ("q_ts", c_i64), ("q_hs", c_i64),
        ("k_bs", c_i64), ("k_ts", c_i64), ("k_hs", c_i64),
        ("v_bs", c_i64), ("v_ts", c_i64), ("v_hs", c_i64),
        ("o_bs", c_i64), ("o_ts", c_i64), ("o_hs", c_i64),
        ("key_mask", c_vp), ("causal", c_i32), ("scale", c_f32), ("impl", c_i32), ("tk_dev", c_vp),
    ]


class AlignArgs(C.Structure):
    """Mirror of `mm_align_args` (include/macaw_b200.h)."""

    _fields_ = [
        ("table", c_vp), ("V", c_i32), ("E", c_i32), ("ldt", c_i64),
        ("qt", c_vp), ("R", c_i32), ("ldq", c_i64),
        ("row_bias", c_vp), ("extra", c_vp), ("stat_stride", c_i64),
        ("out", c_vp), ("ldo", c_i64), ("p_sum_real", c_vp), ("p_extra", c_vp),
        ("P", c_vp), ("ldp", c_i64), ("workspace", c_vp), ("mode", c_i32), ("inv_l", c_vp),
    ]


class ImageArgs(C.Structure):
    """Mirror of `mm_image_args` (include/macaw_b200.h)."""

    _fields_ = [
        ("src", c_vp), ("ld", c_i64), ("row0", c_i32), ("n_rows", c_i32), ("out_h", c_i32), ("out_w", c_i32),
        ("bounds_h", c_vp), ("kk_h", c_vp), ("ksize_h", c_i32), ("bounds_v", c_vp), ("kk_v", c_vp), ("ksize_v", c_i32),
        ("mean", c_f32 * 3), ("std", c_f32 * 3), ("tmp", c_vp), ("out", c_vp), ("out_fp32", c_i32), ("out_u8", c_vp),
    ]


# name -> (restype, argtypes).  Every symbol declared in include/macaw_b200.h must appear here
# (tests/test_abi.py cross-checks the header against this table and against the built library).
SIGNATURES = {
    "mm_last_error": (C.c_char_p, []),
    "mm_abi_version": (c_i32, []),
    "mm_build_hash": (C.c_char_p, []),
    "mm_launch_count": (c_i64, []),
    "mm_launch_count_reset": (None, []),
    "mm_set_act_format": (None, [c_i32]),
    "mm_get_act_format": (c_i32, []),
    "mm_gemm_fwd": (c_i32, [C.POINTER(GemmArgs), c_vp]),
    "mm_gemm_plan": (c_i32, [C.POINTER(GemmArgs), C.POINTER(GemmPlan)]),
    "mm_splitk_reduce": (c_i32, [c_vp, c_i32, c_i32, c_i32, c_vp, c_vp, c_i64, c_i32, c_vp]),
    "mm_attn_fwd": (c_i32, [C.POINTER(AttnArgs), c_vp]),
    "mm_rmsnorm_fwd": (c_i32, [c_vp, c_vp, c_vp, c_i32, c_i32, c_f32, c_vp]),
    "mm_rms_rstd": (c_i32, [c_vp, c_vp, c_i32, c_i32, c_f32, c_vp]),
    "mm_layernorm_fwd": (c_i32, [c_vp, c_i64, c_vp, c_vp, c_vp, c_i64, c_i32, c_i32, c_f32, c_vp]),
    "mm_embed_gather": (c_i32, [c_vp, c_i32, c_i32, c_vp, c_i64, c_vp, c_i64, c_vp]),
    "mm_splice_prefix": (c_i32, [c_vp, c_vp, c_vp, c_i32, c_i32, c_i32, c_i32, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "mm_patchify": (c_i32, [c_vp, c_i32, c_i32, c_i32, c_i32, c_i32, c_vp, c_i64, c_vp]),
    "mm_transpose_pad": (c_i32, [c_vp, c_i32, c_i32, c_i32, c_i32, c_vp, c_vp]),
    "mm_add_rows": (c_i32, [c_vp, c_i64, c_vp, c_i64, c_i32, c_vp, c_i64, c_i32, c_i32, c_vp]),
    "mm_cast_bf16_f16": (c_i32, [c_vp, c_i64, c_vp, c_i64, c_i32, c_i32, c_vp]),
    "mm_copy_rows": (c_i32, [c_vp, c_i64, c_vp, c_i64, c_i32, c_i32, c_vp]),
    "mm_align_fwd": (c_i32, [C.POINTER(AlignArgs), c_vp]),
    "mm_align_workspace_bytes": (c_i64, [c_i32, c_i32]),
    "mm_align_softmax": (c_i32, [c_vp, c_i64, c_vp, c_vp, c_i64, c_vp, c_i64, c_vp, c_vp, c_i32, c_i32, c_vp]),
    "mm_align_ctx_fixup": (c_i32, [c_vp, c_i64, c_vp, c_vp, c_vp, c_vp, c_i32, c_i32, c_i32, c_vp]),
    "mm_kv_append": (c_i32, [c_vp, c_i64, c_i32, c_i32, c_i32, c_vp, c_i32, c_i32, c_vp, c_vp]),
    "mm_gemm_streamk_workspace_bytes": (c_i64, []),
    "mm_gemm_streamk_mode": (c_i32, [c_i32]),
    "mm_gemm_cg2_mode": (c_i32, [c_i32]),
    "mm_thin_fused": (c_i32, [C.POINTER(ThinArgs), c_vp]),
    "mm_thin_reduce": (c_i32, [c_vp, c_i32, c_i32, c_i32, c_i32, c_vp, c_vp, c_i64, c_vp, c_i64, c_vp]),
    "mm_argmax_rows": (c_i32, [c_vp, c_i64, c_i32, c_i32, c_vp, c_vp]),
    "mm_rope_rows": (c_i32, [c_vp, c_i64, c_i32, c_i32, c_vp, c_vp, c_i32, c_vp, c_vp]),
    "mm_swiglu_rows": (c_i32, [c_vp, c_i64, c_i32, c_i32, c_vp, c_i64, c_vp]),
    "mm_rmsnorm_bwd": (c_i32, [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_i32, c_i32, c_vp]),
    "mm_rmsnorm_bwd_parts": (c_i32, [c_i32]),
    "mm_swiglu_fwd": (c_i32, [c_vp, c_vp, c_vp, c_i64, c_vp]),
    "mm_swiglu_bwd": (c_i32, [c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_vp]),
    "mm_attn_softmax_bwd": (c_i32, [c_vp, c_vp, c_vp, c_vp, c_i32, c_i32, c_i32, c_i32, c_i64, c_f32, c_i32, c_vp, c_f32, c_vp,
                                    c_u32, c_vp]),
    "mm_attn_softmax_fwd": (c_i32, [c_vp, c_vp, c_i32, c_i32, c_i32, c_i32, c_i64, c_f32, c_i32, c_vp, c_f32, c_vp, c_u32, c_vp]),
    "mm_align_dropout_fwd": (c_i32, [c_vp, c_vp, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_i32, c_i32, c_f32, c_vp, c_u32, c_vp]),
    "mm_dropout_mask": (c_i32, [c_vp, c_i64, c_i32, c_i32, c_f32, c_vp, c_u32, c_vp]),
    "mm_ce_bwd": (c_i32, [c_vp, c_vp, c_vp, c_i32, c_i32, c_i32, c_vp, c_f32, c_vp, c_vp]),
    "mm_embed_scatter_add": (c_i32, [c_vp, c_i64, c_vp, c_i64, c_i32, c_i32, c_vp, c_vp]),
    "mm_colsum": (c_i32, [c_vp, c_i64, c_i32, c_i32, c_vp, c_vp]),
    "mm_adamw": (c_i32, [c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_f32, c_f32, c_f32, c_f32, c_f32, c_i32, c_vp, c_f32, c_vp]),
    "mm_grad_norm": (c_i32, [c_vp, c_i32, c_vp, c_vp, c_f32, c_i32, c_f32, c_i32, c_i32, c_i32, c_vp]),
    "mm_adamw_sched": (c_i32, [c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_f32, c_f32, c_f32, c_f32, c_vp, c_vp]),
    "mm_image_preprocess": (c_i32, [C.POINTER(ImageArgs), c_vp]),
    "mm_log_mel": (c_i32, [c_vp, c_i32, c_vp, c_vp, c_vp, c_vp, c_vp, c_i32, c_vp]),
    "mm_align_softmax_bwd": (c_i32, [c_vp, c_i64, c_vp, c_i64, c_vp, c_vp, c_vp, c_vp, c_f32, c_vp, c_vp, c_i64, c_vp, c_i32,
                                     c_i32, c_f32, c_vp, c_u32, c_vp]),
    "mm_head_weighted_colsum": (c_i32, [c_vp, c_i64, c_i32, c_vp, c_i64, c_i32, c_i32, c_i32, c_vp, c_vp]),
    "mm_window_gather_add": (c_i32, [c_vp, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, c_vp, c_vp]),
    "mm_cast_f16_bf16": (c_i32, [c_vp, c_i64, c_vp, c_i64, c_i32, c_i32, c_vp]),
    "mm_nccl_unique_id": (c_i32, [c_vp]),
    "mm_nccl_init": (c_i32, [c_vp, c_i32, c_i32]),
    "mm_nccl_allreduce": (c_i32, [c_vp, c_i64, c_i32, c_i32, c_vp]),
    "mm_nccl_destroy": (c_i32, []),
    "mm_ce_loss": (c_i32, [c_vp, c_vp, c_i32, c_i32, c_i32, c_vp, c_vp, c_vp]),
}

_lib = None
ABI_VERSION = 2


def load(build_if_missing: bool = True) -> C.CDLL:
    """Load (building first if necessary) the kernel library and bind every signature."""
    global _lib
    if _lib is not None:
        return _lib
    import importlib.util

    spec = importlib.util.spec_from_file_location("_macaw_b200_build", os.path.join(HERE, "build.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    want = mod.source_hash()
    # stale or missing library: (re)build under build.py's file lock (safe when several ranks arrive at once)
    if not os.path.exists(LIB_PATH) or mod.built_hash() != want:
        if not build_if_missing:
            raise RuntimeError(f"{LIB_PATH} is missing or older than csrc/; run `python macaw-llm_b200/build.py`")
        mod.build()
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError here == ABI drift; fail loudly
        fn.restype = res
        fn.argtypes = args
    got = lib.mm_build_hash().decode()
    if got != want or lib.mm_abi_version() != ABI_VERSION:
        raise RuntimeError(f"libmacaw_b200.so was built from other sources (library {got}, csrc {want}; ABI "
                           f"{lib.mm_abi_version()} vs {ABI_VERSION}): rebuild with `python macaw-llm_b200/build.py --force`")
    _lib = lib
    return lib


def last_error() -> str:
    return load().mm_last_error().decode("utf-8", "replace")
