"""ctypes binding of libvqa_b200.so (the C ABI declared in include/vqa_b200.h).

The shared library is built in-tree by `__graft_entry__.build()` / `python -m t2v_metrics_b200.build`. There is no
fallback: if the library is missing or does not export the ABI, importing the engine fails loudly.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

_HERE = Path(__file__).resolve().parent
LIB_PATH = _HERE / "libvqa_b200.so"

ABI_SYMBOLS = [
    "vqa_version", "vqa_create_clipt5", "vqa_bind_weights", "vqa_finalize_weights", "vqa_clipt5_workspace_bytes",
    "vqa_clipt5_score", "vqa_set_profile", "vqa_profile_read", "vqa_last_launch_count", "vqa_last_error", "vqa_destroy", "vqa_op_gemm_bf16",
    "vqa_op_lmhead_logprob", "vqa_op_attention_d64", "vqa_op_norm", "vqa_op_attention_d128",
    "vqa_create_qwen25vl", "vqa_qwen25vl_set_rope", "vqa_qwen25vl_workspace_bytes", "vqa_qwen25vl_score",
    "vqa_clip_preprocess_workspace_bytes", "vqa_clip_preprocess", "vqa_resample_table", "vqa_qwen_preprocess_plan",
    "vqa_qwen_preprocess", "vqa_clipt5_debug_layout", "vqa_qwen25vl_debug_layout", "vqa_set_gemm_schedule",
    "vqa_qwen25vl_topk", "vqa_op_gemm_bf16_normfuse",
    "vqa_qwen25vl_packed_workspace_bytes", "vqa_qwen25vl_score_packed", "vqa_debug_max_active_clusters", "vqa_op_attention_d128_ex", "vqa_op_gemm_bf16_grouped", "vqa_op_gemm_bf16_splitk",
    "vqa_qwen_video_preprocess_plan", "vqa_qwen_video_preprocess", "vqa_resample_table_tv",
]

VQA_DTYPE_BF16, VQA_DTYPE_F32, VQA_DTYPE_I32 = 0, 1, 2
VQA_RESAMPLE_PIL, VQA_RESAMPLE_TORCHVISION = 0, 1


class VqaClipT5Config(C.Structure):
    _fields_ = [
        ("image_size", C.c_int32), ("patch_size", C.c_int32), ("vit_hidden", C.c_int32), ("vit_heads", C.c_int32),
        ("vit_mlp", C.c_int32), ("vit_layers_run", C.c_int32), ("vit_ln_eps", C.c_float),
        ("d_model", C.c_int32), ("n_heads", C.c_int32), ("d_ff", C.c_int32), ("enc_layers", C.c_int32),
        ("dec_layers", C.c_int32), ("vocab", C.c_int32), ("rel_buckets", C.c_int32), ("rel_max_distance", C.c_int32),
        ("t5_ln_eps", C.c_float), ("image_token_id", C.c_int32), ("pad_token_id", C.c_int32),
        ("decoder_start_id", C.c_int32), ("emulate_bf16_rounding", C.c_int32), ("cross_attention_mode", C.c_int32),
    ]


class VqaQwen25VLConfig(C.Structure):
    _fields_ = [
        ("vit_depth", C.c_int32), ("vit_hidden", C.c_int32), ("vit_heads", C.c_int32), ("vit_head_dim", C.c_int32),
        ("vit_mlp", C.c_int32), ("patch_dim", C.c_int32), ("spatial_merge", C.c_int32), ("out_hidden", C.c_int32),
        ("fullatt_mask", C.c_uint64), ("hidden", C.c_int32), ("layers", C.c_int32), ("heads", C.c_int32),
        ("kv_heads", C.c_int32), ("mlp", C.c_int32), ("vocab", C.c_int32), ("rms_eps", C.c_float),
        ("emulate_bf16_rounding", C.c_int32),
    ]


class VqaTensor(C.Structure):
    _fields_ = [("name", C.c_char_p), ("data", C.c_void_p), ("shape", C.c_int64 * 4), ("ndim", C.c_int32),
                ("dtype", C.c_int32)]


_lib = None


def load() -> C.CDLL:
    """dlopen libvqa_b200.so and declare prototypes. Raises if the library is absent (no CPU fallback exists)."""
    global _lib
    if _lib is not None:
        return _lib
    path = Path(os.environ.get("VQA_B200_LIB", LIB_PATH))
    if not path.exists():
        raise ImportError(
            f"{path} not found: build it first (python -c 'import __graft_entry__ as g; g.build()'). "
            "t2v_metrics_b200 has no CPU or PyTorch fallback for the scoring path.")
    lib = C.CDLL(str(path))
    for sym in ABI_SYMBOLS:
        if not hasattr(lib, sym):
            raise ImportError(f"{path} does not export {sym}")
    vp, i32, f32, i64 = C.c_void_p, C.c_int32, C.c_float, C.c_int64
    lib.vqa_version.restype = C.c_char_p
    lib.vqa_create_clipt5.argtypes = [C.POINTER(VqaClipT5Config), C.c_int, C.POINTER(vp)]
    lib.vqa_create_clipt5.restype = C.c_int
    lib.vqa_bind_weights.argtypes = [vp, C.POINTER(VqaTensor), i32]
    lib.vqa_bind_weights.restype = C.c_int
    lib.vqa_finalize_weights.argtypes = [vp]
    lib.vqa_finalize_weights.restype = C.c_int
    lib.vqa_clipt5_workspace_bytes.argtypes = [vp, i32, i32, i32, i32]
    lib.vqa_clipt5_workspace_bytes.restype = C.c_size_t
    lib.vqa_clipt5_score.argtypes = [vp, vp, i32, i32, vp, vp, vp, vp, i32, i32, i32, vp, vp, vp, C.c_size_t, vp]
    lib.vqa_clipt5_score.restype = C.c_int
    lib.vqa_set_profile.argtypes = [vp, i32]
    lib.vqa_set_profile.restype = C.c_int
    lib.vqa_profile_read.argtypes = [vp, C.POINTER(C.c_float), C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_int64)]
    lib.vqa_profile_read.restype = C.c_int
    lib.vqa_last_launch_count.argtypes = [vp]
    lib.vqa_last_launch_count.restype = i64
    lib.vqa_last_error.argtypes = [vp]
    lib.vqa_last_error.restype = C.c_char_p
    lib.vqa_destroy.argtypes = [vp]
    lib.vqa_destroy.restype = None
    lib.vqa_op_gemm_bf16.argtypes = [vp, i32, vp, i32, i32, vp, i32, i32, i32, i32, vp, vp, i32, i32, i32, i32, vp]
    lib.vqa_op_gemm_bf16.restype = C.c_int
    lib.vqa_op_gemm_bf16_normfuse.argtypes = [vp, i32, vp, i32, i32, vp, i32, i32, i32, i32, vp, i32, i32, i32, vp, vp, i32, i32, f32,
                                              C.POINTER(i32), vp]
    lib.vqa_op_gemm_bf16_normfuse.restype = C.c_int
    lib.vqa_op_lmhead_logprob.argtypes = [vp, i32, vp, i32, i32, i32, i32, vp, vp, vp, vp]
    lib.vqa_op_lmhead_logprob.restype = C.c_int
    lib.vqa_op_attention_d64.argtypes = [vp, vp, i32, i32, i32, vp, vp, f32, i32, i32, vp]
    lib.vqa_op_attention_d64.restype = C.c_int
    lib.vqa_op_norm.argtypes = [vp, vp, vp, vp, i32, i32, f32, vp]
    lib.vqa_op_norm.restype = C.c_int
    lib.vqa_op_attention_d128.argtypes = [vp, i32, i64, i32, i32, i32, vp, i32, i32, i32, i32, i32, i32, vp, vp, f32, i32, vp]
    lib.vqa_op_attention_d128.restype = C.c_int
    lib.vqa_create_qwen25vl.argtypes = [C.POINTER(VqaQwen25VLConfig), C.c_int, C.POINTER(vp)]
    lib.vqa_create_qwen25vl.restype = C.c_int
    lib.vqa_qwen25vl_set_rope.argtypes = [vp, C.POINTER(C.c_float), C.POINTER(i32), i32, C.POINTER(C.c_float), C.POINTER(i32), i32]
    lib.vqa_qwen25vl_set_rope.restype = C.c_int
    lib.vqa_qwen25vl_workspace_bytes.argtypes = [vp, i32, i32, i32]
    lib.vqa_qwen25vl_workspace_bytes.restype = C.c_size_t
    lib.vqa_qwen25vl_score.argtypes = [vp, vp, i32, i32, vp, vp, vp, vp, i32, i32, vp, i32, i32, vp, vp, vp, vp, vp, i32, i32, f32,
                                       f32, vp, vp, vp, C.c_size_t, vp]
    lib.vqa_qwen25vl_score.restype = C.c_int
    lib.vqa_qwen25vl_topk.argtypes = [vp, i32, i64, i32, i32, f32, f32, vp, vp, vp, C.c_size_t, vp]
    lib.vqa_qwen25vl_packed_workspace_bytes.argtypes = [vp, i32, i64, i32]
    lib.vqa_qwen25vl_packed_workspace_bytes.restype = C.c_size_t
    lib.vqa_qwen25vl_score_packed.argtypes = [vp, vp, i32, i32, vp, vp, vp, vp, i32, i32, vp, i32, i32, vp, vp, vp, i32, vp, vp, i32, i32, vp, vp,
                                              vp, i32, i32, f32, f32, vp, vp, vp, C.c_size_t, vp]
    lib.vqa_qwen25vl_score_packed.restype = C.c_int
    lib.vqa_qwen25vl_topk.restype = C.c_int
    lib.vqa_clip_preprocess_workspace_bytes.argtypes = [C.POINTER(i32), C.POINTER(i32), i32, i32, i32]
    lib.vqa_clip_preprocess_workspace_bytes.restype = C.c_size_t
    lib.vqa_clip_preprocess.argtypes = [vp, C.POINTER(i64), C.POINTER(i32), C.POINTER(i32), i32, i32, i32, C.POINTER(C.c_uint8),
                                        C.POINTER(C.c_float), C.POINTER(C.c_float), vp, i32, vp, C.c_size_t, vp, vp]
    lib.vqa_clip_preprocess.restype = C.c_int
    lib.vqa_qwen_preprocess_plan.argtypes = [C.POINTER(i32), C.POINTER(i32), i32, i32, i32, i64, i64, C.POINTER(i32), C.POINTER(i64),
                                             C.POINTER(C.c_size_t)]
    lib.vqa_qwen_preprocess_plan.restype = C.c_int
    lib.vqa_qwen_preprocess.argtypes = [vp, C.POINTER(i64), C.POINTER(i32), C.POINTER(i32), i32, i32, i32, i32, i64, i64,
                                        C.POINTER(C.c_float), C.POINTER(C.c_float), vp, i32, vp, C.c_size_t, vp, vp]
    lib.vqa_qwen_preprocess.restype = C.c_int
    lib.vqa_clipt5_debug_layout.argtypes = [vp, i32, i32, i32, i32, C.POINTER(C.c_size_t), i32]
    lib.vqa_clipt5_debug_layout.restype = C.c_int
    lib.vqa_qwen25vl_debug_layout.argtypes = [vp, i32, i32, i32, C.POINTER(C.c_size_t), i32]
    lib.vqa_qwen25vl_debug_layout.restype = C.c_int
    lib.vqa_set_gemm_schedule.argtypes = [i32, i32]
    lib.vqa_set_gemm_schedule.restype = C.c_int
    lib.vqa_op_attention_d128_ex.argtypes = [vp, i32, i64, i32, i32, i32, vp, i32, i32, i32, i32, i32, vp, vp, f32, i32, i32, i32, i32, vp]
    lib.vqa_op_attention_d128_ex.restype = C.c_int
    lib.vqa_op_gemm_bf16_grouped.argtypes = [vp, i32, vp, i32, i32, vp, i32, i32, i32, i32, vp, i32, i32, i32, vp]
    lib.vqa_op_gemm_bf16_grouped.restype = C.c_int
    lib.vqa_op_gemm_bf16_splitk.argtypes = [vp, i32, vp, i32, i32, vp, i32, i32, i32, i32, vp, vp, i32, i32, vp, C.c_size_t, C.POINTER(i32), vp]
    lib.vqa_op_gemm_bf16_splitk.restype = C.c_int
    lib.vqa_debug_max_active_clusters.argtypes = [i32]
    lib.vqa_debug_max_active_clusters.restype = C.c_int
    lib.vqa_resample_table.argtypes = [i32, i32, i32, i32, C.POINTER(i32), C.POINTER(i32)]
    lib.vqa_resample_table.restype = i32
    lib.vqa_qwen_video_preprocess_plan.argtypes = [C.POINTER(i32), C.POINTER(i32), C.POINTER(i32), C.POINTER(i32), i32, i32, i32, i32,
                                                   C.POINTER(i64), C.POINTER(i64), C.POINTER(i32), C.POINTER(i64), C.POINTER(C.c_size_t)]
    lib.vqa_qwen_video_preprocess_plan.restype = C.c_int
    lib.vqa_qwen_video_preprocess.argtypes = [vp, C.POINTER(i64), C.POINTER(i32), C.POINTER(i32), C.POINTER(i32), C.POINTER(i32), i32, i32,
                                              i32, i32, C.POINTER(i64), C.POINTER(i64), C.POINTER(C.c_float), C.POINTER(C.c_float), vp, i32,
                                              vp, C.c_size_t, vp, vp]
    lib.vqa_qwen_video_preprocess.restype = C.c_int
    lib.vqa_resample_table_tv.argtypes = [i32, i32, i32, i32, C.POINTER(i32), C.POINTER(C.c_float), C.POINTER(i32)]
    lib.vqa_resample_table_tv.restype = i32
    _lib = lib
    return lib


def last_error(handle=None) -> str:
    msg = load().vqa_last_error(handle)
    return msg.decode() if msg else ""
