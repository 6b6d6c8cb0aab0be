"""ctypes binding of the C ABI in include/lrn_b200.h (in-tree liblrn_b200.so).

There is no fallback: importing this module raises if the library has not been built
(``python pointnet_refine_b200/build.py``), and every compute call raises
``RuntimeError`` on a non-zero status (e.g. LRN_ERR_UNSUPPORTED_ARCH off sm_100).
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# LRN_B200_LIB selects another build of the same ABI (tools/timeline.py: the -DLRN_TIMELINE tuning variant)
LIB_PATH = os.environ.get("LRN_B200_LIB") or os.path.join(_HERE, "liblrn_b200.so")
CSRC = os.path.join(_HERE, "csrc")
HEADER = os.path.join(os.path.dirname(_HERE), "include", "lrn_b200.h")

# enums of include/lrn_b200.h
ABI_VERSION = 3      # LRN_ABI_VERSION
LRN_OK = 0
PREC_BF16, PREC_TF32, PREC_FP32X3 = 0, 1, 2
OUT_POOL, OUT_ARGMAX, OUT_FUSED, OUT_MEMORY, OUT_MEMORY_BF16 = 1, 2, 4, 8, 16
PRECISIONS = {"bf16": PREC_BF16, "tf32": PREC_TF32, "fp32x3": PREC_FP32X3}
STAGES = ["embed", "conv2", "conv3", "conv4", "conv5", "fusion", "proj"]


class EncoderParams(C.Structure):
    """struct lrn_encoder_params"""
    _fields_ = (
        [(n, C.c_void_p * 5) for n in ("conv_w", "conv_b", "bn_w", "bn_b", "bn_mean", "bn_var")]
        + [(n, C.c_void_p) for n in ("fusion_w", "fusion_b", "fusion_bn_w", "fusion_bn_b", "fusion_bn_mean",
                                     "fusion_bn_var", "gate0_w", "gate0_b", "gate2_w", "gate2_b", "proj_w", "proj_b")]
        + [("bn_eps", C.c_float)]
    )


class BnRunning(C.Structure):
    """struct lrn_bn_running"""
    _fields_ = [("mean", C.c_void_p * 6), ("var", C.c_void_p * 6)]


class EncoderGrads(C.Structure):
    """struct lrn_encoder_grads"""
    _fields_ = ([(n, C.c_void_p * 5) for n in ("conv_w", "conv_b", "bn_w", "bn_b")]
                + [(n, C.c_void_p) for n in ("fusion_w", "fusion_b", "fusion_bn_w", "fusion_bn_b",
                                             "gate0_w", "gate0_b", "gate2_w", "gate2_b")])


vp, i64, sz, ci, f32, f64, u64 = C.c_void_p, C.c_int64, C.c_size_t, C.c_int, C.c_float, C.c_double, C.c_uint64
# name -> (restype, argtypes) of every entry point declared in include/lrn_b200.h
SIGNATURES = {
    "lrn_abi_version": (ci, []),
    "lrn_status_string": (C.c_char_p, [ci]),
    "lrn_last_error": (C.c_char_p, []),
    "lrn_launch_count": (sz, []),
    "lrn_device_check": (ci, []),
    "lrn_encoder_packed_bytes": (sz, [ci]),
    "lrn_encoder_fold": (ci, [C.POINTER(EncoderParams), ci, vp, sz, vp]),
    "lrn_encoder_workspace_bytes": (sz, [i64, i64, ci, ci, i64]),
    "lrn_encoder_forward": (ci, [vp, ci, vp, i64, i64, ci, vp, vp, vp, vp, i64, vp, sz, vp]),
    "lrn_head_forward": (ci, [vp, vp, vp, vp, vp, i64, vp, vp, vp, vp]),
    "lrn_gemm_bias_act": (ci, [ci, vp, i64, vp, i64, vp, vp, i64, ci, ci, i64, i64, i64, vp]),
    "lrn_profile_enable": (ci, [ci]),
    "lrn_profile_read": (ci, [C.POINTER(f32), C.POINTER(i64)]),
    "lrn_debug_timeline": (ci, [vp]),
    "lrn_train_workspace_bytes": (sz, [i64, i64]),
    "lrn_encoder_train_forward": (ci, [C.POINTER(EncoderParams), C.POINTER(BnRunning), f32, vp, i64, i64, vp, ci, vp, vp,
                                       vp, sz, vp]),
    "lrn_encoder_train_backward": (ci, [C.POINTER(EncoderParams), vp, i64, i64, vp, ci, vp, vp, C.POINTER(EncoderGrads), vp,
                                        sz, vp]),
    "lrn_gemm_tn": (ci, [vp, i64, vp, i64, vp, i64, i64, i64, i64, vp]),
    "lrn_point_embed": (ci, [vp, ci, vp, i64, vp, ci, vp]),
    "lrn_ctx_attention_splits": (ci, [ci, ci]),
    "lrn_ctx_attention": (ci, [vp, vp, i64, vp, i64, ci, ci, ci, vp, ci, vp, vp]),
    "lrn_pos_hidden": (ci, [vp, vp, vp, i64, vp, i64, vp]),
    "lrn_pos_hidden_backward": (ci, [vp, i64, vp, i64, vp, i64, vp, vp, vp]),
    "lrn_scene_workspace_bytes": (sz, [ci, i64]),
    "lrn_scene_segments": (ci, [vp, i64, vp, vp, vp, vp, vp, ci, ci, f64, f64, f64, u64, i64, vp, vp, vp, vp, vp, sz, vp]),
    "lrn_scene_resample": (ci, [vp, vp, ci, ci, vp, vp, vp, vp, vp]),
    "lrn_adam_step": (ci, [vp, vp, vp, vp, i64, f32, f32, f32, f32, f32, i64, vp]),
    "lrn_adam_step_capturable": (ci, [vp, vp, vp, vp, i64, f32, f32, f32, f32, f32, vp, vp]),
    "lrn_l1_deep_supervision": (ci, [vp, vp, ci, i64, vp, vp, vp]),
    "lrn_col_sum_bf16": (ci, [vp, i64, i64, i64, vp, vp]),
    "lrn_gather_heads": (ci, [vp, ci, ci, ci, ci, ci, vp, vp]),
    "lrn_add_layernorm": (ci, [vp, vp, vp, vp, f32, vp, vp, i64, i64, vp]),
    "lrn_add_layernorm_backward": (ci, [vp, vp, vp, vp, vp, vp, vp, vp, i64, i64, vp]),
    "lrn_self_attention32": (ci, [vp, vp, vp, ci, vp]),
    "lrn_head_update": (ci, [vp, vp, vp, i64, vp, vp, vp, vp]),
    "lrn_rows_linear": (ci, [vp, i64, vp, i64, vp, vp, vp, vp, vp, i64, ci, ci, i64, i64, i64, vp]),
    "lrn_query_pos_hidden": (ci, [vp, vp, vp, i64, i64, vp, ci, vp]),
    "lrn_add": (ci, [vp, vp, vp, i64, ci, vp]),
    "lrn_ctx_attention_merge": (ci, [vp, vp, ci, ci, vp, ci, vp]),
    "lrn_cross_attention32": (ci, [vp, vp, vp, i64, ci, ci, vp, vp]),
    "lrn_train_attention_forward": (ci, [vp, vp, i64, vp, i64, ci, ci, vp, vp, f32, u64, vp, vp]),
    "lrn_train_attention_backward": (ci, [vp, vp, i64, vp, i64, ci, ci, vp, vp, vp, vp, vp, i64, vp, i64, f32, u64, vp, vp]),
}
EXPORTS = list(SIGNATURES)


def _load():
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: the CUDA library must be built first "
            "(python pointnet_refine_b200/build.py).  There is no CPU or PyTorch fallback.")
    lib = C.CDLL(LIB_PATH)
    if lib.lrn_abi_version() != ABI_VERSION:
        raise RuntimeError(f"liblrn_b200.so has ABI version {lib.lrn_abi_version()}, this package binds version {ABI_VERSION}; rebuild it "
                           "(python pointnet_refine_b200/build.py --force)")
    for name, (restype, argtypes) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype, fn.argtypes = restype, argtypes
    return lib


lib = _load()


def __getattr__(name):
    # launch_counter: kernels this library has enqueued in this process (bench.py reports the delta), counted by the library
    if name == "launch_counter":
        return lib.lrn_launch_count()
    raise AttributeError(f"module {__name__!r} has no attribute {name!r}")


def check(status: int, what: str) -> None:
    if status != LRN_OK:
        raise RuntimeError(f"{what} failed: {lib.lrn_status_string(status).decode()} "
                           f"[{status}] {lib.lrn_last_error().decode()}")
