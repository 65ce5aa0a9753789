"""ctypes binding of libmmee.so (C ABI declared in include/mmee.h).

The library is built in-tree by `__graft_entry__.build()` (nvcc, sm_100a).  There is no CPU or
eager-PyTorch fallback: if the shared object is missing or no B200 is present, calls fail loudly.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("MMEE_LIB", os.path.join(_HERE, "libmmee.so"))   # MMEE_LIB: developer override for A/B runs
MMEE_MAX_EXITS = 64
COMPUTE_DTYPES = {"bf16": 0, "fp32": 1}      # include/mmee.h MMEE_DTYPE_*

EXPORTED_SYMBOLS = [
    "mmee_create", "mmee_destroy", "mmee_set_weight", "mmee_set_bucket_lut", "mmee_get_bucket_lut",
    "mmee_finalize_weights", "mmee_forward", "mmee_forward_device", "mmee_last_launch_count",
    "mmee_set_profiling", "mmee_collect_profile", "mmee_last_stage_ms", "mmee_debug_read", "mmee_last_error",
    "mmee_version", "mmee_policy_scan", "mmee_forward_submit", "mmee_forward_collect",
    "mmee_temperature_fit", "mmee_calibration_stats", "mmee_sync",
    "mmee_policy_store_create", "mmee_policy_store_destroy", "mmee_policy_store_criteria", "mmee_policy_store_scan",
    "mmee_plan_create", "mmee_plan_forward", "mmee_plan_forward_device", "mmee_plan_destroy",
    "mmee_preprocess_images", "mmee_forward_images",
]


class ModelDesc(C.Structure):
    _fields_ = [
        ("hidden", C.c_int), ("layers", C.c_int), ("heads", C.c_int), ("inter", C.c_int),
        ("n_text", C.c_int), ("image", C.c_int), ("patch", C.c_int), ("channels", C.c_int),
        ("n_labels", C.c_int), ("coord", C.c_int), ("shape", C.c_int),
        ("vocab", C.c_int), ("max_pos", C.c_int), ("max_2d", C.c_int),
        ("rel_bins", C.c_int), ("max_rel", C.c_int), ("rel2d_bins", C.c_int), ("max_rel2d", C.c_int),
        ("pad_id", C.c_int), ("ln_eps", C.c_float), ("vis_ln_eps", C.c_float),
        ("n_exits", C.c_int), ("exit_after_layer", C.c_int * MMEE_MAX_EXITS),
        ("head_kind", C.c_int), ("head_layers", C.c_int), ("compute_dtype", C.c_int),
    ]


class Policy(C.Structure):
    _fields_ = [
        ("criterion", C.c_int), ("mode", C.c_int),
        ("thresholds", C.POINTER(C.c_float)), ("temperatures", C.POINTER(C.c_float)),
    ]


class Outputs(C.Structure):
    _fields_ = [
        ("logits", C.c_void_p), ("exit_index", C.c_void_p), ("criterion", C.c_void_p),
        ("all_exit_logits", C.c_void_p), ("all_head_logits", C.c_void_p), ("all_criteria", C.c_void_p),
        ("exit_hist", C.c_void_p),
    ]


class Images(C.Structure):
    _fields_ = [
        ("data", C.c_void_p), ("offsets", C.c_void_p), ("sizes", C.c_void_p), ("channels", C.c_int),
        ("total_bytes", C.c_int64),
    ]


_lib = None


def load() -> C.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} not found: build the CUDA engine first (python -c 'import __graft_entry__ as g; g.build()'). "
            "mmee has no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    lib.mmee_create.argtypes = [C.POINTER(ModelDesc), C.c_int, C.c_int, C.POINTER(C.c_void_p)]
    lib.mmee_create.restype = C.c_int
    lib.mmee_destroy.argtypes = [C.c_void_p]
    lib.mmee_destroy.restype = None
    lib.mmee_set_weight.argtypes = [C.c_void_p, C.c_char_p, C.c_void_p, C.POINTER(C.c_int64), C.c_int]
    lib.mmee_set_weight.restype = C.c_int
    lib.mmee_set_bucket_lut.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int]
    lib.mmee_set_bucket_lut.restype = C.c_int
    lib.mmee_get_bucket_lut.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int]
    lib.mmee_get_bucket_lut.restype = C.c_int
    lib.mmee_finalize_weights.argtypes = [C.c_void_p]
    lib.mmee_finalize_weights.restype = C.c_int
    fwd_args = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                C.POINTER(Policy), C.POINTER(Outputs)]
    lib.mmee_forward.argtypes = fwd_args
    lib.mmee_forward.restype = C.c_int
    lib.mmee_forward_device.argtypes = fwd_args + [C.c_void_p]
    lib.mmee_forward_device.restype = C.c_int
    lib.mmee_forward_images.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(Images),
                                         C.POINTER(Policy), C.POINTER(Outputs)]
    lib.mmee_forward_images.restype = C.c_int
    lib.mmee_preprocess_images.argtypes = [C.c_void_p, C.c_int, C.POINTER(Images), C.c_void_p, C.c_void_p]
    lib.mmee_preprocess_images.restype = C.c_int
    lib.mmee_forward_submit.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(Policy)]
    lib.mmee_forward_submit.restype = C.c_int
    lib.mmee_forward_collect.argtypes = [C.c_void_p, C.c_int, C.POINTER(Outputs)]
    lib.mmee_forward_collect.restype = C.c_int
    lib.mmee_plan_create.argtypes = [C.c_void_p, C.c_int, C.POINTER(Policy), C.c_int, C.POINTER(C.c_void_p)]
    lib.mmee_plan_create.restype = C.c_int
    plan_args = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(Policy), C.POINTER(Outputs)]
    lib.mmee_plan_forward.argtypes = plan_args
    lib.mmee_plan_forward.restype = C.c_int
    lib.mmee_plan_forward_device.argtypes = plan_args + [C.c_void_p]
    lib.mmee_plan_forward_device.restype = C.c_int
    lib.mmee_plan_destroy.argtypes = [C.c_void_p]
    lib.mmee_plan_destroy.restype = None
    lib.mmee_last_launch_count.argtypes = [C.c_void_p]
    lib.mmee_last_launch_count.restype = C.c_int64
    lib.mmee_set_profiling.argtypes = [C.c_void_p, C.c_int]
    lib.mmee_set_profiling.restype = C.c_int
    lib.mmee_collect_profile.argtypes = [C.c_void_p]
    lib.mmee_collect_profile.restype = C.c_int
    lib.mmee_debug_read.argtypes = [C.c_void_p, C.c_char_p, C.c_void_p, C.c_int64]
    lib.mmee_debug_read.restype = C.c_int64
    lib.mmee_last_stage_ms.argtypes = [C.c_void_p, C.c_char_p]
    lib.mmee_last_stage_ms.restype = C.c_double
    lib.mmee_policy_scan.argtypes = [C.c_int, C.c_int, C.c_int64, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p,
                                     C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.mmee_policy_scan.restype = C.c_int
    lib.mmee_policy_store_create.argtypes = [C.c_int, C.c_int, C.c_int64, C.c_int, C.c_void_p, C.c_void_p, C.c_int,
                                             C.c_void_p, C.POINTER(C.c_void_p)]
    lib.mmee_policy_store_create.restype = C.c_int
    lib.mmee_policy_store_destroy.argtypes = [C.c_void_p]
    lib.mmee_policy_store_destroy.restype = None
    lib.mmee_policy_store_criteria.argtypes = [C.c_void_p, C.c_void_p]
    lib.mmee_policy_store_criteria.restype = C.c_int
    lib.mmee_policy_store_scan.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.mmee_policy_store_scan.restype = C.c_int
    lib.mmee_temperature_fit.argtypes = [C.c_int, C.c_int, C.c_int64, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                         C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.mmee_temperature_fit.restype = C.c_int
    lib.mmee_calibration_stats.argtypes = [C.c_int, C.c_int, C.c_int64, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                           C.c_void_p, C.c_void_p, C.c_void_p]
    lib.mmee_calibration_stats.restype = C.c_int
    lib.mmee_sync.argtypes = [C.c_void_p, C.c_void_p]
    lib.mmee_sync.restype = C.c_int
    lib.mmee_last_error.argtypes = []
    lib.mmee_last_error.restype = C.c_char_p
    lib.mmee_version.argtypes = []
    lib.mmee_version.restype = C.c_char_p
    _lib = lib
    return lib


def check(rc: int) -> None:
    if rc != 0:
        raise RuntimeError("libmmee: " + load().mmee_last_error().decode("utf-8", "replace"))
