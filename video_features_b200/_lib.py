"""ctypes binding of libvfeat.so (the C ABI declared in include/vfeat.h).

There is no fallback: if the shared library is missing or a call fails, an exception is raised.
"""
from __future__ import annotations

import ctypes as C
import os
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
# VF_LIBVFEAT selects another build of the same library (A/B variants of one kernel, scripts/build_variants.sh)
LIB_PATH = os.environ.get("VF_LIBVFEAT") or os.path.join(_HERE, "libvfeat.so")

VF_OK = 0
VF_ACT_NONE, VF_ACT_QUICKGELU, VF_ACT_RELU, VF_ACT_SIGMOID, VF_ACT_TANH = 0, 1, 2, 3, 4
VF_FILTER_BILINEAR, VF_FILTER_BICUBIC = 2, 3


class VfError(RuntimeError):
    def __init__(self, code: int, text: str):
        super().__init__(f"libvfeat error {code}: {text}")
        self.code = code


class ClipLayerWeights(C.Structure):
    _fields_ = [(n, C.POINTER(C.c_float)) for n in (
        "ln_1_w", "ln_1_b", "in_proj_w", "in_proj_b", "out_proj_w", "out_proj_b",
        "ln_2_w", "ln_2_b", "c_fc_w", "c_fc_b", "c_proj_w", "c_proj_b")]


class ClipWeights(C.Structure):
    _fields_ = [(n, C.POINTER(C.c_float)) for n in (
        "conv1_w", "class_embedding", "positional_embedding",
        "ln_pre_w", "ln_pre_b", "ln_post_w", "ln_post_b", "proj")] + [("layers", ClipLayerWeights * 12)]


class ConvUnitW(C.Structure):
    _fields_ = [("w", C.POINTER(C.c_float)), ("bn_w", C.POINTER(C.c_float)), ("bn_b", C.POINTER(C.c_float)),
                ("bn_mean", C.POINTER(C.c_float)), ("bn_var", C.POINTER(C.c_float)),
                ("cout", C.c_int), ("cin", C.c_int), ("k", C.c_int)]


I3D_UNITS = 57


class I3DWeights(C.Structure):
    _fields_ = [("units", ConvUnitW * I3D_UNITS)]


class NamedTensor(C.Structure):
    _fields_ = [("name", C.c_char_p), ("data", C.POINTER(C.c_float)), ("numel", C.c_int64)]


_lock = threading.Lock()
_lib = None

# name -> (restype, argtypes); every symbol declared in include/vfeat.h
SIGNATURES = {
    "vf_version": (C.c_int, []),
    "vf_last_error": (C.c_char_p, []),
    "vf_sample_indices": (C.c_int, [C.c_char_p, C.c_int, C.c_int64, C.c_double, C.POINTER(C.c_int64), C.c_int64,
                                    C.POINTER(C.c_int64)]),
    "vf_shard_range": (C.c_int, [C.c_int64, C.c_int, C.c_int, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "vf_resize_u8": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int,
                               C.c_void_p, C.c_void_p]),
    "vf_resize_geometry": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "vf_clip_normalize_u8": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "vf_gemm_f16": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p,
                              C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "vf_gemm_f16_accumulate": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                         C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "vf_gemm_f16_split": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                    C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "vf_gemm_profile": (C.c_int, [C.c_int]),
    "vf_gemm_profile_read": (C.c_int, [C.POINTER(C.c_double), C.POINTER(C.c_int64), C.POINTER(C.c_double)]),
    "vf_clip_create": (C.c_int, [C.POINTER(C.c_void_p), C.POINTER(ClipWeights), C.c_int, C.c_int]),
    "vf_clip_create_vit": (C.c_int, [C.POINTER(C.c_void_p), C.POINTER(ClipWeights), C.c_int, C.c_int, C.c_int]),
    "vf_clip_destroy": (C.c_int, [C.c_void_p]),
    "vf_clip_encode_f32": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    "vf_clip_encode_u8": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "vf_clip_encode_u8_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "vf_clip_encode_u8_host_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                             C.c_void_p]),
    "vf_clip_encode_u8_host_async": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                               C.c_void_p, C.POINTER(C.c_int64)]),
    "vf_clip_wait": (C.c_int, [C.c_void_p, C.c_int64]),
    "vf_clip_block_attention": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p]),
    "vf_clip_launch_count": (C.c_int64, [C.c_void_p]),
    "vf_i3d_create": (C.c_int, [C.POINTER(C.c_void_p), C.POINTER(I3DWeights), C.c_int, C.c_int, C.c_int, C.c_int]),
    "vf_i3d_destroy": (C.c_int, [C.c_void_p]),
    "vf_i3d_forward_f32": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "vf_i3d_forward_u8": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "vf_i3d_forward_u8_strided": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int64, C.c_int, C.c_int, C.c_void_p,
                                            C.c_void_p]),
    "vf_i3d_forward_flow": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "vf_i3d_read_stage": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int64, C.POINTER(C.c_int), C.c_void_p]),
    "vf_i3d_launch_count": (C.c_int64, [C.c_void_p]),
    "vf_raft_create": (C.c_int, [C.POINTER(C.c_void_p), C.POINTER(NamedTensor), C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]),
    "vf_raft_destroy": (C.c_int, [C.c_void_p]),
    "vf_raft_flow": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                               C.c_void_p, C.c_void_p]),
    "vf_raft_padded_size": (C.c_int, [C.c_int, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "vf_raft_debug_read": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int64, C.POINTER(C.c_int), C.c_void_p]),
    "vf_raft_launch_count": (C.c_int64, [C.c_void_p]),
    "vf_resnet_create": (C.c_int, [C.POINTER(C.c_void_p), C.c_int, C.POINTER(NamedTensor), C.c_int, C.c_int, C.c_int]),
    "vf_resnet_destroy": (C.c_int, [C.c_void_p]),
    "vf_resnet_feature_dim": (C.c_int, [C.c_void_p]),
    "vf_resnet_forward_f32": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    "vf_resnet_forward_u8": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "vf_imagenet_normalize_u8": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "vf_resnet_read_stage": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int64, C.POINTER(C.c_int), C.c_void_p]),
    "vf_resnet_launch_count": (C.c_int64, [C.c_void_p]),
    "vf_clip_profile": (C.c_int, [C.c_void_p, C.c_int]),
    "vf_clip_profile_categories": (C.c_int, [C.c_void_p, C.POINTER(C.c_double)]),
    "vf_clip_profile_read": (C.c_int, [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_int64),
                                       C.POINTER(C.c_double)]),
}


def lib() -> C.CDLL:
    """Load libvfeat.so once; raises if it has not been built (``python -c 'import __graft_entry__ as g; g.build()'``)."""
    global _lib
    if _lib is None:
        with _lock:
            if _lib is None:
                if not os.path.exists(LIB_PATH):
                    raise FileNotFoundError(
                        f"{LIB_PATH} not found: build the CUDA extension first (__graft_entry__.build()). "
                        "There is no CPU fallback.")
                l = C.CDLL(LIB_PATH)
                for name, (res, args) in SIGNATURES.items():
                    fn = getattr(l, name)      # AttributeError if a declared symbol is not exported
                    fn.restype = res
                    fn.argtypes = args
                _lib = l
    return _lib


def check(status: int) -> None:
    if status != VF_OK:
        raise VfError(status, lib().vf_last_error().decode("utf-8", "replace"))
