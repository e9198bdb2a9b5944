"""torch-facing wrappers: PyTorch custom ops (``torch.library``) over the C ABI.

PyTorch is plumbing here -- device memory, streams -- every op hands raw ``data_ptr()``s and the current CUDA
stream to libvfeat.so.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional

import numpy as np
import torch

from . import _lib
from ._lib import check, lib


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _need_cuda(*ts: torch.Tensor) -> None:
    for t in ts:
        if t is not None and not t.is_cuda:
            raise RuntimeError("libvfeat ops run on CUDA tensors only (there is no CPU fallback)")
        if t is not None and not t.is_contiguous():
            raise RuntimeError("libvfeat ops need contiguous tensors")


# ----------------------------------------------------------------------------- GEMM
@torch.library.custom_op("vfeat::gemm_f16", mutates_args=())
def gemm_f16(a: torch.Tensor, b: torch.Tensor, bias: Optional[torch.Tensor], scale: Optional[torch.Tensor],
             act: int, out_f32: bool) -> torch.Tensor:
    """act(a @ b.T * scale + bias); a (M,K) fp16, b (N,K) fp16; fp32 accumulate on tcgen05."""
    _need_cuda(a, b, bias, scale)
    assert a.dtype == torch.float16 and b.dtype == torch.float16 and a.shape[1] == b.shape[1]
    M, K = a.shape
    N = b.shape[0]
    out = torch.empty((M, N), device=a.device, dtype=torch.float32 if out_f32 else torch.float16)
    with torch.cuda.device(a.device):
        check(lib().vf_gemm_f16(a.data_ptr(), K, b.data_ptr(), K, M, N, K, out.data_ptr(), N, int(out_f32),
                                _ptr(bias), _ptr(scale), act, _stream()))
    return out


@gemm_f16.register_fake
def _(a, b, bias, scale, act, out_f32):
    return a.new_empty((a.shape[0], b.shape[0]), dtype=torch.float32 if out_f32 else torch.float16)


@torch.library.custom_op("vfeat::gemm_f16_accumulate", mutates_args=("out",))
def gemm_f16_accumulate(out: torch.Tensor, a: torch.Tensor, b: torch.Tensor, bias: Optional[torch.Tensor], act: int) -> None:
    """out (M,N) fp32 += act(a @ b.T + bias): the residual-stream update, added in the L2 by a TMA reduction."""
    _need_cuda(out, a, b, bias)
    assert out.dtype == torch.float32 and a.dtype == torch.float16 and b.dtype == torch.float16
    M, K = a.shape
    N = b.shape[0]
    assert tuple(out.shape) == (M, N) and b.shape[1] == K
    with torch.cuda.device(a.device):
        check(lib().vf_gemm_f16_accumulate(a.data_ptr(), K, b.data_ptr(), K, M, N, K, out.data_ptr(), N, _ptr(bias), None,
                                           act, _stream()))


# ----------------------------------------------------------------------------- encoders (handles are opaque int64 values)
@torch.library.custom_op("vfeat::clip_encode_u8", mutates_args=())
def clip_encode_u8(handle: int, frames: torch.Tensor) -> torch.Tensor:
    """Fused CLIP transform + ViT-B/32 tower (vf_clip_encode_u8): (N,H,W,3) uint8 on the device -> (N,512) fp32.
    `handle` is the vf_clip_t* of a ClipEngine (ClipEngine.handle)."""
    _need_cuda(frames)
    assert frames.dtype == torch.uint8 and frames.dim() == 4 and frames.shape[3] == 3
    n, hh, ww, _ = frames.shape
    out = torch.empty((n, 512), device=frames.device, dtype=torch.float32)
    with torch.cuda.device(frames.device):
        check(lib().vf_clip_encode_u8(C.c_void_p(handle), frames.data_ptr(), n, hh, ww, out.data_ptr(), _stream()))
    return out


@clip_encode_u8.register_fake
def _(handle, frames):
    return frames.new_empty((frames.shape[0], 512), dtype=torch.float32)


@torch.library.custom_op("vfeat::clip_encode_image", mutates_args=())
def clip_encode_image(handle: int, frames: torch.Tensor) -> torch.Tensor:
    """`model.encode_image(frames)` (vf_clip_encode_f32): (N,3,224,224) fp32 on the device -> (N,512) fp32."""
    _need_cuda(frames)
    assert frames.dtype == torch.float32 and frames.dim() == 4 and tuple(frames.shape[1:]) == (3, 224, 224)
    out = torch.empty((frames.shape[0], 512), device=frames.device, dtype=torch.float32)
    with torch.cuda.device(frames.device):
        check(lib().vf_clip_encode_f32(C.c_void_p(handle), frames.data_ptr(), frames.shape[0], out.data_ptr(), _stream()))
    return out


@clip_encode_image.register_fake
def _(handle, frames):
    return frames.new_empty((frames.shape[0], 512), dtype=torch.float32)


@torch.library.custom_op("vfeat::i3d_forward", mutates_args=())
def i3d_forward(handle: int, x: torch.Tensor) -> torch.Tensor:
    """`I3D(x, features=True)` (vf_i3d_forward_f32): (B,C,T,224,224) fp32 in [-1,1] on the device -> (B,1024) fp32."""
    _need_cuda(x)
    assert x.dtype == torch.float32 and x.dim() == 5 and tuple(x.shape[3:]) == (224, 224)
    out = torch.empty((x.shape[0], 1024), device=x.device, dtype=torch.float32)
    with torch.cuda.device(x.device):
        check(lib().vf_i3d_forward_f32(C.c_void_p(handle), x.data_ptr(), x.shape[0], x.shape[2], out.data_ptr(), _stream()))
    return out


@i3d_forward.register_fake
def _(handle, x):
    return x.new_empty((x.shape[0], 1024), dtype=torch.float32)


@torch.library.custom_op("vfeat::resnet_forward", mutates_args=())
def resnet_forward(handle: int, dim: int, x: torch.Tensor) -> torch.Tensor:
    """`model(x)` of torchvision resnet{depth} with fc = Identity (vf_resnet_forward_f32): (n,3,224,224) fp32 normalised
    on the device -> (n, dim) fp32."""
    _need_cuda(x)
    assert x.dtype == torch.float32 and x.dim() == 4 and tuple(x.shape[1:]) == (3, 224, 224)
    out = torch.empty((x.shape[0], dim), device=x.device, dtype=torch.float32)
    with torch.cuda.device(x.device):
        check(lib().vf_resnet_forward_f32(C.c_void_p(handle), x.data_ptr(), x.shape[0], out.data_ptr(), _stream()))
    return out


@resnet_forward.register_fake
def _(handle, dim, x):
    return x.new_empty((x.shape[0], dim), dtype=torch.float32)


# ----------------------------------------------------------------------------- transforms
@torch.library.custom_op("vfeat::resize_u8", mutates_args=())
def resize_u8(frames: torch.Tensor, out_h: int, out_w: int, filter: int) -> torch.Tensor:
    """Pillow-exact Image.resize of (N,H,W,3) uint8 frames."""
    _need_cuda(frames)
    assert frames.dtype == torch.uint8 and frames.dim() == 4 and frames.shape[3] == 3
    n, h, w, _ = frames.shape
    out = torch.empty((n, out_h, out_w, 3), device=frames.device, dtype=torch.uint8)
    tmp = torch.empty((n, h, out_w, 3), device=frames.device, dtype=torch.uint8)
    with torch.cuda.device(frames.device):
        check(lib().vf_resize_u8(frames.data_ptr(), n, h, w, out.data_ptr(), out_h, out_w, filter, tmp.data_ptr(),
                                 _stream()))
    return out


@resize_u8.register_fake
def _(frames, out_h, out_w, filter):
    return frames.new_empty((frames.shape[0], out_h, out_w, 3))


@torch.library.custom_op("vfeat::clip_normalize_u8", mutates_args=())
def clip_normalize_u8(frames: torch.Tensor) -> torch.Tensor:
    """CenterCrop(224) + ToTensor + Normalize of (N,H,W,3) uint8 -> (N,3,224,224) fp32 (bit-exact)."""
    _need_cuda(frames)
    assert frames.dtype == torch.uint8 and frames.dim() == 4 and frames.shape[3] == 3
    n, h, w, _ = frames.shape
    out = torch.empty((n, 3, 224, 224), device=frames.device, dtype=torch.float32)
    with torch.cuda.device(frames.device):
        check(lib().vf_clip_normalize_u8(frames.data_ptr(), n, h, w, out.data_ptr(), _stream()))
    return out


@clip_normalize_u8.register_fake
def _(frames):
    return frames.new_empty((frames.shape[0], 3, 224, 224), dtype=torch.float32)


def resize_geometry(h: int, w: int, size: int, to_smaller_edge: bool = True):
    oh, ow = C.c_int(), C.c_int()
    check(lib().vf_resize_geometry(h, w, size, int(to_smaller_edge), C.byref(oh), C.byref(ow)))
    return oh.value, ow.value


# ----------------------------------------------------------------------------- host-side integer helpers
def sample_indices(method: str, param: int, frame_cnt: int, fps: float) -> np.ndarray:
    n = C.c_int64()
    check(lib().vf_sample_indices(method.encode(), int(param), int(frame_cnt), float(fps), None, 0, C.byref(n)))
    buf = (C.c_int64 * max(n.value, 1))()
    check(lib().vf_sample_indices(method.encode(), int(param), int(frame_cnt), float(fps), buf, n.value, C.byref(n)))
    return np.frombuffer(buf, dtype=np.int64, count=n.value).copy()


def shard_range(n_items: int, n_parts: int, part: int):
    b, e = C.c_int64(), C.c_int64()
    check(lib().vf_shard_range(n_items, n_parts, part, C.byref(b), C.byref(e)))
    return b.value, e.value


def gemm_profile(enable: bool) -> None:
    check(lib().vf_gemm_profile(int(enable)))


def gemm_profile_read():
    """-> (device ms, launches, executed FLOPs) of the GEMM launches since the last read (this thread)."""
    ms, n, fl = C.c_double(), C.c_int64(), C.c_double()
    check(lib().vf_gemm_profile_read(C.byref(ms), C.byref(n), C.byref(fl)))
    return ms.value, n.value, fl.value
