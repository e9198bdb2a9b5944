"""ResNet feature extractor handle: stands where the reference keeps ``torchvision.models.resnet{depth}(pretrained=True)``
in eval mode with ``fc = Identity`` (models/resnet/extract_resnet.py:54-71); ``engine(x)`` mirrors ``model(x)``.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict

import numpy as np
import torch

from . import ops  # noqa: F401  (registers torch.ops.vfeat.*)
from ._lib import NamedTensor, check, lib


class ResNetEngine:
    """``state_dict``: torchvision's resnet{depth} key layout (``num_batches_tracked`` and ``fc.*`` are not read).
    ``max_frames``: frames per chunk of the device workspace; a call with more frames runs in equal chunks."""

    def __init__(self, state_dict: Dict[str, torch.Tensor], depth: int, device: int = 0, max_frames: int = 256):
        if not torch.cuda.is_available():
            raise RuntimeError("ResNetEngine needs a CUDA device (sm_100a); there is no CPU fallback")
        self.depth = depth
        self.device = torch.device("cuda", device)
        keep, table = [], []
        for k, v in state_dict.items():
            if k.startswith("fc.") or k.endswith("num_batches_tracked"):
                continue
            a = np.ascontiguousarray(v.detach().to("cpu", torch.float32).numpy())
            name = k.encode()
            keep += [a, name]
            table.append(NamedTensor(name, a.ctypes.data_as(C.POINTER(C.c_float)), a.size))
        arr = (NamedTensor * len(table))(*table)
        h = C.c_void_p()
        check(lib().vf_resnet_create(C.byref(h), depth, arr, len(table), device, max_frames))
        self._h = h
        self.dim = int(lib().vf_resnet_feature_dim(h))
        del keep

    def __call__(self, x: torch.Tensor) -> torch.Tensor:
        """x (n, 3, 224, 224) float on this device, normalised -> (n, dim) float32."""
        if not x.is_cuda:
            raise RuntimeError("ResNetEngine expects CUDA input (no CPU fallback)")
        x = x.to(torch.float32).contiguous()
        return torch.ops.vfeat.resnet_forward(int(self._h.value), self.dim, x)    # custom op over vf_resnet_forward_f32

    def forward_frames_u8(self, frames: torch.Tensor, swap_rb: bool = False) -> torch.Tensor:
        """(n, H, W, 3) uint8 frames on this device -> Resize(256) -> CenterCrop(224) -> normalise -> net -> (n, dim).
        ``swap_rb``: the frames are BGR (as cv2 decodes them) and are read as RGB."""
        assert frames.is_cuda and frames.dtype == torch.uint8 and frames.dim() == 4 and frames.shape[3] == 3
        frames = frames.contiguous()
        n, H, W, _ = frames.shape
        out = torch.empty((n, self.dim), device=frames.device, dtype=torch.float32)
        with torch.cuda.device(self.device):
            check(lib().vf_resnet_forward_u8(self._h, frames.data_ptr(), n, H, W, int(swap_rb), out.data_ptr(),
                                             torch.cuda.current_stream().cuda_stream))
        return out

    def forward_frames_u8_host(self, frames: torch.Tensor, swap_rb: bool = False, group: int = 256, wait: bool = True):
        """The same from HOST frames (n, H, W, 3) uint8 (pinned memory for asynchronous copies): the host->device copy
        of group k+1 runs on a copy stream while group k is in the network.  Returns (n, dim) float32 on the host.
        ``wait=False`` returns ``(features, event)`` as soon as everything is enqueued -- the features (pinned) are valid
        after ``event.synchronize()``; ``frames`` must stay untouched until then."""
        assert not frames.is_cuda and frames.dtype == torch.uint8 and frames.dim() == 4 and frames.shape[3] == 3
        n = frames.shape[0]
        out = torch.empty((n, self.dim), dtype=torch.float32).pin_memory()
        if n == 0:
            return out if wait else (out, None)
        with torch.cuda.device(self.device):
            main = torch.cuda.current_stream()
            copy = getattr(self, "_copy_stream", None)
            if copy is None:
                copy = self._copy_stream = torch.cuda.Stream(device=self.device)
            bufs, ready, freed = [None, None], [None, None], [None, None]
            groups = [(a, min(n, a + group)) for a in range(0, n, group)]

            def stage(k):
                a, b = groups[k]
                with torch.cuda.stream(copy):
                    if freed[k & 1] is not None:
                        copy.wait_event(freed[k & 1])          # the network has finished reading this buffer
                    bufs[k & 1] = frames[a:b].to(self.device, non_blocking=True)
                    ready[k & 1] = torch.cuda.Event()
                    ready[k & 1].record(copy)

            stage(0)
            for k, (a, b) in enumerate(groups):
                if k + 1 < len(groups):
                    stage(k + 1)
                main.wait_event(ready[k & 1])
                y = self.forward_frames_u8(bufs[k & 1], swap_rb)
                bufs[k & 1].record_stream(main)
                freed[k & 1] = torch.cuda.Event()
                freed[k & 1].record(main)
                out[a:b].copy_(y, non_blocking=True)
            if not wait:
                done = torch.cuda.Event(blocking=True)
                done.record(main)
                return out, done
            main.synchronize()
        return out

    def read_stage(self, stage: int) -> torch.Tensor:
        """Diagnostics: stage 0 (stem + max pool) .. 4 (layer4) of the last chunk of the last call as fp32 NCHW."""
        dims = (C.c_int * 4)()
        check(lib().vf_resnet_read_stage(self._h, stage, None, 0, dims, None))
        out = torch.empty(tuple(dims), device=self.device, dtype=torch.float32)
        with torch.cuda.device(self.device):
            check(lib().vf_resnet_read_stage(self._h, stage, out.data_ptr(), out.numel(), dims,
                                             torch.cuda.current_stream().cuda_stream))
        return out

    @property
    def launch_count(self) -> int:
        return int(lib().vf_resnet_launch_count(self._h))

    def close(self):
        if getattr(self, "_h", None):
            lib().vf_resnet_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def normalize_u8(frames: torch.Tensor, swap_rb: bool = False) -> torch.Tensor:
    """CenterCrop(224) + ToTensor + Normalize(ImageNet) of resized (n, H, W, 3) uint8 frames on the device ->
    (n, 3, 224, 224) fp32, bit-exact with torchvision."""
    assert frames.is_cuda and frames.dtype == torch.uint8 and frames.dim() == 4 and frames.shape[3] == 3
    frames = frames.contiguous()
    n, h, w, _ = frames.shape
    out = torch.empty((n, 3, 224, 224), device=frames.device, dtype=torch.float32)
    with torch.cuda.device(frames.device):
        check(lib().vf_imagenet_normalize_u8(frames.data_ptr(), n, h, w, int(swap_rb), out.data_ptr(),
                                             torch.cuda.current_stream().cuda_stream))
    return out
