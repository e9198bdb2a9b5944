"""fp32 restatement of torchvision's ResNet-18/34/50/101/152 forward with ``fc = Identity`` and of the ResNet
extractor's transform -- test oracle only.

The reference (models/resnet/extract_resnet.py:54-71) runs ``torchvision.models.resnet{depth}(pretrained=True)`` in eval
mode with ``fc`` replaced by ``Identity``: stem conv 7x7/2 pad 3 -> BN -> ReLU -> max pool 3x3/2 pad 1, layer1-4 of
BasicBlocks (18, 34) or Bottlenecks (50+, stride on the 3x3 conv: torchvision "v1.5"), global average pool.  Convs have
no bias, every BN is eval-mode with eps 1e-5.  Functional, driven by a state dict in torchvision's key layout.  Pinned
against torchvision itself (scripts/make_golden.py resnet -> tests/golden/resnet_outputs.npz).

The transform (extract_resnet.py:32-38) is ToPILImage -> Resize(256) (Pillow bilinear, short side) -> CenterCrop(224)
-> ToTensor -> Normalize(ImageNet mean / std); restated with oracle.pil_resample and torchvision's fp32 arithmetic.
"""
from __future__ import annotations

from typing import Dict

import numpy as np
import torch
import torch.nn.functional as F

from oracle import pil_resample

BN_EPS = 1e-5
MEAN = (0.485, 0.456, 0.406)
STD = (0.229, 0.224, 0.225)
RESIZE, CROP = 256, 224


def _bn(sd, p, x):
    return F.batch_norm(x, sd[p + ".running_mean"], sd[p + ".running_var"], sd[p + ".weight"], sd[p + ".bias"],
                        False, 0.0, BN_EPS)


def _block(sd, p, x, bottleneck, stride):
    if bottleneck:
        y = F.relu(_bn(sd, p + ".bn1", F.conv2d(x, sd[p + ".conv1.weight"])))
        y = F.relu(_bn(sd, p + ".bn2", F.conv2d(y, sd[p + ".conv2.weight"], stride=stride, padding=1)))
        y = _bn(sd, p + ".bn3", F.conv2d(y, sd[p + ".conv3.weight"]))
    else:
        y = F.relu(_bn(sd, p + ".bn1", F.conv2d(x, sd[p + ".conv1.weight"], stride=stride, padding=1)))
        y = _bn(sd, p + ".bn2", F.conv2d(y, sd[p + ".conv2.weight"], padding=1))
    if p + ".downsample.0.weight" in sd:
        x = _bn(sd, p + ".downsample.1", F.conv2d(x, sd[p + ".downsample.0.weight"], stride=stride))
    return F.relu(x + y)


@torch.no_grad()
def forward_features(sd: Dict[str, torch.Tensor], x: torch.Tensor, depth: int, return_stages: bool = False):
    """x (n, 3, 224, 224) normalised -> (n, D).  Stages: 0 = stem + max pool, 1..4 = layer1..4 outputs (NCHW)."""
    from video_features_b200.synthetic_weights import RESNET_BLOCKS
    kind, blocks = RESNET_BLOCKS[depth]
    st = []
    x = F.relu(_bn(sd, "bn1", F.conv2d(x, sd["conv1.weight"], stride=2, padding=3)))
    x = F.max_pool2d(x, 3, 2, 1)
    st.append(x)
    for li, nb in enumerate(blocks):
        for b in range(nb):
            x = _block(sd, f"layer{li + 1}.{b}", x, kind == "bottleneck", 2 if (b == 0 and li > 0) else 1)
        st.append(x)
    out = x.mean(dim=(2, 3))
    return (out, st) if return_stages else out


def resize_geometry(h: int, w: int, size: int = RESIZE):
    """torchvision Resize(int): short side -> size, long side int(size * long / short)."""
    return pil_resample.short_side_geometry(h, w, size)


def crop_offsets(h: int, w: int, size: int = CROP):
    """torchvision CenterCrop: int(round((d - size) / 2)) (Python round, half to even)."""
    return int(round((h - size) / 2.0)), int(round((w - size) / 2.0))


def transform(frame_rgb: np.ndarray) -> torch.Tensor:
    """One (H, W, 3) uint8 RGB frame -> (3, 224, 224) fp32, bit-exact with the reference's Compose."""
    h, w = frame_rgb.shape[:2]
    oh, ow = resize_geometry(h, w)
    r = pil_resample.resize(frame_rgb, oh, ow, pil_resample.BILINEAR)
    y0, x0 = crop_offsets(oh, ow)
    c = r[y0:y0 + CROP, x0:x0 + CROP]
    t = torch.from_numpy(np.ascontiguousarray(c)).permute(2, 0, 1).float().div(255)     # ToTensor
    mean = torch.tensor(MEAN, dtype=torch.float32).view(3, 1, 1)                          # Normalize: (x - m) / s
    std = torch.tensor(STD, dtype=torch.float32).view(3, 1, 1)
    return t.sub(mean).div(std)


def transform_batch(frames_rgb: np.ndarray) -> torch.Tensor:
    return torch.stack([transform(f) for f in frames_rgb])
