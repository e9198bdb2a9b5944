"""Seeded stand-ins for the reference's vendored checkpoints (models/i3d/checkpoints/i3d_{rgb,flow}.pt,
models/raft/checkpoints/raft-sintel.pth; 120 MB, not part of this repository).

A stand-in has the vendored file's keys and shapes; every tensor is drawn from a normal distribution with that tensor's
mean and standard deviation, clamped to its range, as recorded in tests/golden/checkpoint_stats.npz
(scripts/make_golden.py standin).  The tests and the I3D / RAFT legs of bench.py run on them.
"""
from __future__ import annotations

import functools
import os
from collections import OrderedDict

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CHECKPOINT_STATS = os.path.join(ROOT, "tests", "golden", "checkpoint_stats.npz")
NAMES = ("i3d_rgb.pt", "i3d_flow.pt", "raft-sintel.pth")
SEEDS = {"i3d_rgb.pt": 1, "i3d_flow.pt": 2, "raft-sintel.pth": 9}
# Random RAFT weights make the 20-step refinement chaotic (flows of hundreds of px; a 1e-6 relative weight perturbation
# moves the output by 1e-2).  Scaling the flow head's output by this gain keeps the iteration well conditioned.  With
# the seed above the same perturbation moves the output by 3e-6 at 128x160 and 200x200, as with raft-sintel.pth (other
# seeds give 3e-6 .. 2e-5); the mean |flow| is 9 px.  (fp32 oracle on the CPU, oracle/raft_net.py.)  The gain is split
# over the head's two convs (ReLU between them commutes with a positive scale).  A smaller gain gives smaller flows, but
# pushes the head's weights and activations towards the fp16 subnormal range, where the engine's split-fp16 operands
# lose precision; the trained ones stay clear of it.
RAFT_FLOW_HEAD_GAIN = 0.03
# The mask head's logits are halved.  The trained network's low-resolution flow is smooth, so rounding of the mask logits
# hardly moves the convex upsampling; the stand-in's flow is rough, and halving its logits halves the rounding error the
# upsampling adds.  Engine vs fp32 oracle after one iteration on a B200, as printed by
# tests/test_raft_gpu.py::test_raft_stages_and_one_iteration ("flow_up after 1 iteration", run with -s): rel-L2
# 1.0e-4 with a gain of 1.0, 4.9e-5 with 0.5; the low-resolution flow before the upsampling: 1.9e-5 either way.
RAFT_MASK_GAIN = 0.5


@functools.lru_cache(maxsize=None)
def _standin(name: str) -> "OrderedDict[str, torch.Tensor]":
    st = np.load(CHECKPOINT_STATS)
    keys, ndim, dims, stats = (st[f"{name}/{f}"] for f in ("keys", "ndim", "dims", "stats"))
    g = torch.Generator().manual_seed(SEEDS[name])
    sd, at = OrderedDict(), 0
    for key, nd, (mean, std, lo, hi, is_float) in zip(keys, ndim, stats):
        shape = tuple(int(d) for d in dims[at:at + nd])
        at += nd
        if not is_float:
            sd[str(key)] = torch.full(shape, int(mean), dtype=torch.int64)
            continue
        x = torch.randn(shape, generator=g, dtype=torch.float64) * std + mean
        sd[str(key)] = x.clamp(lo, hi).float()
    if name == "raft-sintel.pth":
        head = "module.update_block.flow_head."
        for k in ("conv1.weight", "conv1.bias", "conv2.weight"):
            sd[head + k] *= RAFT_FLOW_HEAD_GAIN ** 0.5
        sd[head + "conv2.bias"] *= RAFT_FLOW_HEAD_GAIN
        for k in ("mask.2.weight", "mask.2.bias"):
            sd["module.update_block." + k] *= RAFT_MASK_GAIN
    return sd


def state_dict(name: str) -> "OrderedDict[str, torch.Tensor]":
    """The stand-in for `name` (one of NAMES).  Returns a fresh copy: callers may move or modify it."""
    return OrderedDict((k, v.clone()) for k, v in _standin(name).items())
