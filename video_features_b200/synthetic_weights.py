"""Seeded synthetic weights in the layouts the engines load -- for benchmarks and tests on machines without the real
checkpoints (the reference downloads ViT-B-32.pt at run time, models/CLIP/extract_clip.py:47; there is no network
here).  ``VF_CLIP_SYNTHETIC=<seed>[:outliers]`` makes ``ExtractCLIP`` use them instead of a checkpoint file.
"""
from __future__ import annotations

from collections import OrderedDict

import torch

WIDTH, LAYERS, TOKENS, PATCH, MLP, EMBED = 768, 12, 50, 32, 3072, 512


def clip_vit_b16_state_dict(seed: int = 0, outliers: bool = False) -> "OrderedDict[str, torch.Tensor]":
    """The same for the ViT-B/16 tower (16-pixel patches, 197 tokens)."""
    return clip_vit_b32_state_dict(seed, outliers, patch=16)


def clip_vit_b32_state_dict(seed: int = 0, outliers: bool = False, patch: int = PATCH) -> "OrderedDict[str, torch.Tensor]":
    """openai ``visual.*`` key layout, fp32.  Initialisation scales are the ones openai/CLIP's
    ``initialize_parameters`` uses (width**-0.5 etc.), with perturbed LayerNorm gains / biases so that every term of the
    forward matters.

    ``outliers=True`` adds what trained ViT-B/32 weights have and random ones lack: a handful of residual-stream
    channels that carry magnitudes of 50-200 through every block (set up by the positional embedding and fed by the
    projection biases), LayerNorm gains with a heavy tail (a few entries near 0.05, a few above 4), and a few large
    rows in the attention / MLP output projections.  This is the regime where fp16 storage of intermediate tensors is
    most at risk."""
    g = torch.Generator().manual_seed(seed)

    def rn(*shape, std=1.0):
        return torch.randn(*shape, generator=g, dtype=torch.float32) * std

    scale = WIDTH ** -0.5
    attn_std = WIDTH ** -0.5
    proj_std = (WIDTH ** -0.5) * ((2 * LAYERS) ** -0.5)
    fc_std = (2 * WIDTH) ** -0.5
    sd: "OrderedDict[str, torch.Tensor]" = OrderedDict()
    sd["visual.class_embedding"] = rn(WIDTH, std=scale)
    sd["visual.positional_embedding"] = rn((224 // patch) ** 2 + 1, WIDTH, std=scale)
    sd["visual.proj"] = rn(WIDTH, EMBED, std=scale)
    sd["visual.conv1.weight"] = rn(WIDTH, 3, patch, patch, std=(3 * patch * patch) ** -0.5)
    for name in ("ln_pre", "ln_post"):
        sd[f"visual.{name}.weight"] = 1.0 + rn(WIDTH, std=0.1)
        sd[f"visual.{name}.bias"] = rn(WIDTH, std=0.05)
    for i in range(LAYERS):
        p = f"visual.transformer.resblocks.{i}."
        sd[p + "attn.in_proj_weight"] = rn(3 * WIDTH, WIDTH, std=attn_std)
        sd[p + "attn.in_proj_bias"] = rn(3 * WIDTH, std=0.02)
        sd[p + "attn.out_proj.weight"] = rn(WIDTH, WIDTH, std=proj_std)
        sd[p + "attn.out_proj.bias"] = rn(WIDTH, std=0.02)
        sd[p + "ln_1.weight"] = 1.0 + rn(WIDTH, std=0.1)
        sd[p + "ln_1.bias"] = rn(WIDTH, std=0.05)
        sd[p + "mlp.c_fc.weight"] = rn(MLP, WIDTH, std=fc_std)
        sd[p + "mlp.c_fc.bias"] = rn(MLP, std=0.02)
        sd[p + "mlp.c_proj.weight"] = rn(WIDTH, MLP, std=proj_std)
        sd[p + "mlp.c_proj.bias"] = rn(WIDTH, std=0.02)
        sd[p + "ln_2.weight"] = 1.0 + rn(WIDTH, std=0.1)
        sd[p + "ln_2.bias"] = rn(WIDTH, std=0.05)
    if outliers:
        dims = torch.randperm(WIDTH, generator=g)[:6]
        sign = torch.tensor([1.0, -1.0, 1.0, -1.0, 1.0, -1.0])
        # ln_pre rescales whatever the embedding holds, so the outlier channels are planted in ln_pre's affine part:
        # the residual stream leaves ln_pre with +-(60..150) in these channels
        sd["visual.ln_pre.bias"][dims] = sign * (60.0 + 90.0 * torch.rand(6, generator=g))
        sd["visual.ln_pre.weight"][dims] = 8.0
        for i in range(LAYERS):
            p = f"visual.transformer.resblocks.{i}."
            for ln in ("ln_1", "ln_2"):
                w = sd[p + ln + ".weight"]
                w.mul_(torch.exp(rn(WIDTH, std=0.35)))                       # heavy-tailed gains
                w[dims[:3]] = 0.05 + 0.05 * torch.rand(3, generator=g)       # trained nets damp their outlier channels ...
                w[dims[3:]] = 3.0 + 2.0 * torch.rand(3, generator=g)         # ... or read them loudly
                sd[p + ln + ".bias"][dims] = rn(6, std=0.5)
            # the projections keep feeding the outlier channels (bias) and have a few loud rows
            sd[p + "attn.out_proj.bias"][dims] = sign * (1.0 + 2.0 * torch.rand(6, generator=g))
            sd[p + "mlp.c_proj.bias"][dims] = sign * (2.0 + 4.0 * torch.rand(6, generator=g))
            loud = torch.randperm(WIDTH, generator=g)[:4]
            sd[p + "attn.out_proj.weight"][loud] *= 6.0
            sd[p + "mlp.c_proj.weight"][loud] *= 6.0
        sd["visual.ln_post.weight"][dims] = 0.05
    return sd


# torchvision resnet{depth}: block type and blocks per stage (torchvision/models/resnet.py)
RESNET_BLOCKS = {18: ("basic", (2, 2, 2, 2)), 34: ("basic", (3, 4, 6, 3)), 50: ("bottleneck", (3, 4, 6, 3)),
                 101: ("bottleneck", (3, 4, 23, 3)), 152: ("bottleneck", (3, 8, 36, 3))}


def resnet_feature_dim(depth: int) -> int:
    return 512 if RESNET_BLOCKS[depth][0] == "basic" else 2048


def resnet_conv_shapes(depth: int) -> "OrderedDict[str, tuple]":
    """torchvision key prefix of every conv -> (cout, cin, k), with the BN that follows it at the same prefix with
    ``conv`` -> ``bn`` (``downsample.0`` -> ``downsample.1``)."""
    kind, blocks = RESNET_BLOCKS[depth]
    exp = 1 if kind == "basic" else 4
    shapes: "OrderedDict[str, tuple]" = OrderedDict()
    shapes["conv1"] = (64, 3, 7)
    cin = 64
    for li, nb in enumerate(blocks):
        planes = 64 << li
        for b in range(nb):
            p = f"layer{li + 1}.{b}"
            if kind == "basic":
                shapes[p + ".conv1"] = (planes, cin, 3)
                shapes[p + ".conv2"] = (planes, planes, 3)
            else:
                shapes[p + ".conv1"] = (planes, cin, 1)
                shapes[p + ".conv2"] = (planes, planes, 3)
                shapes[p + ".conv3"] = (planes * 4, planes, 1)
            if b == 0 and (li > 0 or cin != planes * exp):
                shapes[p + ".downsample.0"] = (planes * exp, cin, 1)
            cin = planes * exp
    return shapes


def resnet_bn_name(conv: str) -> str:
    return conv[:-1] + "1" if conv.endswith("downsample.0") else conv.replace("conv", "bn")


def resnet_state_dict(depth: int, seed: int = 0) -> "OrderedDict[str, torch.Tensor]":
    """torchvision ``resnet{depth}`` key layout, fp32 (``fc.*`` and ``num_batches_tracked`` included, as in a real
    checkpoint).  He-scaled convs and mild BN statistics; the last BN gain of every residual branch is damped to
    0.2 (bn2 of a BasicBlock, bn3 of a Bottleneck), so that the residual stream stays O(1) through 50 blocks instead of
    growing with depth (tests/test_resnet_cpu.py holds the per-stage RMS in a band)."""
    g = torch.Generator().manual_seed(seed)
    kind = RESNET_BLOCKS[depth][0]
    last = ".bn2" if kind == "basic" else ".bn3"
    sd: "OrderedDict[str, torch.Tensor]" = OrderedDict()
    for name, (co, ci, k) in resnet_conv_shapes(depth).items():
        sd[name + ".weight"] = torch.randn(co, ci, k, k, generator=g) * (2.0 / (ci * k * k)) ** 0.5
        bn = resnet_bn_name(name)
        gain = 0.2 if bn.endswith(last) else 1.0
        sd[bn + ".weight"] = gain * (1.0 + 0.1 * torch.randn(co, generator=g))
        sd[bn + ".bias"] = 0.05 * torch.randn(co, generator=g)
        sd[bn + ".running_mean"] = 0.05 * torch.randn(co, generator=g)
        sd[bn + ".running_var"] = 1.0 + 0.1 * torch.rand(co, generator=g)
        sd[bn + ".num_batches_tracked"] = torch.tensor(0, dtype=torch.int64)
    d = resnet_feature_dim(depth)
    sd["fc.weight"] = torch.randn(1000, d, generator=g) * d ** -0.5
    sd["fc.bias"] = torch.zeros(1000)
    return sd


def parse_env(value: str):
    """``VF_CLIP_SYNTHETIC`` value -> (seed, outliers): "3", "3:outliers", "" (seed 0)."""
    head, _, tail = (value or "").partition(":")
    return int(head or 0), tail.strip().lower() == "outliers"
