"""fp32 restatement of the reference's RAFT (full model, test_mode) -- test oracle only.

Follows models/raft/raft_src/: raft.py (InputPadder :27-44, RAFT.forward :115-174, upsample_flow :100-111),
extractor.py (BasicEncoder :118-192, ResidualBlock :6-56), corr.py (CorrBlock :12-60, incl. the transposed 9x9
window), update.py (BasicMotionEncoder :83-101, SepConvGRU :37-64, FlowHead :10-18, BasicUpdateBlock :118-139),
utils/utils.py (bilinear_sampler :57-71, coords_grid :74-77).  Functional, driven by the checkpoint's own state dict
(raft-sintel.pth, keys prefixed ``module.``).  Pinned against the reference module: bit-identical with the vendored
checkpoint (scripts/make_golden.py raft -> tests/golden/raft_outputs.npz, kept as the record of that check) and on the
checkpoint stand-in the tests use (scripts/make_golden.py standin -> tests/golden/standin_outputs.npz).
"""
from __future__ import annotations

from typing import Dict

import torch
import torch.nn.functional as F

CORR_LEVELS, CORR_RADIUS, HDIM, CDIM = 4, 4, 128, 128


def pad_amounts(ht: int, wd: int):
    """InputPadder(mode='sintel'): [left, right, top, bottom] replicate padding to multiples of 8 (raft.py:29-34)."""
    pad_ht = (((ht // 8) + 1) * 8 - ht) % 8
    pad_wd = (((wd // 8) + 1) * 8 - wd) % 8
    return [pad_wd // 2, pad_wd - pad_wd // 2, pad_ht // 2, pad_ht - pad_ht // 2]


def pad(x: torch.Tensor) -> torch.Tensor:
    return F.pad(x, pad_amounts(*x.shape[-2:]), mode='replicate')


def unpad(x: torch.Tensor, ht: int, wd: int) -> torch.Tensor:
    p = pad_amounts(ht, wd)
    H, W = x.shape[-2:]
    return x[..., p[2]:H - p[3], p[0]:W - p[1]]


def _strip(sd):
    return {(k[7:] if k.startswith("module.") else k): v for k, v in sd.items()}


def _conv(sd, name, x, stride=1, padding=0):
    return F.conv2d(x, sd[name + ".weight"], sd[name + ".bias"], stride=stride, padding=padding)


def _norm(sd, name, x, kind):
    if kind == "instance":      # nn.InstanceNorm2d: no affine, no running stats, eps 1e-5
        return F.instance_norm(x, eps=1e-5)
    if kind == "batch":         # eval-mode BatchNorm2d
        return F.batch_norm(x, sd[name + ".running_mean"], sd[name + ".running_var"], sd[name + ".weight"],
                            sd[name + ".bias"], False, 0.0, 1e-5)
    raise ValueError(kind)


def _resblock(sd, p, x, kind, stride):
    y = F.relu(_norm(sd, p + ".norm1", _conv(sd, p + ".conv1", x, stride, 1), kind))
    y = F.relu(_norm(sd, p + ".norm2", _conv(sd, p + ".conv2", y, 1, 1), kind))
    if stride != 1:
        # downsample = Sequential(conv1x1 stride, norm3); norm3 is registered both as p.norm3 and p.downsample.1
        x = _norm(sd, p + ".downsample.1", _conv(sd, p + ".downsample.0", x, stride, 0), kind)
    return F.relu(x + y)


def encoder(sd, p, x, kind):
    """BasicEncoder.forward (extractor.py:168-192)."""
    x = F.relu(_norm(sd, p + ".norm1", _conv(sd, p + ".conv1", x, 2, 3), kind))
    for layer, stride in (("layer1", 1), ("layer2", 2), ("layer3", 2)):
        x = _resblock(sd, f"{p}.{layer}.0", x, kind, stride)
        x = _resblock(sd, f"{p}.{layer}.1", x, kind, 1)
    return _conv(sd, p + ".conv2", x)


def corr_pyramid(fmap1, fmap2):
    """CorrBlock.__init__ / .corr (corr.py:13-27,52-60)."""
    b, d, h, w = fmap1.shape
    c = torch.matmul(fmap1.view(b, d, h * w).transpose(1, 2), fmap2.view(b, d, h * w))
    c = c.view(b, h, w, 1, h, w) / torch.sqrt(torch.tensor(d).float())
    c = c.reshape(b * h * w, 1, h, w)
    pyr = [c]
    for _ in range(CORR_LEVELS - 1):
        c = F.avg_pool2d(c, 2, stride=2)
        pyr.append(c)
    return pyr


def _bilinear_sampler(img, coords):
    H, W = img.shape[-2:]
    xg, yg = coords.split([1, 1], dim=-1)
    xg = 2 * xg / (W - 1) - 1
    yg = 2 * yg / (H - 1) - 1
    return F.grid_sample(img, torch.cat([xg, yg], dim=-1), align_corners=True)


def corr_lookup(pyr, coords):
    """CorrBlock.__call__ (corr.py:29-50).  NB the window: delta = stack(meshgrid(dy, dx)) is added to (x, y), so
    window axis 0 offsets x and axis 1 offsets y (the trained weights depend on it)."""
    r = CORR_RADIUS
    coords = coords.permute(0, 2, 3, 1)
    b, h1, w1, _ = coords.shape
    out = []
    for i in range(CORR_LEVELS):
        dx = torch.linspace(-r, r, 2 * r + 1)
        dy = torch.linspace(-r, r, 2 * r + 1)
        delta = torch.stack(torch.meshgrid(dy, dx, indexing="ij"), dim=-1).to(coords.device)
        centroid = coords.reshape(b * h1 * w1, 1, 1, 2) / 2 ** i
        c = _bilinear_sampler(pyr[i], centroid + delta.view(1, 2 * r + 1, 2 * r + 1, 2))
        out.append(c.view(b, h1, w1, -1))
    return torch.cat(out, dim=-1).permute(0, 3, 1, 2).contiguous().float()


def motion_encoder(sd, flow, corr):
    p = "update_block.encoder."
    cor = F.relu(_conv(sd, p + "convc1", corr))
    cor = F.relu(_conv(sd, p + "convc2", cor, 1, 1))
    flo = F.relu(_conv(sd, p + "convf1", flow, 1, 3))
    flo = F.relu(_conv(sd, p + "convf2", flo, 1, 1))
    out = F.relu(_conv(sd, p + "conv", torch.cat([cor, flo], 1), 1, 1))
    return torch.cat([out, flow], 1)


def sep_conv_gru(sd, h, x):
    p = "update_block.gru."
    for sfx, pd in (("1", (0, 2)), ("2", (2, 0))):
        hx = torch.cat([h, x], 1)
        z = torch.sigmoid(_conv(sd, p + "convz" + sfx, hx, 1, pd))
        r = torch.sigmoid(_conv(sd, p + "convr" + sfx, hx, 1, pd))
        q = torch.tanh(_conv(sd, p + "convq" + sfx, torch.cat([r * h, x], 1), 1, pd))
        h = (1 - z) * h + z * q
    return h


def upsample_flow(flow, mask):
    N, _, H, W = flow.shape
    mask = torch.softmax(mask.view(N, 1, 9, 8, 8, H, W), dim=2)
    up = F.unfold(8 * flow, [3, 3], padding=1).view(N, 2, 9, 1, 1, H, W)
    up = torch.sum(mask * up, dim=2).permute(0, 1, 4, 2, 5, 3)
    return up.reshape(N, 2, 8 * H, 8 * W)


@torch.no_grad()
def forward(sd_in: Dict[str, torch.Tensor], image1: torch.Tensor, image2: torch.Tensor, iters: int = 20,
            return_lowres: bool = False):
    """RAFT.forward(image1, image2, iters=20, test_mode=True) -> flow_up (B,2,H,W); images float [0,255], H,W % 8 == 0."""
    sd = _strip(sd_in)
    image1 = 2 * (image1 / 255.0) - 1.0
    image2 = 2 * (image2 / 255.0) - 1.0
    f = encoder(sd, "fnet", torch.cat([image1, image2], 0), "instance")
    fmap1, fmap2 = torch.split(f, [image1.shape[0]] * 2, 0)
    pyr = corr_pyramid(fmap1.float(), fmap2.float())
    cnet = encoder(sd, "cnet", image1, "batch")
    net, inp = torch.split(cnet, [HDIM, CDIM], 1)
    net, inp = torch.tanh(net), torch.relu(inp)
    N, _, H, W = image1.shape
    ys, xs = torch.meshgrid(torch.arange(H // 8), torch.arange(W // 8), indexing="ij")
    coords0 = torch.stack([xs, ys], 0).float()[None].repeat(N, 1, 1, 1).to(image1.device)
    coords1 = coords0.clone()
    flow_up = None
    for _ in range(iters):
        corr = corr_lookup(pyr, coords1)
        flow = coords1 - coords0
        x = torch.cat([inp, motion_encoder(sd, flow, corr)], 1)
        net = sep_conv_gru(sd, net, x)
        p = "update_block.flow_head."
        delta = _conv(sd, p + "conv2", F.relu(_conv(sd, p + "conv1", net, 1, 1)), 1, 1)
        coords1 = coords1 + delta
    mask = 0.25 * _conv(sd, "update_block.mask.2", F.relu(_conv(sd, "update_block.mask.0", net, 1, 1)))
    flow_up = upsample_flow(coords1 - coords0, mask)      # only the last iteration's result is returned (raft.py:172)
    return (flow_up, coords1 - coords0) if return_lowres else flow_up


def synthetic_frames(n: int, h: int, w: int, seed: int = 0, shift=(1.7, -0.9)) -> torch.Tensor:
    """Smooth textured frames translating by a sub-pixel shift per frame (non-degenerate flow): (n,3,h,w) in [0,255]."""
    g = torch.Generator().manual_seed(seed)
    base = torch.rand(1, 3, h // 4 + 8, w // 4 + 8, generator=g)
    base = F.interpolate(base, size=(h + 64, w + 64), mode="bicubic", align_corners=False).clamp(0, 1)
    ys, xs = torch.meshgrid(torch.arange(h).float(), torch.arange(w).float(), indexing="ij")
    out = []
    for i in range(n):
        gx = (xs + 32 + shift[0] * i) / (w + 63) * 2 - 1
        gy = (ys + 32 + shift[1] * i) / (h + 63) * 2 - 1
        out.append(F.grid_sample(base, torch.stack([gx, gy], -1)[None], align_corners=True)[0])
    return (torch.stack(out) * 255).round()
