"""RAFT flow through the C ABI against the fp32 oracle (oracle/raft_net.py, pinned bit-for-bit to the reference
module) and against the reference module's own output (tests/golden/standin_outputs.npz).

Bar (SURVEY 8d): rel-L2 <= 1e-3 and max-abs <= 1e-3 * max|ref| on the flow field.  RAFT's 20 refinement steps amplify
operand rounding by two to three orders of magnitude on hard inputs (the fp32 oracle itself moves by 2.5e-5 between 1
and 16 CPU threads on block-compressed frames), so the engine carries EVERY GEMM operand as a split-fp16 pair
(activations [hi | lo] with duplicated weight columns, weights as hi + lo passes, DESIGN.md §2).  Measured: rel-L2
5.5e-6 / max 3.8e-5 at 128x160, 1.7e-5 / 1.8e-4 at 270x480, 5.7e-5 on block-compressed video
(test_extract_i3d_raft_gpu.py) -- both parts of the bar are met with margin.  (Those figures are for the vendored
raft-sintel.pth.)  The weights are a seeded stand-in of that checkpoint (oracle/checkpoint_standins.py): plain random
weights make RAFT's iteration chaotic, so the stand-in damps the flow head to keep it well conditioned."""
import os

import numpy as np
import pytest
import torch

import video_features_b200  # noqa: F401

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _err(y, ref):
    y, ref = y.double().cpu(), ref.double().cpu()
    return float((y - ref).norm() / ref.norm()), float((y - ref).abs().max() / ref.abs().max())


@pytest.fixture(scope="module")
def raft(cuda_device):
    from helpers import checkpoint
    from video_features_b200.raft_engine import RAFTEngine
    sd = checkpoint("raft-sintel.pth")
    eng = RAFTEngine(sd, 0, max_frames=5, max_h=272, max_w=480)
    yield sd, eng
    eng.close()


def test_raft_stages_and_one_iteration(raft, cuda_device):
    """Encoders, correlation lookup and one GRU step against the oracle's intermediates."""
    from oracle import raft_net as R
    sd, eng = raft
    sdg = {k: v.to(cuda_device) for k, v in R._strip(sd).items()}
    fr = R.synthetic_frames(3, 128, 160, seed=128)
    x = fr.to(cuda_device)
    y1 = eng.flow(x, iters=1, unpad=False)
    img = 2 * (x / 255.0) - 1.0
    fmap = R.encoder(sdg, "fnet", img, "instance")
    e = _err(eng.debug_read(0), fmap)
    print("fnet features:", e)
    cnet = R.encoder(sdg, "cnet", img[:-1], "batch")
    e2 = _err(eng.debug_read(1), cnet)
    print("cnet output:", e2)
    # measured on a B200 with the stand-in: 5.6e-6 / 2.0e-6 (vendored checkpoint: 3.8e-6 / 6.8e-6)
    assert e[0] < 1e-4 and e2[0] < 1e-4
    # first lookup (coords = grid) against the oracle's pyramid lookup
    pyr = R.corr_pyramid(fmap[:-1].float(), fmap[1:].float())
    H8, W8 = 16, 20
    ys, xs = torch.meshgrid(torch.arange(H8), torch.arange(W8), indexing="ij")
    coords0 = torch.stack([xs, ys], 0).float()[None].repeat(2, 1, 1, 1).to(cuda_device)
    look = R.corr_lookup(pyr, coords0)
    eng.flow(x, iters=1, unpad=False)
    e = _err(eng.debug_read(4), look)       # (the last lookup of a 1-iteration run is the first one)
    print("corr lookup:", e)
    assert e[0] < 1e-4                          # measured with the stand-in: 3.5e-6
    ref1, low1 = R.forward(sd_to(sd, cuda_device), x[:-1], x[1:], 1, return_lowres=True)
    e = _err(eng.debug_read(3), low1)
    print("low-res flow after 1 iteration:", e)
    assert e[0] < 1e-4                          # measured with the stand-in: 1.9e-5
    e = _err(y1, ref1)
    print("flow_up after 1 iteration:", e)
    assert e[0] < 1e-4 and e[1] < 1e-3          # measured with the stand-in: 4.9e-5 / 1.8e-4


def test_raft_odd_map_size(raft, cuda_device):
    """200x200 frames: the 25x25 = 625-position /8 map is not a multiple of 8 (padded GEMM width, odd pooling sizes)."""
    from oracle import raft_net as R
    sd, eng = raft
    x = R.synthetic_frames(2, 200, 200, seed=7).to(cuda_device)
    y = eng.flow(x, iters=12, unpad=True)
    ref = R.forward(sd_to(sd, cuda_device), x[:-1], x[1:], 12)
    rel, mx = _err(y, ref)
    print(f"200x200: rel-L2 {rel:.3e} max {mx:.3e}")
    assert torch.isfinite(y).all() and rel < 1e-4 and mx < 1e-3     # measured with the stand-in: 2.6e-5 / 1.4e-4


def sd_to(sd, dev):
    return {k: v.to(dev) for k, v in sd.items()}


@pytest.mark.parametrize("h,w,n", [(128, 160, 3), (270, 480, 2)])
def test_raft_20_iterations_vs_oracle_and_reference_golden(raft, cuda_device, h, w, n):
    from oracle import raft_net as R
    sd, eng = raft
    fr = R.synthetic_frames(n, h, w, seed=h)
    x = fr.to(cuda_device)
    y = eng.flow(x, iters=20, unpad=True)
    xp = R.pad(x)
    ref = R.unpad(R.forward(sd_to(sd, cuda_device), xp[:-1], xp[1:], 20), h, w)
    rel, mx = _err(y, ref)
    print(f"{h}x{w}: vs oracle rel-L2 {rel:.3e} max {mx:.3e}; mean |flow| {float(ref.abs().mean()):.3f}; launches {eng.launch_count}")
    d = (y.double().cpu() - ref.double().cpu()).abs().flatten()
    print(f"    abs err px: max {float(d.max()):.4f}  p99.9 {float(d.kthvalue(int(d.numel() * 0.999)).values):.4f}  "
          f"median {float(d.median()):.5f}  (max |flow| {float(ref.abs().max()):.3f})")
    # north-star bars 1e-3; measured on a B200 with the stand-in: rel 3.0e-5 / 2.1e-5 (vendored checkpoint: 5.5e-6 /
    # 1.7e-5), max-abs 1.6e-4 / 1.4e-4 (vendored: 3.8e-5 / 1.8e-4)
    assert rel < 1e-4
    assert mx < 1e-3
    fixture = np.load(os.path.join(ROOT, "tests", "golden", "standin_outputs.npz"))
    gold, stride = fixture[f"raft_flow_{h}x{w}"], int(fixture[f"raft_stride_{h}x{w}"])     # a strided grid of the flow
    got = y.cpu().numpy()[:, :, ::stride, ::stride]
    rel_g = float(np.linalg.norm(got - gold) / np.linalg.norm(gold))
    print(f"{h}x{w}: vs reference-module golden rel-L2 {rel_g:.3e}")
    assert rel_g < 1e-4
    # uint8 HWC entry == float CHW entry on integer-valued frames
    y8 = eng.flow(fr.permute(0, 2, 3, 1).contiguous().to(torch.uint8).to(cuda_device), iters=20, unpad=True)
    assert torch.equal(y8, y)
    # unpadded window of the padded output
    yp = eng.flow(x, iters=20, unpad=False)
    assert torch.equal(R.unpad(yp, h, w), y)


def test_raft_graph_cache_is_bounded(raft, cuda_device):
    """More distinct (frames, H, W, iterations) keys than the engine keeps graphs for: evicted graphs are re-captured on
    the next use and the results do not change."""
    from oracle import raft_net as R
    sd, eng = raft
    x = R.synthetic_frames(3, 64, 96, seed=5).to(cuda_device)
    first = eng.flow(x, iters=2).clone()
    for k in range(18):                                    # 18 further keys (the cache holds 16)
        eng.flow(R.synthetic_frames(2, 64 + 8 * (k % 6), 96 + 8 * (k // 6), seed=k).to(cuda_device), iters=2)
    again = eng.flow(x, iters=2)
    torch.cuda.synchronize()
    # (InstanceNorm statistics are accumulated with atomics: the sum order, hence the last bits, may differ between runs)
    assert float((first - again).abs().max()) <= 1e-4 * float(first.abs().max())
