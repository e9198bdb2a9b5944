"""I3D features through the C ABI against the fp32 oracle (oracle/i3d_net.py, pinned to the reference module).

Bar (north_star): 1e-3 relative vs the fp32 torch path.  Synthetic weights, and seeded stand-ins of the reference's
vendored checkpoints with their per-tensor statistics (oracle/checkpoint_standins.py)."""
import os

import numpy as np
import pytest
import torch

import video_features_b200  # noqa: F401

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _rel(y, ref):
    y, ref = y.double().cpu(), ref.double().cpu()
    return float(((y - ref).norm(dim=-1) / ref.norm(dim=-1)).max()), float(
        ((y - ref).abs().amax(-1) / ref.abs().amax(-1)).max())


def _oracle_gpu(sd, x, dev, stages=False):
    from oracle import i3d_net
    sdg = {k: v.to(dev) for k, v in sd.items()}
    return i3d_net.forward_features(sdg, x.to(dev), return_stages=stages)


@pytest.mark.parametrize("modality,T", [("rgb", 16), ("flow", 12), ("rgb", 11)])
def test_i3d_synthetic_weights_vs_oracle(cuda_device, modality, T):
    from oracle import i3d_net
    from video_features_b200.i3d_engine import I3DEngine
    sd = i3d_net.synthetic_state_dict(modality, 0)
    cin = 3 if modality == "rgb" else 2
    x = torch.rand(2, cin, T, 224, 224, generator=torch.Generator().manual_seed(T)) * 2 - 1
    eng = I3DEngine(sd, modality, 0, max_stacks=2, max_T=16)
    y = eng(x.to(cuda_device))
    ref, st = _oracle_gpu(sd, x, cuda_device, stages=True)
    for sid, name in ((0, "1a"), (1, "2c"), (4, "5c")):
        got = eng.read_stage(sid)
        want = st[name]
        assert got.shape == want.shape, (name, got.shape, want.shape)
        err = float((got - want).norm() / want.norm())
        print(f"stage {name}: rel {err:.3e}")
        assert err < 5e-3, (name, err)
    rel, mx = _rel(y, ref)
    print(f"{modality} T={T}: rel-L2 {rel:.3e} max {mx:.3e}; launches {eng.launch_count}")
    assert rel < 1e-3 and mx < 1e-3
    eng.close()


@pytest.mark.parametrize("modality", ["rgb", "flow"])
def test_i3d_reference_checkpoint_vs_oracle_and_golden(cuda_device, modality):
    from helpers import checkpoint
    from video_features_b200.i3d_engine import I3DEngine
    sd = checkpoint(f"i3d_{modality}.pt")
    cin = 3 if modality == "rgb" else 2
    eng = I3DEngine(sd, modality, 0, max_stacks=1, max_T=64)
    gold = np.load(os.path.join(ROOT, "tests", "golden", "standin_outputs.npz"))
    for T in (16, 11):
        x = torch.rand(1, cin, T, 224, 224, generator=torch.Generator().manual_seed(100 + T)) * 2 - 1
        y = eng(x.to(cuda_device))
        ref = torch.from_numpy(gold[f"i3d_{modality}_T{T}"])      # the reference module's own output (fixture)
        rel, mx = _rel(y, ref)
        print(f"{modality} checkpoint stand-in T={T}: rel-L2 {rel:.3e} max {mx:.3e}")
        # measured on a B200 with the stand-ins: rel 5.2e-5 .. 2.7e-4, max 6.2e-5 .. 3.2e-4 (vendored checkpoints:
        # 1.9e-4 .. 4.0e-4 / 2.6e-4 .. 4.7e-4; pair tensors, DESIGN §2)
        assert rel < 6e-4 and mx < 1e-3
    x = torch.rand(1, cin, 64, 224, 224, generator=torch.Generator().manual_seed(5)) * 2 - 1
    y = eng(x.to(cuda_device))
    ref = _oracle_gpu(sd, x, cuda_device)
    rel, mx = _rel(y, ref)
    print(f"{modality} checkpoint stand-in T=64: rel-L2 {rel:.3e} max {mx:.3e}")
    assert rel < 6e-4 and mx < 1e-3          # measured with the stand-ins: 4.1e-5 .. 2.1e-4 / 4.0e-5 .. 2.2e-4
    eng.close()


def test_i3d_fused_stream_transforms(cuda_device):
    """forward_frames_u8 / forward_flow == oracle transform (extract_i3d.py:62-73) + oracle net on the same data,
    including the reference's quirks: floor-offset crop, +20 px flow quantised to 256."""
    from oracle import i3d_net
    from video_features_b200.i3d_engine import I3DEngine
    g = torch.Generator().manual_seed(3)
    # rgb: 12 resized frames 256x341 (the 4:3 sample geometry)
    sd = i3d_net.synthetic_state_dict("rgb", 1)
    frames = torch.randint(0, 256, (1, 12, 256, 341, 3), dtype=torch.uint8, generator=g)
    eng = I3DEngine(sd, "rgb", 0, max_stacks=1, max_T=16)
    y = eng.forward_frames_u8(frames.to(cuda_device))
    x = i3d_net.rgb_transform(frames[0].permute(0, 3, 1, 2).float())
    ref = _oracle_gpu(sd, x, cuda_device)
    rel, mx = _rel(y, ref)
    print(f"rgb u8 path: {rel:.3e} {mx:.3e}")
    assert rel < 1e-3 and mx < 1e-3
    # the fused transform must equal transform-then-forward bit for bit
    assert torch.equal(y, eng(x.to(cuda_device)))
    # a window stacks[:, :12] of longer (13-frame) stacks is read in place (the reference's rgb_stack[:-1]): same bits
    longer = torch.cat([frames, torch.randint(0, 256, (1, 1, 256, 341, 3), dtype=torch.uint8, generator=g)], 1).to(cuda_device)
    win = longer[:, :12]
    assert not win.is_contiguous() or win.shape[0] == 1
    assert torch.equal(eng.forward_frames_u8(win), y)
    eng.close()
    eng2 = I3DEngine(sd, "rgb", 0, max_stacks=2, max_T=16)
    two = torch.randint(0, 256, (2, 13, 256, 341, 3), dtype=torch.uint8, generator=g).to(cuda_device)
    assert not two[:, :12].is_contiguous()
    assert torch.equal(eng2.forward_frames_u8(two[:, :12]), eng2.forward_frames_u8(two[:, :12].contiguous()))
    # host entry (pipelined H2D): 5 stacks in groups of 2 == device entry
    five = torch.randint(0, 256, (5, 13, 256, 341, 3), dtype=torch.uint8, generator=g).pin_memory()
    yh = eng2.forward_frames_u8_host(five, 12, group=2)
    assert not yh.is_cuda and torch.equal(yh, eng2.forward_frames_u8(five.to(cuda_device)[:, :12]).cpu())
    eng2.close()
    # flow: values beyond +-20, exact +-20 and half-way quantisation points
    sdf = i3d_net.synthetic_state_dict("flow", 2)
    flow = torch.randn(1, 12, 2, 256, 344, generator=g) * 12
    flow[0, 0, 0, 20:30, 70:90] = 20.0
    flow[0, 1, 1, 40:50, 70:90] = -20.0
    flow[0, 2, 0, 60:70, 70:90] = (0.5 - 128) * 40 / 255      # 128 + 6.375 f lands on x.5
    engf = I3DEngine(sdf, "flow", 0, max_stacks=1, max_T=16)
    yf = engf.forward_flow(flow.to(cuda_device))
    xf = i3d_net.flow_transform(flow[0])
    reff = _oracle_gpu(sdf, xf, cuda_device)
    rel, mx = _rel(yf, reff)
    print(f"flow path: {rel:.3e} {mx:.3e}")
    assert rel < 1e-3 and mx < 1e-3
    assert torch.equal(yf, engf(xf.to(cuda_device)))
    engf.close()


def test_i3d_host_stacks_pipelined_calls(cuda_device):
    """forward_frames_u8_host: host stacks in groups (copy of group k+1 under the network of group k) and, with
    wait=False, two calls in flight -- same features as the device-resident call."""
    from oracle import i3d_net
    from video_features_b200.i3d_engine import I3DEngine
    sd = i3d_net.synthetic_state_dict("rgb", 3)
    eng = I3DEngine(sd, "rgb", 0, max_stacks=2, max_T=16)
    g = torch.Generator().manual_seed(4)
    a = torch.randint(0, 256, (5, 17, 224, 224, 3), dtype=torch.uint8, generator=g).pin_memory()
    b = torch.randint(0, 256, (3, 17, 224, 224, 3), dtype=torch.uint8, generator=g).pin_memory()
    ref_a = eng.forward_frames_u8(a.to(cuda_device)[:, :16]).cpu()
    ref_b = eng.forward_frames_u8(b.to(cuda_device)[:, :16]).cpu()
    assert torch.equal(eng.forward_frames_u8_host(a, 16, group=2), ref_a)
    ya, ea = eng.forward_frames_u8_host(a, 16, group=2, wait=False)
    yb, eb = eng.forward_frames_u8_host(b, 16, group=2, wait=False)
    ea.synchronize()
    eb.synchronize()
    assert torch.equal(ya, ref_a) and torch.equal(yb, ref_b)
    eng.close()
