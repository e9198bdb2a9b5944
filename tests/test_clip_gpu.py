"""CLIP ViT-B/32 tower through the C ABI against the fp32 oracle (oracle/clip_tower.py), same seeded frames.

Tolerance (BASELINE.json north_star): 1e-3 relative vs the fp32 torch path --
per row  ||y - y_ref||_2 / ||y_ref||_2 <= 1e-3  and  max|y - y_ref| <= 1e-3 * max|y_ref|.
CLIP caveat: synthetic weights, restated oracle (the reference's `clip` package and weights are absent offline).
"""
import numpy as np
import pytest
import torch

import video_features_b200  # noqa: F401  (registers torch.ops.vfeat)

pytestmark = pytest.mark.gpu

MEAN = torch.tensor([0.48145466, 0.4578275, 0.40821073])
STD = torch.tensor([0.26862954, 0.26130258, 0.27577711])


def _transform_224(frames_u8: torch.Tensor) -> torch.Tensor:
    """ToTensor + Normalize on 224x224 frames (Resize/CenterCrop are identities at this size)."""
    x = frames_u8.permute(0, 3, 1, 2).to(torch.float32).div(255)
    return x.sub(MEAN[None, :, None, None]).div(STD[None, :, None, None])


@pytest.fixture(scope="module")
def tower(cuda_device):
    from oracle import clip_tower
    from video_features_b200.clip_engine import ClipEngine
    sd = clip_tower.synthetic_state_dict(0)
    eng = ClipEngine(sd, device=0)
    yield sd, eng
    eng.close()


def _check_rows(y, ref, tol=1e-3):
    y, ref = y.double().cpu(), ref.double().cpu()
    rel = ((y - ref).norm(dim=1) / ref.norm(dim=1)).max().item()
    mx = ((y - ref).abs().amax(dim=1) / ref.abs().amax(dim=1)).max().item()
    assert rel <= tol, f"row rel-L2 {rel:.3e} > {tol}"
    assert mx <= tol, f"row max-abs {mx:.3e} > {tol}"
    return rel, mx


def test_transform_is_bit_exact(cuda_device):
    g = torch.Generator().manual_seed(3)
    frames = torch.randint(0, 256, (5, 224, 224, 3), dtype=torch.uint8, generator=g)
    got = torch.ops.vfeat.clip_normalize_u8(frames.to(cuda_device)).cpu()
    assert torch.equal(got, _transform_224(frames))


def test_encode_small_batch_vs_cpu_oracle(tower, cuda_device):
    from oracle import clip_tower
    sd, eng = tower
    g = torch.Generator().manual_seed(0)
    frames = torch.randint(0, 256, (8, 224, 224, 3), dtype=torch.uint8, generator=g)
    ref = clip_tower.encode_image(sd, _transform_224(frames))            # fp32 on CPU
    y_u8 = eng.encode_frames_u8(frames.to(cuda_device))
    y_f32 = eng.encode_image(_transform_224(frames).to(cuda_device))
    y_host = eng.encode_frames_u8_host(frames)
    torch.cuda.synchronize()
    print("u8 path:", _check_rows(y_u8, ref))
    _check_rows(y_f32, ref)
    assert torch.equal(y_u8.cpu(), y_f32.cpu()), "uint8 and fp32 entry points must agree bit-for-bit"
    assert torch.equal(y_u8.cpu(), y_host), "host-buffer entry point must agree bit-for-bit"


def test_encode_multi_chunk_vs_gpu_fp32_oracle(tower, cuda_device):
    """270 frames = 2 full chunks of 120 + a ragged tail of 30; oracle runs in fp32 (TF32 off) on the GPU."""
    from oracle import clip_tower
    sd, eng = tower
    g = torch.Generator().manual_seed(1)
    frames = torch.randint(0, 256, (270, 224, 224, 3), dtype=torch.uint8, generator=g)
    sd_gpu = {k: v.to(cuda_device) for k, v in sd.items()}
    ref = torch.cat([clip_tower.encode_image(sd_gpu, _transform_224(frames[i:i + 54]).to(cuda_device))
                     for i in range(0, 270, 54)])
    y = eng.encode_frames_u8(frames.to(cuda_device))
    y_host = eng.encode_frames_u8_host(frames)
    print("multi-chunk:", _check_rows(y, ref))
    assert torch.equal(y.cpu(), y_host)
    # batch-composition independence: a frame's features do not depend on its neighbours
    y1 = eng.encode_frames_u8(frames[100:101].to(cuda_device))
    assert torch.equal(y1.cpu(), y[100:101].cpu())


def test_encode_with_outlier_channel_weights(cuda_device):
    """Trained ViT-B/32 weights have what random ones lack: residual-stream channels of magnitude 50-200, heavy-tailed
    LayerNorm gains, loud projection rows (synthetic_weights.clip_vit_b32_state_dict(outliers=True)).  The engine stores
    QKV / attention / MLP activations in fp16: this is the regime that would break it.  Same 1e-3 / 1e-3 bar."""
    from oracle import clip_tower
    from video_features_b200 import synthetic_weights
    from video_features_b200.clip_engine import ClipEngine
    sd = synthetic_weights.clip_vit_b32_state_dict(5, outliers=True)
    g = torch.Generator().manual_seed(4)
    frames = torch.randint(0, 256, (24, 224, 224, 3), dtype=torch.uint8, generator=g)
    frames[12:] = frames[12:] // 4 + 96                                    # half of them low-contrast
    sd_gpu = {k: v.to(cuda_device) for k, v in sd.items()}
    ref, hidden = clip_tower.encode_image(sd_gpu, _transform_224(frames).to(cuda_device), return_hidden=True)
    peak = max(float(h.abs().max()) for h in hidden)
    assert peak > 50.0, f"the outlier regime was not reached (residual peak {peak:.1f})"
    eng = ClipEngine(sd, device=0)
    try:
        y = eng.encode_frames_u8(frames.to(cuda_device))
        print(f"outlier weights: residual peak {peak:.1f};", _check_rows(y, ref))
    finally:
        eng.close()


@pytest.mark.parametrize("n_frames", [1, 4, 5, 7, 23, 250])
def test_fused_qkv_attention_vs_fp32_reference_and_split_path(tower, cuda_device, n_frames):
    """The QKV-projection + attention kernel (one tile = 5 frames x 1 head on a CTA pair, the third frame straddling the
    pair through distributed shared memory) against nn.MultiheadAttention's math in fp32, and against the split path (QKV
    GEMM + stand-alone attention kernel).  Frame counts: single frame, below / at / above one 5-frame group, a ragged
    last group, a full chunk."""
    sd, eng = tower
    g = torch.Generator().manual_seed(40 + n_frames)
    x = torch.randn(n_frames * 50, 768, generator=g).half().to(cuda_device)
    layer = 3
    p = f"visual.transformer.resblocks.{layer}."
    w, b = sd[p + "attn.in_proj_weight"].to(cuda_device), sd[p + "attn.in_proj_bias"].to(cuda_device)
    qkv = x.float() @ w.half().float().t() + b                     # fp16 operands, fp32 accumulate, like the engine
    q, k, v = (t.half().float().view(n_frames, 50, 12, 64).transpose(1, 2) for t in qkv.split(768, dim=1))
    att = torch.softmax(q @ k.transpose(-1, -2) * 0.125, dim=-1)
    ref = (att @ v).transpose(1, 2).reshape(n_frames * 50, 768)
    fused = eng.block_attention(layer, x, fused=True)
    split = eng.block_attention(layer, x, fused=False)
    torch.cuda.synchronize()
    for name, y in (("fused", fused), ("split", split)):
        err = float((y.float() - ref).norm() / ref.norm())
        mx = float((y.float() - ref).abs().max() / ref.abs().max())
        print(f"{name} attention, {n_frames} frames: rel-L2 {err:.2e}, max-abs {mx:.2e}")
        assert err < 1e-3 and mx < 2e-3, (name, err, mx)
    # same arithmetic in both paths: identical up to the fp16 rounding of q, k, v (bit-identical in practice)
    d = float((fused.float() - split.float()).abs().max())
    print(f"fused vs split: max |diff| {d:.3e}, identical: {torch.equal(fused, split)}")
    assert d <= 2e-3 * float(ref.abs().max())


def test_encode_empty_and_single(tower, cuda_device):
    sd, eng = tower
    out = eng.encode_frames_u8(torch.empty((0, 224, 224, 3), dtype=torch.uint8, device=cuda_device))
    assert out.shape == (0, 512)


def test_resize_path_matches_pillow_then_oracle(tower, cuda_device):
    """240x320 frames: Resize(224, bicubic) -> CenterCrop -> normalise, Pillow/torchvision semantics."""
    from PIL import Image
    from oracle import clip_tower
    sd, eng = tower
    g = torch.Generator().manual_seed(2)
    frames = torch.randint(0, 256, (3, 240, 320, 3), dtype=torch.uint8, generator=g)
    tens = []
    for f in frames.numpy():
        im = Image.fromarray(f).resize((298, 224), Image.BICUBIC)
        a = torch.from_numpy(np.asarray(im).copy())[:, 37:37 + 224, :]
        tens.append(a)
    ref = clip_tower.encode_image(sd, _transform_224(torch.stack(tens)))
    y = eng.encode_frames_u8(frames.to(cuda_device))
    _check_rows(y, ref)


def test_async_host_calls_match_the_synchronous_call(tower, cuda_device):
    """vf_clip_encode_u8_host_async: six calls of different sizes / geometries enqueued back to back (more than the four
    tickets the handle keeps), waited for out of order and from another thread -- bit-identical to the synchronous call."""
    import threading
    sd, eng = tower
    g = torch.Generator().manual_seed(11)
    shapes = [(300, 224, 224), (7, 240, 320), (513, 224, 224), (1, 224, 224), (64, 120, 160), (256, 224, 224)]
    frames = [torch.randint(0, 256, (n, h, w, 3), dtype=torch.uint8, generator=g).pin_memory() for n, h, w in shapes]
    ref = [eng.encode_frames_u8_host(f).clone() for f in frames]
    outs = [torch.empty((f.shape[0], 512), dtype=torch.float32).pin_memory() for f in frames]
    tickets = []
    devs = []
    for f, o in zip(frames, outs):
        t, d = eng.encode_frames_u8_host_async(f, o, out_dev=True)
        tickets.append(t)
        devs.append(d)
    assert tickets == list(range(tickets[0], tickets[0] + 6))
    th = threading.Thread(target=lambda: [eng.wait(t) for t in reversed(tickets)])
    th.start()
    th.join()
    eng.wait(-1)
    for o, d, r in zip(outs, devs, ref):
        assert torch.equal(o, r)
        assert torch.equal(d.cpu(), r)
    with pytest.raises(RuntimeError):
        eng.wait(tickets[-1] + 1)            # never issued


# ---------------------------------------------------------------- ViT-B/16 (the reference's 'CLIP-ViT-B/16' feature type)
@pytest.fixture(scope="module")
def tower16(cuda_device):
    from oracle import clip_tower
    from video_features_b200.clip_engine import ClipEngine
    sd = clip_tower.synthetic_state_dict(1, patch=16)
    eng = ClipEngine(sd, device=0)
    assert eng.patch == 16 and eng.tokens == 197
    yield sd, eng
    eng.close()


def test_b16_encode_small_batch_vs_cpu_oracle(tower16, cuda_device):
    from oracle import clip_tower
    sd, eng = tower16
    g = torch.Generator().manual_seed(2)
    frames = torch.randint(0, 256, (5, 224, 224, 3), dtype=torch.uint8, generator=g)
    ref = clip_tower.encode_image(sd, _transform_224(frames))            # fp32 on CPU
    y_u8 = eng.encode_frames_u8(frames.to(cuda_device))
    y_f32 = eng.encode_image(_transform_224(frames).to(cuda_device))
    y_host = eng.encode_frames_u8_host(frames)
    torch.cuda.synchronize()
    _check_rows(y_u8, ref)
    _check_rows(y_f32, ref)
    assert torch.equal(y_u8.cpu(), y_f32.cpu()) and torch.equal(y_u8.cpu(), y_host)


def test_b16_multi_chunk_vs_gpu_fp32_oracle(tower16, cuda_device):
    """More frames than one chunk (63) and a ragged tail; the fp32 oracle runs on the GPU with TF32 off."""
    from oracle import clip_tower
    sd, eng = tower16
    g = torch.Generator().manual_seed(7)
    frames = torch.randint(0, 256, (150, 224, 224, 3), dtype=torch.uint8, generator=g)
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    sd_dev = {k: v.to(cuda_device) for k, v in sd.items()}
    ref = torch.cat([clip_tower.encode_image(sd_dev, _transform_224(frames[i:i + 50]).to(cuda_device))
                     for i in range(0, 150, 50)])
    y = eng.encode_frames_u8(frames.to(cuda_device))
    torch.cuda.synchronize()
    _check_rows(y, ref)


def test_b16_attention_vs_fp32_reference(tower16, cuda_device):
    """QKV GEMM + the 197-token attention kernel of block 0 against an fp32 computation on the same fp16 input."""
    sd, eng = tower16
    g = torch.Generator(device="cpu").manual_seed(5)
    x = (torch.randn(3 * 197, 768, generator=g) * 0.8).to(torch.float16)
    got = eng.block_attention(0, x.to(cuda_device), fused=False).float().cpu()
    w = sd["visual.transformer.resblocks.0.attn.in_proj_weight"].to(torch.float16).float()
    b = sd["visual.transformer.resblocks.0.attn.in_proj_bias"].float()
    qkv = (x.float() @ w.t() + b).to(torch.float16).float().view(3, 197, 3, 12, 64)
    q, k, v = (qkv[:, :, i].transpose(1, 2) for i in range(3))
    att = torch.softmax((q * 0.125) @ k.transpose(-1, -2), dim=-1) @ v
    ref = att.transpose(1, 2).reshape(3 * 197, 768)
    err = (got - ref).abs().max().item()
    assert err <= 2e-3 * ref.abs().max().item(), err


def test_b16_feature_type_through_extractor(cuda_device, tmp_path, monkeypatch):
    """'CLIP-ViT-B/16' runs through ExtractCLIP (synthetic weights of that geometry) on the sample video and agrees
    with the oracle on the same decoded frames."""
    import argparse
    import os
    from oracle import clip_preprocess, clip_tower
    from video_features_b200 import synthetic_weights, utils
    from video_features_b200.extract.extract_clip import ExtractCLIP
    monkeypatch.setenv("VF_CLIP_SYNTHETIC", "9")
    video = os.path.join(os.path.dirname(__file__), "golden", "v_GGSY1Qvo990.mp4")
    out = str(tmp_path / "out")
    args = argparse.Namespace(feature_type='CLIP-ViT-B/16', video_paths=[video], flow_paths=None,
                              file_with_video_paths=None, video_dir=None, flow_dir=None, extraction_fps=None,
                              extract_method="uni_5", on_extraction='save_numpy', output_path=out, output_direct=True,
                              tmp_path=os.path.join(out, 'tmp'))
    ex = ExtractCLIP(args, external_call=True)
    d = ex(torch.zeros([1], dtype=torch.long, device=cuda_device))[0]
    feats = d['CLIP-ViT-B/16']
    assert feats.shape == (5, 512)
    frames, _, _ = utils.extract_frames(video, "uni_5")
    sd = synthetic_weights.clip_vit_b32_state_dict(9, patch=16)
    ref = clip_tower.encode_image(sd, clip_preprocess.preprocess_batch(frames))
    _check_rows(torch.from_numpy(np.asarray(feats)), ref)


def test_bench_dump_outputs_are_the_headline_features(cuda_device, tmp_path):
    """bench.py --dump-outputs: the (1000, 512) features of the last timed step, on the seeded frames of rank 0."""
    import os
    import subprocess
    import sys
    from oracle import clip_tower
    from video_features_b200 import synthetic_weights
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    p = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--steps", "2", "--warmup", "3", "--no-cpu",
                        "--no-secondary", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=900)
    assert p.returncode == 0, p.stderr[-2000:]
    y = np.load(tmp_path / "features.npy")
    assert y.dtype == np.float32 and y.shape == (1000, 512)
    frames = torch.randint(0, 256, (1000, 224, 224, 3), dtype=torch.uint8, generator=torch.Generator().manual_seed(100))
    sd = synthetic_weights.clip_vit_b32_state_dict(0)
    rows = [0, 1, 499, 998, 999]
    ref = clip_tower.encode_image(sd, _transform_224(frames[rows]))
    _check_rows(torch.from_numpy(y[rows]), ref)
