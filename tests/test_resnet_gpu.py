"""ResNet engine and ExtractResNet on the B200 against the fp32 oracle (oracle/resnet_net.py, pinned to torchvision by
tests/test_resnet_cpu.py).  Bar, per output row: rel-L2 <= 1e-3 and max-abs <= 1e-3 * max |ref|."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import pil_resample, resnet_net
from video_features_b200 import synthetic_weights as sw

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
VIDEO = os.path.join(ROOT, "tests", "golden", "v_GGSY1Qvo990.mp4")


@pytest.fixture(autouse=True)
def _fp32_oracle():
    """The oracle runs on the GPU here: keep its convolutions in fp32."""
    c, m = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = c, m


def _oracle(sd, x, depth, stages=False):
    return resnet_net.forward_features({k: v.cuda() for k, v in sd.items()}, x.cuda(), depth, stages)


def _bar(y, ref):
    y, ref = y.double().cpu(), ref.double().cpu()
    rel = ((y - ref).norm(dim=1) / ref.norm(dim=1)).max().item()
    mx = ((y - ref).abs().amax(dim=1) / ref.abs().amax(dim=1)).max().item()
    assert rel <= 1e-3 and mx <= 1e-3, (rel, mx)
    return rel, mx


def _frames(n, h, w, seed):
    return np.random.default_rng([seed, h, w]).integers(0, 256, (n, h, w, 3), dtype=np.uint8)


def _resized(frames):
    h, w = frames.shape[1:3]
    oh, ow = resnet_net.resize_geometry(h, w)
    return np.stack([pil_resample.resize(f, oh, ow, pil_resample.BILINEAR) for f in frames])


_engines = {}


def _engine(depth, max_frames=64):
    from video_features_b200.resnet_engine import ResNetEngine
    key = (depth, max_frames)
    if key not in _engines:
        _engines[key] = (ResNetEngine(sw.resnet_state_dict(depth, 0), depth, 0, max_frames=max_frames),
                         sw.resnet_state_dict(depth, 0))
    return _engines[key]


@pytest.mark.parametrize("swap", [False, True])
def test_imagenet_normalize_bit_exact(swap):
    from video_features_b200.resnet_engine import normalize_u8
    rgb = _frames(3, 240, 320, 4)
    ref = resnet_net.transform_batch(rgb)
    r = _resized(rgb)
    src = r[..., ::-1].copy() if swap else r
    y = normalize_u8(torch.from_numpy(src).cuda(), swap_rb=swap).cpu()
    assert torch.equal(y, ref)


def test_stage_parity_depth50():
    """Stage outputs (stem + pool, layer1..4) against the oracle's intermediates.  These are fp16 tensors, and the error
    they carry grows through the blocks: 1.02e-3 rel-L2 at layer4 on a B200.  The pooled feature averages that error
    down to <= 4e-4, and the 1e-3 bar applies to the feature.  So the stage bar is 2e-3."""
    eng, sd = _engine(50)
    x = resnet_net.transform_batch(_frames(4, 240, 320, 6))
    eng(x.cuda())
    _, st = _oracle(sd, x, 50, stages=True)
    rels = []
    for s in range(5):
        y = eng.read_stage(s)
        assert y.shape == st[s].shape
        rels.append(float((y.double() - st[s].double()).norm() / st[s].double().norm()))
    print("stage rel-L2", ["%.2e" % r for r in rels])
    assert all(r <= 2e-3 for r in rels), rels


@pytest.mark.parametrize("depth", [18, 34, 50, 101, 152])
def test_features_meet_bar_every_depth(depth):
    eng, sd = _engine(depth)
    x = resnet_net.transform_batch(_frames(4, 240, 320, depth))
    y = eng(x.cuda())
    assert y.shape == (4, sw.resnet_feature_dim(depth))
    _bar(y, _oracle(sd, x, depth))


def test_resnet50_300_frames_geometries_and_chunks():
    """300 frames in three geometries (240x320, portrait, up-scaled from below 256) through the u8 entry; 64 frames per
    chunk, so calls of 120 / 100 / 80 frames run as balanced chunks with ragged sizes."""
    eng, sd = _engine(50, max_frames=64)
    for (h, w, n) in ((240, 320, 120), (320, 240, 100), (180, 200, 80)):
        rgb = _frames(n, h, w, 9)
        y = eng.forward_frames_u8(torch.from_numpy(rgb).cuda())
        _bar(y, _oracle(sd, resnet_net.transform_batch(rgb), 50))


def test_u8_entry_equals_f32_entry():
    eng, _ = _engine(50)
    rgb = _frames(5, 240, 320, 12)
    y8 = eng.forward_frames_u8(torch.from_numpy(rgb[..., ::-1].copy()).cuda(), swap_rb=True)
    y32 = eng(resnet_net.transform_batch(rgb).cuda())
    assert torch.equal(y8, y32)


def test_call_split_and_host_pipeline_bit_identical():
    eng, _ = _engine(50, max_frames=64)
    rgb = torch.from_numpy(_frames(270, 240, 320, 13))
    dev = rgb.cuda()
    whole = eng.forward_frames_u8(dev)
    for k in (1, 7, 256):
        parts = torch.cat([eng.forward_frames_u8(dev[a:a + k]) for a in range(0, min(270, 3 * k + 5), k)])
        assert torch.equal(parts, whole[:parts.shape[0]]), k
    host = eng.forward_frames_u8_host(rgb.pin_memory(), group=100)
    assert torch.equal(host, whole.cpu())


def _decoded_rgb():
    import cv2
    cap = cv2.VideoCapture(VIDEO)
    out = []
    while True:
        ok, bgr = cap.read()
        if not ok:
            break
        out.append(cv2.cvtColor(bgr, cv2.COLOR_BGR2RGB))
    cap.release()
    return np.stack(out)


def _run_main(out_dir, *extra, videos=(VIDEO,)):
    env = dict(os.environ, VF_RESNET_SYNTHETIC="0")
    cmd = [sys.executable, os.path.join(ROOT, "main.py"), "--feature_type", "resnet50", "--on_extraction", "save_numpy",
           "--output_path", str(out_dir), "--video_paths", *videos, *extra]
    return subprocess.run(cmd, env=env, cwd=ROOT, capture_output=True, text=True, timeout=900)


def test_main_resnet50_on_sample_video(tmp_path):
    broken = tmp_path / "broken.mp4"
    broken.write_bytes(b"not a video")
    r1 = _run_main(tmp_path / "b1", videos=(str(broken), VIDEO))
    assert r1.returncode == 0, r1.stderr[-2000:]
    assert "Extraction failed at" in r1.stdout and "broken.mp4" in r1.stdout
    f1 = tmp_path / "b1" / "resnet50" / "v_GGSY1Qvo990_resnet50.npy"
    a = np.load(f1)
    assert a.dtype == np.float64 and a.shape == (355, 2048)
    r128 = _run_main(tmp_path / "b128", "--batch_size", "128", "--gather_features", str(tmp_path / "g.npz"))
    assert r128.returncode == 0, r128.stderr[-2000:]
    b = np.load(tmp_path / "b128" / "resnet50" / "v_GGSY1Qvo990_resnet50.npy")
    assert np.array_equal(a, b)
    g = np.load(tmp_path / "g.npz")
    assert np.array_equal(g["features"], b.astype(g["features"].dtype)) and list(g["rows_per_video"]) == [355]
    rgb = _decoded_rgb()
    assert rgb.shape[0] == 355
    sd = sw.resnet_state_dict(50, 0)
    ref = torch.cat([_oracle(sd, resnet_net.transform_batch(rgb[i:i + 64]), 50).cpu() for i in range(0, 355, 64)])
    _bar(torch.from_numpy(a), ref)
