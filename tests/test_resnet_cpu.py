"""ResNet extractor, CPU side: the oracle against torchvision (tests/golden/resnet_outputs.npz, made by
scripts/make_golden.py resnet), the transform restatement, the checkpoint loader, the synthetic weights' scale, and the
CLI routing."""
import hashlib
import os
import types

import numpy as np
import pytest
import torch

from oracle import resnet_net
from video_features_b200 import synthetic_weights as sw

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden", "resnet_outputs.npz")
VIDEO = os.path.join(ROOT, "tests", "golden", "v_GGSY1Qvo990.mp4")
DEPTHS = (18, 34, 50, 101, 152)
GEOMETRIES = ((240, 320), (320, 240), (180, 200))     # seeds and geometries as in scripts/make_golden.py


def _frame(h, w, seed=21):
    return np.random.default_rng([seed, h, w]).integers(0, 256, (h, w, 3), dtype=np.uint8)


@pytest.mark.parametrize("depth", DEPTHS)
def test_oracle_matches_torchvision_fixture(depth):
    g = np.load(GOLD)
    x = torch.randn(2, 3, 224, 224, generator=torch.Generator().manual_seed(5))
    y = resnet_net.forward_features(sw.resnet_state_dict(depth, 0), x, depth).double()
    ref = torch.from_numpy(g[f"resnet{depth}"]).double()
    assert y.shape == (2, sw.resnet_feature_dim(depth))
    assert float((y - ref).norm() / ref.norm()) <= 1e-6


@pytest.mark.parametrize("hw", GEOMETRIES)
def test_transform_bit_exact_with_torchvision_fixture(hw):
    g = np.load(GOLD)
    y = resnet_net.transform(_frame(*hw)).numpy()
    assert y.dtype == np.float32 and y.shape == (3, 224, 224)
    assert hashlib.sha256(np.ascontiguousarray(y).tobytes()).hexdigest() == str(g[f"transform_{hw[0]}x{hw[1]}_sha256"])


def test_transform_bit_exact_on_sample_video_frames():
    cv2 = pytest.importorskip("cv2")
    T = pytest.importorskip("torchvision.transforms")
    tf = T.Compose([T.ToPILImage(), T.Resize(256), T.CenterCrop(224), T.ToTensor(),
                    T.Normalize(mean=[0.485, 0.456, 0.406], std=[0.229, 0.224, 0.225])])
    cap = cv2.VideoCapture(VIDEO)
    frames = []
    while len(frames) < 120:
        ok, bgr = cap.read()
        if not ok:
            break
        frames.append(cv2.cvtColor(bgr, cv2.COLOR_BGR2RGB))
    cap.release()
    for f in frames[::40]:
        assert torch.equal(resnet_net.transform(f), tf(f))


@pytest.mark.parametrize("depth", DEPTHS)
def test_synthetic_weights_stage_rms_in_band(depth):
    """Seeded weights keep every stage's activation RMS within [1, 10] -- neither exploding nor vanishing through up
    to 50 blocks -- so the parity tests run on well-scaled activations (measured: 2.2 .. 7.8, highest at depth 152)."""
    x = resnet_net.transform_batch(np.stack([_frame(240, 320, s) for s in (1, 2)]))
    _, st = resnet_net.forward_features(sw.resnet_state_dict(depth, 0), x, depth, return_stages=True)
    rms = [float(s.pow(2).mean().sqrt()) for s in st]
    assert all(1.0 <= r <= 10.0 for r in rms), rms


def test_checkpoint_loader_round_trip_and_missing_key(tmp_path, monkeypatch):
    from video_features_b200.extract import extract_resnet
    sd = sw.resnet_state_dict(18, 3)
    hub = tmp_path / "hub"
    (hub / "checkpoints").mkdir(parents=True)
    torch.save(sd, hub / "checkpoints" / "resnet18-f37072fd.pth")       # the file name pretrained=True caches
    monkeypatch.delenv("VF_RESNET_SYNTHETIC", raising=False)
    monkeypatch.delenv("VF_RESNET_CKPT", raising=False)
    monkeypatch.setattr(torch.hub, "get_dir", lambda: str(hub))
    got = extract_resnet.load_resnet_state_dict("resnet18")
    want = {k: v for k, v in sd.items() if not (k.startswith("fc.") or k.endswith("num_batches_tracked"))}
    assert set(got) == set(want)
    assert all(torch.equal(got[k], want[k]) for k in want)
    broken = dict(sd)
    del broken["layer3.1.bn2.running_var"]
    torch.save(broken, tmp_path / "broken.pth")
    monkeypatch.setenv("VF_RESNET_CKPT", str(tmp_path / "broken.pth"))
    with pytest.raises(KeyError, match="layer3.1.bn2.running_var"):
        extract_resnet.load_resnet_state_dict("resnet18")
    monkeypatch.setenv("VF_RESNET_CKPT", str(tmp_path / "absent.pth"))
    monkeypatch.setattr(torch.hub, "get_dir", lambda: str(tmp_path / "nowhere"))
    with pytest.raises(FileNotFoundError, match="absent.pth"):
        extract_resnet.load_resnet_state_dict("resnet18")


def _args(**kw):
    import main
    a = main.make_parser().parse_args(["--feature_type", kw.pop("feature_type"), "--video_paths", VIDEO])
    for k, v in kw.items():
        setattr(a, k, v)
    return a


@pytest.mark.parametrize("ft", ["resnet18", "resnet34", "resnet50", "resnet101", "resnet152"])
def test_main_routes_resnet_types(ft):
    import main
    from video_features_b200.extract.extract_resnet import ExtractResNet
    ex = main.build_extractor(_args(feature_type=ft))
    assert isinstance(ex, ExtractResNet)
    assert ex.feature_type == ft and ex.output_path.endswith(ft) and ex.batch_size == 1


def test_main_refuses_extraction_fps():
    import main
    with pytest.raises(NotImplementedError, match="extraction_fps"):
        main.build_extractor(_args(feature_type="resnet50", extraction_fps=5.0))
