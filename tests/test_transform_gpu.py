"""Pillow-compatible resize kernel (vf_resize_u8) -- byte-exact against the committed Pillow / reference fixtures
and against the numpy oracle on fresh random images (integer arithmetic: the bar is bit-exact)."""
import os

import numpy as np
import pytest
import torch

import video_features_b200  # noqa: F401

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _resize(img: np.ndarray, oh: int, ow: int, filt: int) -> np.ndarray:
    t = torch.from_numpy(img)[None].cuda()
    return torch.ops.vfeat.resize_u8(t, oh, ow, filt)[0].cpu().numpy()


def test_resize_matches_pillow_fixture(cuda_device):
    from helpers import pillow_resize_cases
    cases = pillow_resize_cases()
    for n, (im, out, filt) in enumerate(cases):
        assert np.array_equal(_resize(im, out.shape[0], out.shape[1], filt), out), f"case {n}"
    assert len(cases) >= 6


def test_resize_matches_reference_i3d_chain_fixture(cuda_device):
    """ToPILImage -> ResizeImproved(256) -> PILToTensor of the reference (extract_i3d.py:55-60) == bilinear kernel."""
    from video_features_b200 import ops
    g = np.load(os.path.join(GOLD, "i3d_resize.npz"))
    for i in range(3):
        src, out = g[f"src{i}"], g[f"out{i}"]
        oh, ow = ops.resize_geometry(src.shape[0], src.shape[1], 256, True)
        assert (oh, ow) == out.shape[:2]
        assert np.array_equal(_resize(src, oh, ow, 2), out)


@pytest.mark.parametrize("h,w,oh,ow,filt", [(270, 480, 256, 455, 2), (240, 320, 224, 298, 3), (480, 270, 398, 224, 3),
                                             (64, 64, 224, 224, 3), (720, 1280, 224, 398, 3), (37, 53, 37, 20, 2)])
def test_resize_matches_numpy_oracle_batched(cuda_device, h, w, oh, ow, filt):
    from oracle import pil_resample
    rng = np.random.default_rng(h * w + oh)
    imgs = rng.integers(0, 256, (3, h, w, 3), dtype=np.uint8)
    got = torch.ops.vfeat.resize_u8(torch.from_numpy(imgs).cuda(), oh, ow, filt).cpu().numpy()
    for i in range(3):
        assert np.array_equal(got[i], pil_resample.resize(imgs[i], oh, ow, filt))


def test_clip_transform_on_sample_video_frames(cuda_device):
    """BASELINE config 1 frames (decoded by the reference's sampler, fixture): GPU resize + crop + normalise must be
    bit-identical to torchvision's CPU transform."""
    from oracle import clip_preprocess
    g = np.load(os.path.join(GOLD, "config1_sample_video.npz"))
    frames = torch.from_numpy(g["frames"]).cuda()                      # (2,240,320,3)
    resized = torch.ops.vfeat.resize_u8(frames, 224, 298, 3)
    assert np.array_equal(resized[:, :, 37:261].cpu().numpy(), g["resized_cropped"])
    got = torch.ops.vfeat.clip_normalize_u8(resized).cpu()
    ref = clip_preprocess.preprocess_batch(g["frames"])
    assert torch.equal(got, ref)
