"""ExtractI3D / ExtractRAFT (reference-facing classes) on a synthetic video, seeded stand-ins of the reference's
checkpoints (oracle/checkpoint_standins.py), against the oracle run on the same decoded frames."""
import argparse
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
import sys
sys.path.insert(0, os.path.join(ROOT, "scripts", "precision"))
from helpers import checkpoint  # noqa: E402


@pytest.fixture
def standin_checkpoints(monkeypatch):
    """The extractors load the checkpoint stand-ins instead of files from $VF_CKPT_DIR / checkpoints/."""
    from video_features_b200.extract import extract_i3d
    monkeypatch.setattr(extract_i3d, "_STATE_DICTS", {k: checkpoint(n) for k, n in extract_i3d._CKPT.items()})


def _write_video(path, n, h=120, w=160, fps=25.0, shift=(0.8, 0.5)):
    import cv2
    from oracle import raft_net
    fr = raft_net.synthetic_frames(n, h, w, seed=11, shift=shift).permute(0, 2, 3, 1).numpy().astype(np.uint8)
    vw = cv2.VideoWriter(path, cv2.VideoWriter_fourcc(*"mp4v"), fps, (w, h))
    assert vw.isOpened()
    for f in fr:
        vw.write(f)
    vw.release()


def _ns(**kw):
    d = dict(feature_type='i3d', video_paths=None, flow_paths=None, file_with_video_paths=None, video_dir=None, flow_dir=None,
             extraction_fps=None, extract_method=None, on_extraction='save_numpy', output_path='./output',
             output_direct=False, tmp_path='./tmp', streams=None, flow_type='raft', stack_size=None, step_size=None,
             show_pred=False, keep_tmp_files=False, batch_size=1, resize_to_smaller_edge=True, side_size=None)
    d.update(kw)
    return argparse.Namespace(**d)


@pytest.mark.parametrize("clip,shift", [("low_motion", (0.8, 0.5)), ("high_motion", (4.5, -3.0))])
def test_extract_i3d_two_streams_vs_oracle(cuda_device, standin_checkpoints, tmp_path, clip, shift):
    from PIL import Image
    from flow_quantiser_sensitivity import feature_sensitivity            # scripts/precision/
    from oracle import i3d_net, raft_net
    from video_features_b200 import utils
    from video_features_b200.extract.extract_i3d import ExtractI3D
    from video_features_b200.raft_engine import RAFTEngine
    vid = str(tmp_path / "clip.mp4")
    _write_video(vid, 20, shift=shift)
    out = str(tmp_path / "out")
    ex = ExtractI3D(_ns(video_paths=[vid], output_path=out, tmp_path=str(tmp_path / "tmp"), stack_size=12, step_size=12),
                    external_call=True)
    res = ex(torch.zeros([1], dtype=torch.long, device=cuda_device))[0]
    assert set(res) == {'rgb', 'flow', 'fps', 'timestamps_ms'}
    # a 20-frame video is shorter than 65 frames: the reference resamples it to 65 (extract_i3d.py:250-255), so with
    # stack_size = step_size = 12 there are (65-1)//12 = 5 stacks
    assert res['rgb'].shape == (5, 1024) and res['flow'].shape == (5, 1024) and res['rgb'].dtype == np.float64
    res = {k: (v[:1] if k in ('rgb', 'flow') else v) for k, v in res.items()}       # compare the first stack
    # oracle on the same decoded frames: PIL bilinear resize to 256 -> rgb / RAFT+flow transforms -> I3D
    rd = utils.VideoReader(vid)
    ix = np.linspace(1, rd.frame_cnt - 1, 65).astype(int)[:13]
    frames = [rd.get_frame(int(i)) for i in ix]
    rs = torch.stack([torch.from_numpy(np.asarray(Image.fromarray(f).resize((341, 256), Image.BILINEAR)).copy())
                      for f in frames]).permute(0, 3, 1, 2).float().to(cuda_device)
    sd_rgb = {k: v.to(cuda_device) for k, v in checkpoint("i3d_rgb.pt").items()}
    ref_rgb = i3d_net.forward_features(sd_rgb, i3d_net.rgb_transform(rs[:-1]))
    rel = float((torch.from_numpy(res['rgb']).to(cuda_device) - ref_rgb).norm() / ref_rgb.norm())
    print(f"[{clip}] ExtractI3D rgb vs oracle:", rel)
    assert rel < 1e-3
    sd_raft_cpu = checkpoint("raft-sintel.pth")
    sd_raft = {k: v.to(cuda_device) for k, v in sd_raft_cpu.items()}
    xp = raft_net.pad(rs)
    flow = raft_net.forward(sd_raft, xp[:-1], xp[1:], 20)                # padded, never unpadded (extract_i3d.py:172)
    sd_flow = {k: v.to(cuda_device) for k, v in checkpoint("i3d_flow.pt").items()}
    ref_flow = i3d_net.forward_features(sd_flow, i3d_net.flow_transform(flow))
    rel = float((torch.from_numpy(res['flow']).to(cuda_device) - ref_flow).norm() / ref_flow.norm())
    # The flow stream passes through the reference's 8-bit quantiser `round(128 + 255/40 f)` (transforms.py:43-51), a
    # staircase: a flow perturbation of 1e-5 px already moves the oracle's OWN feature by 3e-3 .. 4e-3 on these clips, and
    # the fp32 oracle with a different thread count differs from itself by more than that
    # (scripts/precision/flow_quantiser_sensitivity.py -> profiles/r2_flow_sensitivity.json).  No implementation whose
    # flow differs from the oracle's at all can therefore be held to 1e-3 on the composite.  The bar is derived, not
    # guessed: (1) the engine's flow must meet the 1e-3 RAFT bar on this very clip, (2) quantiser + I3D on identical flow
    # is asserted elsewhere (test_i3d_gpu.py, 2e-4), and (3) the composite may not exceed 2x the oracle's own
    # sensitivity to Gaussian flow noise of the SAME rms as the engine's measured flow error.
    eng = RAFTEngine(sd_raft_cpu, 0, max_frames=13, max_h=256, max_w=341)
    eflow = eng.flow(rs.permute(0, 2, 3, 1).contiguous().to(torch.uint8), iters=20, unpad=False)
    eng.close()
    d = eflow - flow
    flow_rel, flow_rms = float(d.norm() / flow.norm()), float(d.pow(2).mean().sqrt())
    flow_max = float(d.abs().max()) / float(flow.abs().max())
    # rel-L2 at the RAFT bar; the max-abs half is asserted on the RAFT tests proper (test_raft_gpu.py, ExtractRAFT below).
    # Here every third "pair" is the SAME decoded frame twice (a 20-frame video resampled to 65 indices): RAFT on identical
    # frames is a badly conditioned iteration and single pixels move by a few 1e-3 px (measured 3.2e-3 of max |flow|).
    assert flow_rel <= 1e-3 and flow_max <= 5e-3, (flow_rel, flow_max)
    sens = feature_sensitivity(sd_flow, flow, [flow_rms], draws=5)[flow_rms]["feature_rel"]
    bar = max(1e-3, 2.0 * sens)
    print(f"[{clip}] ExtractI3D flow (RAFT -> quantiser -> I3D) vs oracle: {rel:.3e}; engine flow error {flow_rel:.2e} rel (max {flow_max:.2e}) / "
          f"{flow_rms:.2e} px rms; oracle's own sensitivity at that rms: {sens:.3e}; bar {bar:.3e}")
    assert rel <= bar, (rel, bar)


def test_extract_i3d_mixed_aspect_ratios_and_precomputed_flow(cuda_device, standin_checkpoints, tmp_path):
    """(a) a list whose second video is wider than the first: the RAFT engine's workspace must follow (the reference
    handles any resolution per video); (b) --flow_type flow: pre-computed flow_x / flow_y jpg pairs
    (extract_i3d.py:195-229,266-278) against the oracle fed with the very same jpgs."""
    import cv2
    from oracle import i3d_net
    from video_features_b200.extract.extract_i3d import ExtractI3D
    a, b = str(tmp_path / "narrow.mp4"), str(tmp_path / "wide.mp4")
    _write_video(a, 14, h=120, w=160)                     # -> 256x341
    _write_video(b, 14, h=96, w=192)                      # -> 256x512: wider than the engine created for `a`
    ex = ExtractI3D(_ns(video_paths=[a, b], output_path=str(tmp_path / "o"), tmp_path=str(tmp_path / "t"), stack_size=10,
                        step_size=10, streams=['flow']), external_call=True)
    res = ex(torch.arange(2, device=cuda_device))
    assert len(res) == 2 and res[0]['flow'].shape == (6, 1024) and res[1]['flow'].shape == (6, 1024)
    assert np.isfinite(res[1]['flow']).all() and np.abs(res[1]['flow']).max() > 0

    # ---- pre-computed flow images
    fdir = tmp_path / "flows" / "narrow"
    fdir.mkdir(parents=True)
    rng = np.random.default_rng(5)
    base = cv2.GaussianBlur(rng.integers(0, 256, (256, 344), dtype=np.uint8), (0, 0), 6)
    for i in range(14):
        cv2.imwrite(str(fdir / f"flow_x_{i:05d}.jpg"), np.roll(base, 2 * i, axis=1))
        cv2.imwrite(str(fdir / f"flow_y_{i:05d}.jpg"), np.roll(base, 3 * i, axis=0))
    exf = ExtractI3D(_ns(video_paths=[a], flow_paths=[str(fdir)], output_path=str(tmp_path / "o"),
                         tmp_path=str(tmp_path / "t"), stack_size=12, step_size=12, flow_type='flow'), external_call=True)
    assert exf.path_list == [(a, str(fdir))]
    got = exf(torch.zeros([1], dtype=torch.long, device=cuda_device))[0]
    # 14 frames < 65: resampled to 65 indices; zip(frames, flows) stops at the 14 flow pairs -> one stack of 12
    assert got['flow'].shape == (1, 1024) and got['rgb'].shape == (1, 1024)
    imgs = torch.stack([torch.stack([torch.from_numpy(cv2.imread(str(fdir / f"flow_{c}_{i:05d}.jpg"), cv2.IMREAD_GRAYSCALE))
                                     for c in "xy"]) for i in range(12)])            # uint8 (12,2,256,344), as mmcv.imread
    sd_flow = {k: v.to(cuda_device) for k, v in checkpoint("i3d_flow.pt").items()}
    # the reference applies its flow transform to these uint8 grey levels as they are: clamp(-20,20) keeps [0,20]
    ref = i3d_net.forward_features(sd_flow, i3d_net.flow_transform(imgs.float().to(cuda_device)))
    rel = float((torch.from_numpy(got['flow']).to(cuda_device) - ref).norm() / ref.norm())
    print("ExtractI3D --flow_type flow vs oracle:", rel)
    assert rel < 1e-3


def test_extract_raft_writes_flow(cuda_device, standin_checkpoints, tmp_path):
    from oracle import raft_net
    from video_features_b200.extract.extract_raft import ExtractRAFT
    vid = str(tmp_path / "clip2.mp4")
    _write_video(vid, 6, h=128, w=160)
    out = str(tmp_path / "out")
    ex = ExtractRAFT(_ns(feature_type='raft', video_paths=[vid], output_path=out, tmp_path=str(tmp_path / "tmp"), batch_size=2))
    assert ex(torch.zeros([1], dtype=torch.long, device=cuda_device)) is None
    flow = np.load(os.path.join(out, "raft", "clip2_raft.npy"))
    assert flow.shape == (5, 2, 128, 160) and flow.dtype == np.float64
    import cv2
    cap = cv2.VideoCapture(vid)
    fr = []
    while True:
        ok, f = cap.read()
        if not ok:
            break
        fr.append(cv2.cvtColor(f, cv2.COLOR_BGR2RGB))
    x = torch.from_numpy(np.stack(fr)).permute(0, 3, 1, 2).float().to(cuda_device)
    sd = {k: v.to(cuda_device) for k, v in checkpoint("raft-sintel.pth").items()}
    ref = raft_net.forward(sd, x[:-1], x[1:], 20).cpu().numpy()
    rel = np.linalg.norm(flow - ref) / np.linalg.norm(ref)
    print("ExtractRAFT vs oracle:", rel)
    # Decoded (block-compressed) 128x160 frames are the hard case for reduced-precision RAFT: rounding only the conv
    # INPUTS to fp16 gives 7.6e-3 here in a CPU emulation, fp16 weights alone 6e-4 with a 4.6e-3 max-abs outlier.  With
    # every operand carried as a split-fp16 pair the engine measures 5.7e-5 (the fp32 oracle's own thread-count noise
    # on these frames is 2.5e-5).
    assert rel < 5e-4
