"""Generates tests/golden/*.npz by running the REFERENCE's own python (imported from /root/reference, never
copied) and the third-party libraries it relies on (Pillow) in the build container.  /root/reference does not
exist on the GPU box, so tests read only the committed fixtures.

    python scripts/make_golden.py            # needs /root/reference
"""
import os
import sys
import types

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = "/root/reference"
OUT = os.path.join(ROOT, "tests", "golden")
sys.path.insert(0, ROOT)


def install_mmcv_shim():
    """mmcv is un-vendored and absent: the reference only uses VideoReader(.fps,.frame_cnt,.get_frame) and imread.
    The shim decodes with cv2 exactly as mmcv does (seek with CAP_PROP_POS_FRAMES, frames are BGR), or -- for
    paths of the form 'synthetic:<frame_cnt>:<fps>' -- fabricates a video whose frame i is the integer i."""
    import cv2

    class VideoReader:
        def __init__(self, path):
            self._synthetic = str(path).startswith("synthetic:")
            if self._synthetic:
                _, cnt, fps = str(path).split(":")
                self.frame_cnt, self.fps = int(cnt), float(fps)
            else:
                self._cap = cv2.VideoCapture(str(path))
                self.fps = self._cap.get(cv2.CAP_PROP_FPS)
                self.frame_cnt = int(self._cap.get(cv2.CAP_PROP_FRAME_COUNT))

        def get_frame(self, i):
            if self._synthetic:
                return int(i)
            self._cap.set(cv2.CAP_PROP_POS_FRAMES, int(i))
            ok, frame = self._cap.read()
            return frame if ok else None

    m = types.ModuleType("mmcv")
    m.VideoReader = VideoReader
    m.imread = lambda p, flag="color": cv2.imread(p, cv2.IMREAD_GRAYSCALE if flag == "grayscale" else cv2.IMREAD_COLOR)
    sys.modules["mmcv"] = m


def main():
    assert os.path.isdir(REF), "needs the reference checkout"
    os.makedirs(OUT, exist_ok=True)
    install_mmcv_shim()
    sys.path.insert(0, REF)
    cwd = os.getcwd()
    os.chdir(REF)
    try:
        from utils.utils import extract_frames          # the reference's sampler, unmodified
        # ---- 1. sampler indices over a grid of (frame_cnt, fps, method)
        cases, flat, offs = [], [], [0]
        for cnt in (3, 4, 10, 65, 100, 355, 420, 1000, 2997, 18000):
            for fps in (19.62, 23.976, 25.0, 29.97, 30.0, 60.0):
                for method in ("uni_1", "uni_2", "uni_12", "uni_64", "fix_1", "fix_2", "fix_5"):
                    frames, fps_out, ts = extract_frames(f"synthetic:{cnt}:{fps}", method)
                    cases.append((cnt, fps, method))
                    flat.extend(int(f) for f in frames)
                    offs.append(len(flat))
        np.savez_compressed(os.path.join(OUT, "sampler_indices.npz"),
                            frame_cnt=np.array([c[0] for c in cases], np.int64),
                            fps=np.array([c[1] for c in cases], np.float64),
                            method=np.array([c[2] for c in cases]),
                            flat=np.array(flat, np.int64), offsets=np.array(offs, np.int64))
        print("sampler cases:", len(cases))

        # ---- 2. BASELINE config 1: uni_12 on the sample video through the reference sampler (real decode)
        frames, fps, ts = extract_frames(os.path.join(REF, "sample", "v_GGSY1Qvo990.mp4"), "uni_12")
        frames = np.stack(frames)                        # (12,240,320,3) uint8 BGR
        import cv2
        cap = cv2.VideoCapture(os.path.join(REF, "sample", "v_GGSY1Qvo990.mp4"))
        cnt = int(cap.get(cv2.CAP_PROP_FRAME_COUNT))
        idx = np.linspace(1, cnt - 2, 12).astype(int)
        # the reference transform on two of them: Image.fromarray (no BGR swap) -> torchvision Resize/CenterCrop
        from PIL import Image
        import torchvision.transforms as T
        tf = T.Compose([T.Resize(224, interpolation=T.InterpolationMode.BICUBIC), T.CenterCrop(224)])
        keep = [0, 7]
        cropped = np.stack([np.asarray(tf(Image.fromarray(frames[i]))) for i in keep])
        np.savez_compressed(os.path.join(OUT, "config1_sample_video.npz"), indices=idx, fps=np.float64(fps),
                            frame_cnt=np.int64(cnt), timestamps_ms=np.array(ts, np.float64),
                            frames=frames[keep], kept=np.array(keep), resized_cropped=cropped,
                            frame_checksums=np.array([int(f.astype(np.uint64).sum()) for f in frames], np.uint64))
        print("config1: indices", idx.tolist(), "fps", fps)

        # ---- 3. I3D host resize chain (ToPILImage -> ResizeImproved(256) bilinear) from the reference transforms
        from models.i3d.transforms.transforms import ResizeImproved, PILToTensor, TensorCenterCrop
        import torch
        import torchvision
        rng = np.random.default_rng(5)
        src = [frames[0], rng.integers(0, 256, (135, 240, 3), dtype=np.uint8),
               rng.integers(0, 256, (150, 128, 3), dtype=np.uint8)]
        outs = []
        for s in src:
            t = torch.from_numpy(s).permute(2, 0, 1)
            r = PILToTensor()(ResizeImproved(256)(torchvision.transforms.ToPILImage()(t)))
            outs.append(r.permute(1, 2, 0).numpy())
        np.savez_compressed(os.path.join(OUT, "i3d_resize.npz"),
                            **{f"src{i}": s for i, s in enumerate(src)}, **{f"out{i}": o for i, o in enumerate(outs)})
        print("i3d resize:", [o.shape for o in outs])
    finally:
        os.chdir(cwd)

    # ---- 4. Pillow itself (third-party; the CLIP transform's Resize) on random images, incl. an up-scale
    from PIL import Image
    rng = np.random.default_rng(0)
    d = {}
    for n, (h, w, oh, ow, f) in enumerate([(240, 320, 224, 298, Image.BICUBIC), (90, 120, 56, 74, Image.BICUBIC),
                                           (100, 60, 373, 224, Image.BICUBIC), (120, 160, 128, 170, Image.BILINEAR),
                                           (135, 240, 128, 227, Image.BILINEAR), (64, 48, 31, 17, Image.BICUBIC)]):
        im = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
        if n == 4:      # replayed from the seed by the test instead of stored: keeps the file under 1 MB
            d[f"shape{n}"] = np.array(im.shape, np.int64)
        else:
            d[f"in{n}"] = im
        d[f"out{n}"] = np.asarray(Image.fromarray(im).resize((ow, oh), f))
        d[f"filter{n}"] = np.int64(f)
    import PIL
    d["pillow_version"] = np.array(PIL.__version__)
    np.savez_compressed(os.path.join(OUT, "pillow_resize.npz"), **d)

    # ---- 5. CLIP tower: oracle restatement vs HF transformers (independent implementation), seeded
    import torch
    from transformers import CLIPVisionConfig, CLIPVisionModelWithProjection
    from oracle import clip_tower
    sd = clip_tower.synthetic_state_dict(0)
    hf = CLIPVisionModelWithProjection(CLIPVisionConfig()).eval()
    missing = hf.load_state_dict(clip_tower.to_hf_state_dict(sd), strict=False)
    g = torch.Generator().manual_seed(11)
    x = torch.randn(4, 3, 224, 224, generator=g)
    with torch.no_grad():
        y_hf = hf(pixel_values=x).image_embeds
    y_or = clip_tower.encode_image(sd, x)
    print("oracle vs HF rel:", float((y_or - y_hf).norm() / y_hf.norm()), "missing:", missing.missing_keys)
    np.savez_compressed(os.path.join(OUT, "clip_tower_seed0.npz"), x_seed=np.int64(11), y_hf=y_hf.numpy(),
                        y_oracle=y_or.numpy())




def i3d_golden():
    """Reference I3D module + vendored checkpoints vs the restated oracle, seeded inputs; stores only the outputs."""
    import torch
    sys.path.insert(0, REF)
    cwd = os.getcwd()
    os.chdir(REF)
    try:
        from models.i3d.i3d_src.i3d_net import I3D
        from oracle import i3d_net
        d = {}
        for mod, cin in (("rgb", 3), ("flow", 2)):
            sd = torch.load(f"models/i3d/checkpoints/i3d_{mod}.pt", map_location="cpu")
            net = I3D(num_classes=400, modality=mod).eval()
            net.load_state_dict(sd)
            for T in (16, 11):
                x = torch.rand(1, cin, T, 224, 224, generator=torch.Generator().manual_seed(100 + T)) * 2 - 1
                with torch.no_grad():
                    y_ref = net(x, features=True)
                y_or = i3d_net.forward_features(sd, x)
                rel = float((y_or - y_ref).norm() / y_ref.norm())
                print(f"i3d {mod} T={T}: oracle vs reference rel {rel:.2e}")
                assert rel < 1e-5
                d[f"{mod}_T{T}"] = y_ref.numpy()
        # synthetic-weight outputs, so the oracle is also pinned where the checkpoints are not available
        for mod, cin in (("rgb", 3), ("flow", 2)):
            sd = i3d_net.synthetic_state_dict(mod, 0)
            net = I3D(num_classes=400, modality=mod).eval()
            net.load_state_dict(sd, strict=False)
            x = torch.rand(1, cin, 12, 224, 224, generator=torch.Generator().manual_seed(7)) * 2 - 1
            with torch.no_grad():
                y_ref = net(x, features=True)
            y_or = i3d_net.forward_features(sd, x)
            print(f"i3d {mod} synthetic: rel {float((y_or - y_ref).norm() / y_ref.norm()):.2e}")
            d[f"{mod}_synth_T12"] = y_ref.numpy()
        np.savez_compressed(os.path.join(OUT, "i3d_outputs.npz"), **d)
    finally:
        os.chdir(cwd)


if __name__ == "__main__" and len(sys.argv) > 1 and sys.argv[1] == "i3d":
    i3d_golden()
    raft_golden()


if __name__ == "__main__" and len(sys.argv) == 1:
    main()
    i3d_golden()
    raft_golden()


def raft_golden():
    """Reference RAFT module + vendored raft-sintel.pth vs the restated oracle on synthetic moving frames."""
    import torch
    sys.path.insert(0, REF)
    cwd = os.getcwd()
    os.chdir(REF)
    try:
        from models.raft.raft_src.raft import RAFT, InputPadder
        from oracle import raft_net
        sd = torch.load("models/raft/checkpoints/raft-sintel.pth", map_location="cpu")
        net = torch.nn.DataParallel(RAFT(), device_ids=None)
        net.load_state_dict(sd)
        net = net.module.eval()
        d = {}
        for (h, w, n) in ((128, 160, 3), (270, 480, 2)):
            fr = raft_net.synthetic_frames(n, h, w, seed=h)
            padder = InputPadder(fr.shape)
            x = padder.pad(fr)
            assert torch.equal(x, raft_net.pad(fr))
            with torch.no_grad():
                y_ref = net(x[:-1], x[1:], iters=20)
            y_or = raft_net.forward(sd, x[:-1], x[1:], 20)
            rel = float((y_or - y_ref).norm() / y_ref.norm())
            print(f"raft {h}x{w}: oracle vs reference rel {rel:.2e}; mean |flow| {float(y_ref.abs().mean()):.3f}")
            assert rel < 1e-4
            full = padder.unpad(y_ref).numpy().astype(np.float32)
            d[f"flow_{h}x{w}"] = full if h < 200 else full[:, :, ::3, ::3]      # keep the fixture small
        np.savez_compressed(os.path.join(OUT, "raft_outputs.npz"), **d)
    finally:
        os.chdir(cwd)


if __name__ == "__main__" and len(sys.argv) > 1 and sys.argv[1] == "raft":
    raft_golden()


def checkpoint_stats():
    """Per-tensor statistics of the reference's vendored checkpoints -> tests/golden/checkpoint_stats.npz, from which
    oracle/checkpoint_standins.py draws seeded stand-ins (the checkpoints themselves are not part of the repository)."""
    import torch
    d = {}
    for name, rel in (("i3d_rgb.pt", "models/i3d/checkpoints/i3d_rgb.pt"), ("i3d_flow.pt", "models/i3d/checkpoints/i3d_flow.pt"),
                      ("raft-sintel.pth", "models/raft/checkpoints/raft-sintel.pth")):
        sd = torch.load(os.path.join(REF, rel), map_location="cpu")
        stats = []
        for v in sd.values():
            x = v.double()
            stats.append([float(x.mean()), float(x.std()) if x.numel() > 1 else 0.0, float(x.min()), float(x.max()),
                          float(v.is_floating_point())])
        d[f"{name}/keys"] = np.array(list(sd))
        d[f"{name}/ndim"] = np.array([v.dim() for v in sd.values()], np.int64)
        d[f"{name}/dims"] = np.array([s for v in sd.values() for s in v.shape], np.int64)
        d[f"{name}/stats"] = np.array(stats, np.float64)
    np.savez_compressed(os.path.join(OUT, "checkpoint_stats.npz"), **d)


def standin_golden():
    """The reference's I3D and RAFT modules on the checkpoint stand-ins of oracle/checkpoint_standins.py, seeded inputs
    (the same the tests draw) -> tests/golden/standin_outputs.npz.  The flow fields are kept on a strided grid (small
    fixture); `raft_stride_<h>x<w>` records the stride."""
    import torch
    from oracle.checkpoint_standins import state_dict as checkpoint
    sys.path.insert(0, REF)
    cwd = os.getcwd()
    os.chdir(REF)
    try:
        from models.i3d.i3d_src.i3d_net import I3D
        from models.raft.raft_src.raft import RAFT, InputPadder
        from oracle import i3d_net, raft_net
        d = {}
        for mod, cin in (("rgb", 3), ("flow", 2)):
            sd = checkpoint(f"i3d_{mod}.pt")
            net = I3D(num_classes=400, modality=mod).eval()
            net.load_state_dict(sd)
            for T in (16, 11):
                x = torch.rand(1, cin, T, 224, 224, generator=torch.Generator().manual_seed(100 + T)) * 2 - 1
                with torch.no_grad():
                    y_ref = net(x, features=True)
                rel = float((i3d_net.forward_features(sd, x) - y_ref).norm() / y_ref.norm())
                print(f"i3d {mod} stand-in T={T}: oracle vs reference rel {rel:.2e}; |y| {float(y_ref.norm()):.3e}")
                assert rel < 1e-5
                d[f"i3d_{mod}_T{T}"] = y_ref.numpy()
        sd = checkpoint("raft-sintel.pth")
        net = torch.nn.DataParallel(RAFT(), device_ids=None)
        net.load_state_dict(sd)
        net = net.module.eval()
        for (h, w, n, step) in RAFT_GOLDEN_CASES:
            fr = raft_net.synthetic_frames(n, h, w, seed=h)
            padder = InputPadder(fr.shape)
            x = padder.pad(fr)
            with torch.no_grad():
                y_ref = net(x[:-1], x[1:], iters=20)
            rel = float((raft_net.forward(sd, x[:-1], x[1:], 20) - y_ref).norm() / y_ref.norm())
            print(f"raft stand-in {h}x{w}: oracle vs reference rel {rel:.2e}; mean |flow| {float(y_ref.abs().mean()):.3f}")
            assert rel < 1e-4
            d[f"raft_flow_{h}x{w}"] = padder.unpad(y_ref).numpy().astype(np.float32)[:, :, ::step, ::step]
            d[f"raft_stride_{h}x{w}"] = np.int64(step)
        np.savez_compressed(os.path.join(OUT, "standin_outputs.npz"), **d)
    finally:
        os.chdir(cwd)


RAFT_GOLDEN_CASES = ((128, 160, 3, 4), (270, 480, 2, 6))       # (h, w, frames, stride of the stored grid)

if __name__ == "__main__" and len(sys.argv) > 1 and sys.argv[1] == "standin":
    checkpoint_stats()
    standin_golden()
