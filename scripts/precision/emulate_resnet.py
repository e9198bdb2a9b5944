"""CPU emulation behind DESIGN.md §4.6 (ResNet precision policy): which fp16-rounded tensors the feature error of the
seeded ResNet weights (video_features_b200.synthetic_weights, seed 0) comes from, for depth 50 and 152, on uniform
noise frames and on frames of the sample video (tests/golden/v_GGSY1Qvo990.mp4, cv2 read, BGR->RGB, the extractor's
transform).  The engine applies BN as an fp32 scale / bias in the GEMM epilogue, so the weights rounded are the raw
conv weights; "split" stands for a split-fp16 pair (hi + lo, ~2^-22 relative), emulated as fp32.

Tensor groups: stem input (the normalised frame), residual stream (block inputs / outputs, read by the 1x1 convs and
the downsample), branch intermediates (the inputs of the 3x3 convs and of the bottleneck's last 1x1), weights.

Bar (per output row, against the fp32 oracle): rel-L2 <= 1e-3 and max-abs <= 1e-3 * max |ref|.  The output of the run
is committed as profiles/resnet_precision.txt.
"""
import os
import sys

import numpy as np
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import resnet_net as N  # noqa: E402
from video_features_b200 import synthetic_weights as sw  # noqa: E402


def q(x, on):
    return x.half().float() if on else x


def forward(sd, x, depth, pol):
    """pol: dict of booleans: stem / stream / inner (activations rounded to single fp16), weights (fp16 weights)."""
    kind, blocks = sw.RESNET_BLOCKS[depth]

    def conv(name, t, stride=1, padding=0):
        w = sd[name + ".weight"]
        y = F.conv2d(t, q(w, pol["weights"]), stride=stride, padding=padding)
        return N._bn(sd, sw.resnet_bn_name(name), y)

    x = F.relu(conv("conv1", q(x, pol["stem"]), 2, 3))
    x = q(F.max_pool2d(x, 3, 2, 1), pol["stream"])
    for li, nb in enumerate(blocks):
        for b in range(nb):
            p, s = f"layer{li + 1}.{b}", (2 if (b == 0 and li > 0) else 1)
            if kind == "bottleneck":
                y = q(F.relu(conv(p + ".conv1", x)), pol["inner"])
                y = q(F.relu(conv(p + ".conv2", y, s, 1)), pol["inner"])
                y = q(conv(p + ".conv3", y), pol["inner"])
            else:
                y = q(F.relu(conv(p + ".conv1", x, s, 1)), pol["inner"])
                y = q(conv(p + ".conv2", y, 1, 1), pol["inner"])
            r = q(conv(p + ".downsample.0", x, s), pol["inner"]) if p + ".downsample.0.weight" in sd else x
            x = q(F.relu(r + y), pol["stream"])
    return x.mean(dim=(2, 3))


def frames(kind, n=8):
    if kind == "noise":
        g = np.random.default_rng(1)
        u8 = g.integers(0, 256, (n, 240, 320, 3), dtype=np.uint8)
    else:
        import cv2
        cap = cv2.VideoCapture(os.path.join(ROOT, "tests", "golden", "v_GGSY1Qvo990.mp4"))
        out = []
        while len(out) < 40 * n:
            ok, f = cap.read()
            if not ok:
                break
            out.append(cv2.cvtColor(f, cv2.COLOR_BGR2RGB))
        u8 = np.stack(out[::40][:n])
    return N.transform_batch(u8)


def main():
    torch.set_num_threads(os.cpu_count() or 1)
    pols = {
        "all single fp16 (weights, stem, stream, inner)": dict(weights=1, stem=1, stream=1, inner=1),
        "fp16 weights only, activations split": dict(weights=1, stem=0, stream=0, inner=0),
        "single fp16 stem input only": dict(weights=0, stem=1, stream=0, inner=0),
        "single fp16 residual stream only": dict(weights=0, stem=0, stream=1, inner=0),
        "single fp16 branch intermediates only": dict(weights=0, stem=0, stream=0, inner=1),
        "fp16 weights + single fp16 intermediates, split stream": dict(weights=1, stem=0, stream=0, inner=1),
        "fp16 weights + single fp16 stream, split intermediates": dict(weights=1, stem=0, stream=1, inner=0),
    }
    print("per-row worst case over the frames: rel-L2 / max-abs relative to max |ref| (bar: 1e-3 / 1e-3)")
    for depth in (50, 152):
        sd = sw.resnet_state_dict(depth, 0)
        for fk in ("noise", "video"):
            x = frames(fk)
            ref = N.forward_features(sd, x, depth).double()
            for tag, pol in pols.items():
                with torch.no_grad():
                    y = forward(sd, x, depth, pol).double()
                rel = ((y - ref).norm(dim=1) / ref.norm(dim=1)).max().item()
                mx = ((y - ref).abs().amax(dim=1) / ref.abs().amax(dim=1)).max().item()
                print(f"resnet{depth:<3d} {fk:5s} {tag:58s} {rel:.2e} / {mx:.2e}", flush=True)


if __name__ == "__main__":
    main()
