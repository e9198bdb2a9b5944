"""ResNet throughput on one GPU: one JSON line per depth.

    python scripts/resnet_bench.py [--depths 18 34 50 101 152] [--frames 1000] [--reps 5] [--out DIR]

Per depth (seeded synthetic weights, seeded uint8 frames; inputs of 1000 frames are 230 MB of 240x320 uint8 and 600 MB
of fp32 224x224, larger than the 126 MB L2):
  * engine frames/s, device-resident: 240x320 uint8 (resize + crop + normalise + net) and 224x224 uint8 (crop only);
  * engine frames/s end to end from pinned host buffers (forward_frames_u8_host, 240x320);
  * GEMM time share and executed / algorithmic FLOPs (vf_gemm_profile in a separate eager pass; algorithmic FLOPs
    from the conv shapes here, 2 * MACs);
  * the torch bar on the same frames: the oracle's functional torch modules (oracle/resnet_net.py) in fp32 with TF32
    off, with TF32, and fp16 channels-last with cudnn.benchmark;
  * GPU name and power limit, read in the same run.
Every shape is warmed up first; each timing is the median of --reps repetitions, with min and max beside it.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import resnet_net  # noqa: E402
from video_features_b200 import ops, synthetic_weights as sw  # noqa: E402
from video_features_b200.resnet_engine import ResNetEngine  # noqa: E402


def algorithmic_flops(depth):
    """2 * MACs of every conv at 224x224 input (the fc is removed; pools and adds not counted)."""
    total = 0
    for name, (co, ci, k) in sw.resnet_conv_shapes(depth).items():
        out = 112 if name == "conv1" else 56 >> (int(name[5]) - 1)      # output side of the conv
        if k == 1 and name.endswith(".0.conv1") and name[5] != "1" and sw.RESNET_BLOCKS[depth][0] == "bottleneck":
            out *= 2                                                     # the 1x1 before the strided 3x3
        total += 2 * co * ci * k * k * out * out
    return total


def timed(fn, reps):
    ts = []
    for _ in range(reps):
        torch.cuda.synchronize()
        t = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        ts.append(time.perf_counter() - t)
    return float(np.median(ts)), float(min(ts)), float(max(ts))


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else torch.cuda.get_device_name(0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--depths", type=int, nargs="+", default=[18, 34, 50, 101, 152])
    ap.add_argument("--frames", type=int, default=1000)
    ap.add_argument("--chunk", type=int, default=256)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "resnet_bench needs a GPU"
    info = gpu_info()
    n = a.frames
    g = torch.Generator().manual_seed(3)
    u8_240 = torch.randint(0, 256, (n, 240, 320, 3), dtype=torch.uint8, generator=g)
    u8_224 = u8_240[:, 8:232, 48:272].contiguous()
    d240, d224 = u8_240.cuda(), u8_224.cuda()
    host = u8_240.pin_memory()
    lines = []
    for depth in a.depths:
        sd = sw.resnet_state_dict(depth, 0)
        eng = ResNetEngine(sd, depth, 0, max_frames=a.chunk)
        r = {"depth": depth, "gpu": info, "frames": n, "chunk": a.chunk}
        eng.forward_frames_u8(d240); eng.forward_frames_u8(d224); eng.forward_frames_u8_host(host)   # warm-up
        for tag, fn in (("dev_240x320", lambda: eng.forward_frames_u8(d240)),
                        ("dev_224x224", lambda: eng.forward_frames_u8(d224)),
                        ("host_240x320", lambda: eng.forward_frames_u8_host(host))):
            med, lo, hi = timed(fn, a.reps)
            r[f"fps_{tag}"] = n / med
            r[f"fps_{tag}_min_max"] = [n / hi, n / lo]
        launches0 = eng.launch_count
        eng.forward_frames_u8(d224)
        torch.cuda.synchronize()
        r["launches_per_call"] = eng.launch_count - launches0
        ops.gemm_profile(True)
        t0 = time.perf_counter()
        eng.forward_frames_u8(d224)
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        gms, gl, gf = ops.gemm_profile_read()
        ops.gemm_profile(False)
        alg = algorithmic_flops(depth) * n
        r.update(gemm_ms=gms, gemm_launches=gl, gemm_share_of_eager_wall=gms / 1e3 / wall, executed_flops=gf,
                 algorithmic_flops=alg, executed_over_algorithmic=gf / alg, gemm_tflops_executed=gf / (gms / 1e3) / 1e12)
        eng.close()
        # torch bar on the same 224x224 frames
        sdc = {k: v.cuda() for k, v in sd.items()}
        mean = torch.tensor(resnet_net.MEAN, device="cuda").view(1, 3, 1, 1)
        std = torch.tensor(resnet_net.STD, device="cuda").view(1, 3, 1, 1)
        x = (d224.permute(0, 3, 1, 2).float().div(255) - mean) / std
        for tag, tf32, half in (("torch_fp32", False, False), ("torch_tf32", True, False), ("torch_fp16_cl", False, True)):
            torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = tf32
            torch.backends.cudnn.benchmark = half
            if half:
                sdh = {k: (v.half() if v.is_floating_point() else v) for k, v in sdc.items()}
                sdh = {k: (v.to(memory_format=torch.channels_last) if v.dim() == 4 else v) for k, v in sdh.items()}
                xi = x.half().to(memory_format=torch.channels_last)
            else:
                sdh, xi = sdc, x
            def run():
                for i in range(0, n, a.chunk):
                    resnet_net.forward_features(sdh, xi[i:i + a.chunk], depth)
            run()
            med, lo, hi = timed(run, a.reps)
            r[f"fps_{tag}"] = n / med
            r[f"fps_{tag}_min_max"] = [n / hi, n / lo]
        torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
        torch.backends.cudnn.benchmark = False
        print(json.dumps(r), flush=True)
        lines.append(r)
        del sdc
        torch.cuda.empty_cache()
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "resnet_bench.json"), "w") as f:
            for r in lines:
                f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
