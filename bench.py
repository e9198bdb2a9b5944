#!/usr/bin/env python
"""bench.py -- frames/sec of the CLIP ViT-B/32 hot path (BASELINE.json configs[1]) on N B200s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

A "step" is one pass of the hot path (uint8 frames -> transform -> ViT-B/32 tower -> (n,512) fp32 features)
over one batch of 1000 synthetic 224x224x3 uint8 frames per GPU.  Prints ONE JSON line (rank 0):
  value     whole-job frames/s, inputs resident in HBM, CUDA-event timed, max over ranks
  e2e       same metric through the host-buffer C-ABI call (pinned host frames in, host features out; the H2D and
            D2H copies are inside the timed region)
  roofline  tensor-pipe roofline of the dominant kernel (the tcgen05 GEMM), from per-launch CUDA events
  cpu_baseline  the oracle port (PIL transform + fp32 torch tower) timed on this box's host cores (N=1, rank 0)
`--impl reference` times only that CPU path (the reference's `--cpu` path restated; see DESIGN.md) and prints the
same line with "impl": "reference".
`--dump-outputs DIR` writes what the timed path returned in its last timed step as DIR/<name>.npy (float32): the
(n, 512) features (all ranks' rows, gathered, when N > 1; with --impl reference the first 32 frames' rows).  Inputs and
weights are seeded, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time
import traceback

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

# stdout carries exactly ONE JSON line: everything else a library prints there (NCCL's version banner, ...) is sent to
# stderr by pointing fd 1 at fd 2 for the life of the process and writing the result to the saved descriptor.
_REAL_STDOUT = os.dup(1)
os.dup2(2, 1)


def emit(line: dict) -> None:
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


FRAMES_PER_STEP = 1000
REFERENCE_FRAMES_PER_STEP = 32           # --impl reference: frames of the 1000 the CPU oracle port runs per step
METRIC = "frames/sec CLIP-ViT-B/32 @224px"
UNIT = "frames/s"
WORKLOAD = "CLIP-ViT-B/32 fix_2 on 1k synthetic 224x224 RGB frames (BASELINE.json configs[1])"
GEMM_FLOP_PER_FRAME = 231_211_008 + 12 * (715_468_800 - 2 * 3_840_000) + 786_432   # 2*M*N*K of the GEMM launches
FLOP_PER_FRAME = 231_211_008 + 12 * 715_468_800 + 786_432                            # SURVEY.md 8(d): 8.818 GFLOP
# algorithmic HBM bytes per frame of the memory-bound kernel classes (DESIGN.md 4): LayerNorm = 24 passes over the
# 50x768 residual rows + the embedding pass; attention = q,k,v in + o out per (frame, head, layer); transform = u8 in +
# fp16 patch matrix out
HBM_BYTES_PER_FRAME = {"layernorm": 24 * 50 * 768 * 6 + 50 * 768 * 8,   # x fp32 read + h fp16 written = 6 B / element (the residual
                                                                        # add happens in the GEMM epilogue); embed pass 8 B
                       "attention": 12 * 50 * 768 * 2 * 4, "transform": 150_528 + 301_056}


def base_config(n_gpus: int) -> dict:
    return {
        "workload": WORKLOAD,
        "feature_type": "CLIP-ViT-B/32",
        "frames_per_step_per_gpu": FRAMES_PER_STEP,
        "frame": "224x224x3 uint8 HWC",
        "weights": "synthetic, seed 0, openai visual.* layout (real CLIP weights are not available offline)",
        "accumulate": "fp32",
        "l2": "inputs are 150.5 MB per step per GPU > 126 MB L2 (no explicit flush needed)",
        "parallelism": f"dp{n_gpus}: frame list sharded per rank, one NCCL all_gather of the (n,512) features per step "
                       "(side stream: overlaps the next step's tower)" if n_gpus > 1 else "dp1",
    }


def ncu_traffic_per_launch():
    """Mean DRAM bytes (read + write) per launch of the dominant kernel, from the committed ncu --set full capture
    (profiles/r2_prof_gemm_raw.csv, else round 1's: consecutive GEMM launches of one 250-frame chunk); None if absent."""
    import csv
    p = os.path.join(ROOT, "profiles", "r2_prof_gemm_raw.csv")
    if not os.path.exists(p):
        p = os.path.join(ROOT, "profiles", "r1_prof_gemm_raw.csv")
    try:
        rows = list(csv.reader(open(p)))
        hdr, units, data = rows[0], rows[1], rows[2:]
        mult = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
        ir, iw = hdr.index("dram__bytes_read.sum"), hdr.index("dram__bytes_write.sum")
        tot = [float(d[ir]) * mult[units[ir]] + float(d[iw]) * mult[units[iw]] for d in data]
        return sum(tot) / len(tot)
    except Exception:
        return None


def load_peaks() -> dict:
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"tflops_sustained": float(d.get("bf16_tflops_sustained", d.get("bf16_tflops", 1400.0))),
                "tflops_burst": float(d.get("bf16_tflops", 1590.0)), "hbm_gbs": float(d.get("hbm_gbs", 6650.0)),
                "source": "measured (MEASURED_PEAKS.json)"}
    return {"tflops_sustained": 1400.0, "tflops_burst": 1590.0, "hbm_gbs": 6650.0,
            "source": "fallback (B200_PROFILING.md)"}


# ----------------------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.path = tempfile.mktemp(prefix="vf_clocks_", suffix=".csv")
        self.proc = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(gpu_index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-lms", "50"], stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.06)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        try:
            for line in open(self.path):
                f = [x.strip() for x in line.split(",")]
                if len(f) < 7:
                    continue
                try:
                    sm.append(float(f[0])); mx.append(float(f[1])); pw.append(float(f[2]))
                except ValueError:
                    continue
                for n, v in zip(names, f[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            os.unlink(self.path)
        except Exception:
            pass
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        # "under load": samples in the upper half of the observed power range
        thr = (max(pw) + min(pw)) / 2 if pw else 0
        loaded = [s for s, p in zip(sm, pw) if p >= thr] or sm
        return {"sm_mhz": statistics.median(loaded), "sm_max_mhz": max(mx), "power_w_max": max(pw),
                "samples": len(sm), "reasons": sorted(reasons)}


# ----------------------------------------------------------------------------------------- CPU (oracle) arm
def synth_frames_host(n: int, seed: int):
    import torch
    g = torch.Generator().manual_seed(seed)
    return torch.randint(0, 256, (n, 224, 224, 3), dtype=torch.uint8, generator=g)


def dump_outputs(out_dir: str, arrays: dict) -> None:
    """--dump-outputs: one float32 DIR/<name>.npy per array."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        a = a.detach().cpu().numpy() if hasattr(a, "detach") else np.asarray(a)
        np.save(os.path.join(out_dir, f"{name}.npy"), a.astype(np.float32))


def cpu_step(sd, frames_np):
    """The reference's per-video flow (models/CLIP/extract_clip.py:107-131) on the oracle port:
    PIL transform per frame -> stack -> fp32 tower -> numpy."""
    import torch
    from oracle import clip_preprocess, clip_tower
    batch = clip_preprocess.preprocess_batch(frames_np)
    with torch.no_grad():
        return clip_tower.encode_image(sd, batch).numpy()


def usable_cores() -> int:
    """Host cores this process may actually use: affinity mask capped by the cgroup CPU quota (os.cpu_count()
    reports the whole machine inside a container and oversubscribing OpenMP threads stalls for minutes)."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    quota = None
    try:
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if q != "max":
            quota = float(q) / float(p)
    except Exception:
        try:
            q = float(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            p = float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                quota = q / p
        except Exception:
            pass
    if quota:
        n = min(n, max(1, int(quota + 0.5)))
    return max(1, n)


def time_cpu(reps: int, warm: int, budget_s: float = 20.0, sample: int = 0):
    """Times the oracle port on the first `sample` frames of the engine arm's rank-0 step (the same seeded frames, so
    its features are rows 0 .. sample-1 of that step's).  sample = 0: chosen from a probe so that warm-up + reps stay
    near `budget_s` seconds of CPU work.  -> (per-rep seconds, cores, sample, features of the last rep)"""
    import torch
    from video_features_b200 import synthetic_weights
    cores = usable_cores()
    torch.set_num_threads(cores)
    sd = synthetic_weights.clip_vit_b32_state_dict(0)
    frames = synth_frames_host(FRAMES_PER_STEP, 100).numpy()
    cpu_step(sd, frames[:4])                                   # page in / thread pool start
    if not sample:
        t0 = time.perf_counter()
        cpu_step(sd, frames[:16])
        probe = max(time.perf_counter() - t0, 1e-3)
        per_frame = probe / 16
        sample = int(max(16, min(256, budget_s / max(reps + warm, 1) / per_frame)))
        sample -= sample % 8
    frames = frames[:sample]
    for _ in range(warm):
        cpu_step(sd, frames)
    ts, y = [], None
    for _ in range(reps):
        t0 = time.perf_counter()
        y = cpu_step(sd, frames)
        ts.append(time.perf_counter() - t0)
    return ts, cores, sample, y


def cpu_model_name() -> str:
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


def run_reference(args, rank: int) -> None:
    if rank != 0:
        return
    # each step is a fixed sample of the headline step's frames, so the arm's time grows linearly with --steps and its
    # --dump-outputs rows are the same from run to run (and equal rows 0 .. sample-1 of the engine arm's dump)
    ts, cores, sample, y = time_cpu(args.steps, min(max(args.warmup, 1), 3), sample=REFERENCE_FRAMES_PER_STEP)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"features": y})
    total = sum(ts)
    value = sample * len(ts) / total
    desc = (f"{sample} of the 1000 frames per step; PIL transform + fp32 torch tower (oracle port of the "
            f"reference --cpu path), torch threads={cores}, {cpu_model_name()}")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": len(ts), "warmup": min(max(args.warmup, 1), 3), "ms_per_step": 1e3 * total / len(ts),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": base_config(args.gpus),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": desc},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


# ----------------------------------------------------------------------------------------- GPU arm
def run_engine(args, rank: int, world: int, local_rank: int) -> None:
    import torch
    import torch.distributed as dist
    from video_features_b200 import synthetic_weights
    from video_features_b200.clip_engine import ClipEngine

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the engine has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    sd = synthetic_weights.clip_vit_b32_state_dict(0)
    eng = ClipEngine(sd, device=local_rank, chunk_frames=args.chunk)
    n = FRAMES_PER_STEP
    frames_host = synth_frames_host(n, 100 + rank).pin_memory()
    frames_dev = frames_host.to(dev)
    out_host = torch.empty((n, 512), dtype=torch.float32).pin_memory()
    # e2e: consecutive steps alternate between two pinned input / output buffer pairs (step k+1 is enqueued while step k
    # runs, as a list of videos is processed: the second pair stands for "the next batch the decoder filled")
    frames_host_b = synth_frames_host(n, 300 + rank).pin_memory()
    out_host_b = torch.empty((n, 512), dtype=torch.float32).pin_memory()
    inflight = []
    # N > 1: the all-gather of step k runs on a side stream while the tower of step k+1 runs (two landing buffers);
    # the timed region ends only after the last gather has finished
    gathered = [torch.empty((world * n, 512), dtype=torch.float32, device=dev) for _ in range(2)] if world > 1 else None
    side = torch.cuda.Stream(device=dev) if world > 1 else None
    tick = [0]
    last = {}

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def gather_async(y):
        ev = torch.cuda.Event()
        ev.record()
        side.wait_event(ev)
        with torch.cuda.stream(side):
            dist.all_gather_into_tensor(gathered[tick[0] & 1], y)
        y.record_stream(side)
        tick[0] += 1

    def step_dev():
        y = eng.encode_frames_u8(frames_dev)
        if world > 1:
            gather_async(y)
        last["y"] = y
        return y

    def step_host():
        # every step: H2D of its own pinned frames, tower, D2H of its features into its own pinned buffer.  The call is
        # asynchronous (vf_clip_encode_u8_host_async); the PREVIOUS step's result is awaited right after this one is
        # enqueued, so at most two steps are in flight and every result is on the host inside the timed region.
        a = len(inflight) == 0 or inflight[-1][1] is out_host_b
        fr, oh = (frames_host, out_host) if a else (frames_host_b, out_host_b)
        # N > 1: the features also stay on the device for the gather
        ticket, y = eng.encode_frames_u8_host_async(fr, oh, out_dev=world > 1)
        if world > 1:
            gather_async(y)
        inflight.append((ticket, oh))
        while len(inflight) > 1:
            eng.wait(inflight.pop(0)[0])
        return y

    def drain_host():
        while inflight:
            eng.wait(inflight.pop(0)[0])

    def timed(fn, steps, drain=None):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        if drain is not None:
            drain()
        if side is not None:
            torch.cuda.current_stream().wait_stream(side)
        e1.record()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        barrier()
        return float(ms.item())

    W, K = max(args.warmup, 3), args.steps
    for _ in range(W):
        step_dev()
    launches0 = eng.launch_count
    sampler = ClockSampler(local_rank) if rank == 0 else None
    ms_total = timed(step_dev, K)
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"features": gathered[(tick[0] - 1) & 1] if world > 1 else last["y"]})
    launches = (eng.launch_count - launches0) // K
    value = world * n * K / (ms_total / 1e3)

    # end-to-end through the host-buffer entry point
    for _ in range(2):
        step_host()
    drain_host()
    ms_e2e = timed(step_host, K, drain_host)
    e2e_value = world * n * K / (ms_e2e / 1e3)

    # roofline of the dominant kernel: per-launch CUDA events around every tcgen05 GEMM launch, separate pass over
    # the same steps so the timed region above is not perturbed
    eng.profile(True)
    pk = min(K, 5)
    for _ in range(pk):
        eng.encode_frames_u8(frames_dev)
    gemm_ms, gemm_launches, gemm_flops = eng.profile_read()
    cats = {k: v / pk for k, v in eng.profile_categories().items()}
    eng.profile(False)
    peaks = load_peaks()
    # algorithmic FLOPs of the reference's GEMMs (SURVEY.md 8d) over the measured GEMM time; the engine executes
    # 5.9 % fewer (the last block's out-proj / MLP run on the CLS rows only), reported separately
    # The dominant kernel is the plain tcgen05 GEMM (patch embedding, out-proj, fc1, fc2, final projection; plus QKV when
    # VF_CLIP_ATTN=split).  With the default fused path the QKV projection runs inside vf::qkv_attention_kernel together
    # with the attention core: that kernel is timed as its own class ("attention") and reported under `qkv_attention`.
    fused = not os.environ.get("VF_CLIP_ATTN", "").startswith("s")
    QKV_FLOP, ATT_CORE_FLOP = 12 * 176_947_200, 12 * 2 * 3_840_000
    alg_flop = GEMM_FLOP_PER_FRAME - (QKV_FLOP if fused else 0)
    achieved = alg_flop * n * pk / (gemm_ms / 1e3) / 1e12 if gemm_ms > 0 else 0.0
    executed = gemm_flops / (gemm_ms / 1e3) / 1e12 if gemm_ms > 0 else 0.0
    roofline = {
        "bound": "tensor", "kernel": "vf::gemm_f16_pair_kernel + vf::qkv_attention_kernel (tcgen05.mma cta_group::2 kind::f16, fp32 "
                                     "accumulate in TMEM)",
        "achieved": achieved, "peak": peaks["tflops_sustained"], "unit": "TFLOP/s",
        "frac": achieved / peaks["tflops_sustained"], "peak_source": peaks["source"] + ", bf16 dense sustained",
        "traffic": ncu_traffic_per_launch(), "traffic_unit": "bytes/launch (ncu dram__bytes_read+write, mean of 4 launches)",
        "executed_tflops": executed,
        "executed_over_algorithmic": gemm_flops / (alg_flop * n * pk),
        "algorithmic_gflop_per_frame": alg_flop / 1e9,
        "launches_per_step": gemm_launches // pk, "avg_launch_us": 1e3 * gemm_ms / max(gemm_launches, 1),
        "algorithmic_flop_per_launch_avg": alg_flop * n * pk / max(gemm_launches, 1),
        "gemm_share_of_step": (gemm_ms / pk) / (ms_total / K),
        "eager_ms_per_step_by_kernel": cats,
        "qkv_attention": ({"kernel": "vf::qkv_attention_kernel (QKV projection on tcgen05 + 50-token attention on mma.sync in the epilogue)",
                           "algorithmic_gflop_per_frame": (QKV_FLOP + ATT_CORE_FLOP) / 1e9, "ms_per_step": cats.get("attention", 0.0),
                           "achieved_tflops": (QKV_FLOP + ATT_CORE_FLOP) * n / (cats["attention"] / 1e3) / 1e12 if cats.get("attention") else None,
                           "frac": ((QKV_FLOP + ATT_CORE_FLOP) * n / (cats["attention"] / 1e3) / 1e12 / peaks["tflops_sustained"])
                           if cats.get("attention") else None} if fused else None),
        "whole_step_tflops": value / world * FLOP_PER_FRAME / 1e12,
        "whole_step_frac": value / world * FLOP_PER_FRAME / 1e12 / peaks["tflops_sustained"],
        # the memory-bound kernels against the HBM roofline: ALGORITHMIC bytes per frame (DESIGN.md 4) over their
        # event-timed device time; the chunk's activations partly live in the 126 MB L2, so > 1 is possible
        "hbm": {k: {"algorithmic_bytes_per_frame": b, "ms_per_step": cats.get(k, 0.0),
                    "achieved_gbs": (b * n / (cats[k] / 1e3) / 1e9) if cats.get(k) else None,
                    "frac_of_hbm_peak": (b * n / (cats[k] / 1e3) / 1e9 / peaks["hbm_gbs"]) if cats.get(k) else None}
                for k, b in HBM_BYTES_PER_FRAME.items() if not (fused and k == "attention")},
        "hbm_peak_gbs": peaks["hbm_gbs"],
    }

    # the Pillow-exact resample on config 1's geometry (240x320 -> 224x298 bicubic; the headline workload is 224x224 and
    # never resizes): algorithmic bytes = source + 2 x horizontal-pass intermediate + destination
    if rank == 0:
        import video_features_b200  # noqa: F401  (registers torch.ops.vfeat)
        from video_features_b200._lib import VF_FILTER_BICUBIC
        rn = 512
        rsrc = torch.randint(0, 256, (rn, 240, 320, 3), dtype=torch.uint8, device=dev)
        for _ in range(3):
            torch.ops.vfeat.resize_u8(rsrc, 224, 298, VF_FILTER_BICUBIC)
        torch.cuda.synchronize()
        r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        r0.record()
        for _ in range(10):
            torch.ops.vfeat.resize_u8(rsrc, 224, 298, VF_FILTER_BICUBIC)
        r1.record()
        torch.cuda.synchronize()
        rms = r0.elapsed_time(r1) / 10
        rbytes = rn * 3 * (240 * 320 + 2 * 240 * 298 + 224 * 298)
        roofline["hbm"]["resize_240x320_to_224x298_bicubic"] = {
            "algorithmic_bytes_per_frame": rbytes // rn, "ms_per_512_frames": rms, "achieved_gbs": rbytes / (rms / 1e3) / 1e9,
            "frac_of_hbm_peak": rbytes / (rms / 1e3) / 1e9 / peaks["hbm_gbs"], "frames_per_sec": rn / (rms / 1e3)}
        del rsrc

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": ms_total / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f16", "data": "synthetic",
        "config": dict(base_config(world), chunk_frames=args.chunk or "256 -> 4 balanced chunks of 250"),
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": UNIT, "ms_per_step": ms_e2e / K,
                "h2d_bytes_per_step": int(frames_host.numel()) * world,
                "d2h_bytes_per_step": int(out_host.numel() * 4) * world,
                "api": "vf_clip_encode_u8_host_async + vf_clip_wait (ClipEngine.encode_frames_u8_host_async), pinned host "
                       "buffers, two steps in flight"},
        "gpu_launches": int(launches * K),
        "gpu_launches_per_step": int(launches),
        "roofline": roofline,
    }
    if rank == 0 and world == 1 and not args.no_cpu:
        ts, cores, sample, _ = time_cpu(3, 1, budget_s=20.0)
        v = sample * len(ts) / sum(ts)
        line["cpu_baseline"] = {
            "value": v, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"{sample} of the 1000 frames x {len(ts)} reps (+1 warm-up); PIL transform + fp32 torch tower "
                      f"(oracle port of the reference --cpu path), torch threads={cores}, {cpu_model_name()}",
            "median_s_per_rep": statistics.median(ts)}
    if rank == 0 and world == 1 and args.torch_gpu:
        from oracle import clip_tower                  # the library-call bar: the oracle's torch modules on this GPU
        sdg = {k: v.to(dev) for k, v in sd.items()}
        xg = torch.randn(250, 3, 224, 224, device=dev)
        leg = _torch_gpu_leg(lambda: clip_tower.encode_image(sdg, xg), 250, UNIT,
                             "oracle port of the ViT-B/32 tower (torch eager, cuBLAS), 250 pre-normalised frames per call, transform excluded")
        # fp16 weights and activations: what `clip.load` gives the reference on a CUDA device (its GPU arithmetic)
        sdh = {k: v.half() for k, v in sdg.items()}
        xh = xg.half()
        with torch.no_grad():
            for _ in range(2):
                clip_tower.encode_image(sdh, xh)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(8):
                clip_tower.encode_image(sdh, xh)
            e1.record()
            torch.cuda.synchronize()
        leg["fp16"] = 250 * 8 / (e0.elapsed_time(e1) / 1e3)
        line["torch_gpu_baseline"] = leg
    eng.close()
    del eng, frames_dev
    torch.cuda.empty_cache()
    # ---- secondary workloads, measured by the same (driver-run) command: the video-list product path (BASELINE.json
    # configs[4], every N), I3D rgb (configs[2], N = 1) and RAFT -> I3D flow (configs[3], N = 1 and its 2-GPU form)
    if not args.no_secondary:
        sec = {}
        # watchdog: the secondary workloads contain collectives; if one ever hangs, the headline line (already complete)
        # is still emitted and every rank leaves -- a secondary line never takes the headline down with it
        import threading

        def _bail():
            line["secondary"] = dict(sec, error="timeout: secondary workloads did not finish within 240 s")
            if rank == 0:
                emit(line)
            os._exit(0)

        watchdog = threading.Timer(240.0, _bail)
        watchdog.daemon = True
        watchdog.start()
        for name, fn, ok in (("c5_video_list", lambda: run_c5(args, rank, world, local_rank, quick=True), True),
                             ("clip_vit_b16", lambda: run_b16(args, quick=True), world == 1),
                             ("i3d_rgb", lambda: run_i3d(args, quick=True), world == 1),
                             ("raft_i3d_flow", lambda: run_raft(args, rank, world, local_rank, quick=True), world <= 2)):
            if not ok:
                continue
            try:
                sec[name] = fn()
            except BaseException as err:               # a secondary line never takes the headline down with it
                sec[name] = {"error": f"{type(err).__name__}: {err}"}
                print(f"[bench rank {rank}] secondary workload {name} failed: {type(err).__name__}: {err}", file=sys.stderr, flush=True)
                traceback.print_exc()
        watchdog.cancel()
        line["secondary"] = sec
    if rank == 0:
        emit(line)
    if world > 1:
        dist.destroy_process_group()


# ----------------------------------------------------------------------------------------- secondary workloads
# BASELINE.json configs[2] (I3D rgb, 64-frame 224x224 stacks) and configs[3] (RAFT on 480x270 pairs -> I3D flow).
# They print the same kind of JSON line (metric stacks/s resp. pairs/s) for profiles/; the headline stays CLIP.
I3D_GFLOP = {"rgb": 222.30, "flow": 204.68}          # per 64-frame stack (SURVEY.md 8d / Appendix A)
RAFT_GFLOP_272x480 = 309.82                          # per pair, 20 iterations, reference algorithm (SURVEY.md 8d)


def _weights(kind: str):
    """Seeded stand-in of the reference's vendored checkpoint (oracle/checkpoint_standins.py): the same weights on every
    machine, so runs are comparable; the time does not depend on the values."""
    from oracle import checkpoint_standins
    name = {"rgb": "i3d_rgb.pt", "flow": "i3d_flow.pt", "raft": "raft-sintel.pth"}[kind]
    return checkpoint_standins.state_dict(name), f"seeded stand-in of {name} (per-tensor statistics of the vendored file)"


def _timed_loop(fn, steps, warm):
    import torch
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def _gemm_roofline(fn, reps, algorithmic_flops_per_step, step_ms):
    from video_features_b200 import ops
    ops.gemm_profile(True)
    for _ in range(reps):
        fn()
    ms, launches, executed = ops.gemm_profile_read()
    ops.gemm_profile(False)
    peaks = load_peaks()
    ach = algorithmic_flops_per_step * reps / (ms / 1e3) / 1e12 if ms > 0 else 0.0
    return {"bound": "tensor", "kernel": "vf::gemm_f16_pair_kernel (tcgen05, shifted-row conv mode)",
            "achieved": ach, "peak": peaks["tflops_sustained"], "unit": "TFLOP/s", "frac": ach / peaks["tflops_sustained"],
            "peak_source": peaks["source"] + ", bf16 dense sustained", "traffic": None,
            "executed_tflops": executed / (ms / 1e3) / 1e12 if ms > 0 else 0.0,
            "executed_over_algorithmic": executed / (algorithmic_flops_per_step * reps),
            "launches_per_step": launches // reps, "gemm_share_of_step": (ms / reps) / step_ms}


def _torch_gpu_leg(fn, units, unit, what):
    """The oracle's fp32 torch modules (cuDNN / cuBLAS library calls) on the same GPU: the "library call" bar of
    SURVEY 8(d).  Measured with TF32 off (the oracle's numerics) and on (the library's fast fp32 path)."""
    import torch
    out = {"unit": unit, "what": what}
    for tf32 in (False, True):
        torch.backends.cudnn.allow_tf32 = tf32
        torch.backends.cuda.matmul.allow_tf32 = tf32
        with torch.no_grad():
            fn(); torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(2):
                fn()
            e1.record(); torch.cuda.synchronize()
        out["tf32" if tf32 else "fp32"] = units * 2 / (e0.elapsed_time(e1) / 1e3)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    return out


def run_i3d(args, quick: bool = False):
    import torch
    from video_features_b200.i3d_engine import I3DEngine
    torch.cuda.set_device(0)
    sd, wsrc = _weights("rgb")
    S = int(os.environ.get("VF_BENCH_I3D_STACKS", "32"))
    eng = I3DEngine(sd, "rgb", 0, max_stacks=S, max_T=64)
    g = torch.Generator().manual_seed(1)
    frames_host = torch.randint(0, 256, (S, 65, 224, 224, 3), dtype=torch.uint8, generator=g).pin_memory()
    frames = frames_host.cuda()
    fn = lambda: eng.forward_frames_u8(frames[:, :64])
    W, K = max(args.warmup, 3), max(args.steps, 1)
    if quick:
        W, K = 3, min(K, 8)
    sampler = ClockSampler(0)
    ms = _timed_loop(fn, K, W)
    clocks = sampler.stop()
    pending = []

    def host_fn():      # pinned host stacks in, host features out; H2D of group k+1 overlaps the network on group k, and
        # the first copy of step k+1 overlaps the network of step k (the previous step's features are awaited right
        # after this step is enqueued: two steps in flight, every result on the host inside the timed region)
        pending.append(eng.forward_frames_u8_host(frames_host, 64, group=max(1, S // 2), wait=False))
        while len(pending) > 1:
            pending.pop(0)[1].synchronize()

    for _ in range(2):
        host_fn()
    while pending:
        pending.pop(0)[1].synchronize()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(K):
        host_fn()
    while pending:
        pending.pop(0)[1].synchronize()
    e1.record()
    torch.cuda.synchronize()
    ms_e2e = e0.elapsed_time(e1)
    roof = _gemm_roofline(fn, min(K, 3), I3D_GFLOP["rgb"] * 1e9 * S, ms / K)
    line = {"metric": "stacks/sec I3D rgb (64x224x224)", "value": S * K / (ms / 1e3), "unit": "stacks/s", "n_gpus": 1,
            "steps": K, "warmup": W, "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f16", "data": "synthetic",
            "config": {"workload": "I3D rgb stream, stack_size=64, synthetic 224x224 clips (BASELINE.json configs[2])",
                       "stacks_per_step": S, "frames_per_sec": S * 64 * K / (ms / 1e3), "weights": wsrc,
                       "precision": "fp16 activations, hi+lo fp16 weights (2 MMA passes), fp32 accumulate"},
            "clocks": clocks,
            "e2e": {"value": S * K / (ms_e2e / 1e3), "unit": "stacks/s", "h2d_bytes_per_step": int(frames_host.numel()),
                    "d2h_bytes_per_step": S * 1024 * 4},
            "gpu_launches": int(eng.launch_count), "roofline": roof}
    if not args.no_cpu and not quick:
        from oracle import i3d_net
        cores = usable_cores()
        torch.set_num_threads(cores)
        x = i3d_net.rgb_transform(frames_host[0, :64].permute(0, 3, 1, 2).float())
        i3d_net.forward_features(sd, x[:, :, :16])
        t0 = time.perf_counter(); i3d_net.forward_features(sd, x); dt = time.perf_counter() - t0
        line["cpu_baseline"] = {"value": 1.0 / dt, "unit": "stacks/s", "cores": cores, "kind": "port",
                                "sample": f"1 stack (64x224x224), oracle port of I3D fp32, torch threads={cores}, {cpu_model_name()}"}
    if args.torch_gpu and not quick:
        from oracle import i3d_net
        sdg = {k: v.cuda() for k, v in sd.items()}
        xg = torch.cat([i3d_net.rgb_transform(frames_host[i, :64].permute(0, 3, 1, 2).float()) for i in range(2)]).cuda()
        line["torch_gpu_baseline"] = _torch_gpu_leg(lambda: i3d_net.forward_features(sdg, xg), 2, "stacks/s",
                                                    "oracle port of I3D (torch conv3d / cuDNN, eager), 2 stacks per call")
    eng.close()
    del eng, frames
    torch.cuda.empty_cache()
    return line


def smooth_frames(n: int, h: int, w: int, seed: int, shift=(1.7, -0.9)):
    """Smooth texture translating by a sub-pixel shift per frame (non-degenerate optical flow): (n,h,w,3) uint8."""
    import torch
    import torch.nn.functional as F
    g = torch.Generator().manual_seed(seed)
    base = torch.rand(1, 3, h // 4 + 8, w // 4 + 8, generator=g)
    base = F.interpolate(base, size=(h + 64, w + 64), mode="bicubic", align_corners=False).clamp(0, 1)
    ys, xs = torch.meshgrid(torch.arange(h).float(), torch.arange(w).float(), indexing="ij")
    out = []
    for i in range(n):
        gx = (xs + 32 + shift[0] * i) / (w + 63) * 2 - 1
        gy = (ys + 32 + shift[1] * i) / (h + 63) * 2 - 1
        out.append(F.grid_sample(base, torch.stack([gx, gy], -1)[None], align_corners=True)[0])
    return (torch.stack(out) * 255).round().permute(0, 2, 3, 1).contiguous().to(torch.uint8)


def run_raft(args, rank: int = 0, world: int = 1, local_rank: int = 0, quick: bool = False):
    """BASELINE.json configs[3]: RAFT on 480x270 frame pairs -> I3D flow branch.  world = 2 is the configuration the
    baseline names (2 x B200): stacks are sharded over the ranks (each runs RAFT -> I3D flow on its own 64 pairs, no
    data-path collective) and the (1, 1024) features are all-gathered."""
    import torch
    import torch.distributed as dist
    from video_features_b200.i3d_engine import I3DEngine
    from video_features_b200.raft_engine import RAFTEngine
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1 and not dist.is_initialized():
        dist.init_process_group("nccl", device_id=dev)
    sd, wsrc = _weights("raft")
    sdf, _ = _weights("flow")
    F = 65
    eng = RAFTEngine(sd, local_rank, max_frames=F, max_h=270, max_w=480)
    i3d = I3DEngine(sdf, "flow", local_rank, max_stacks=1, max_T=64)
    frames_host = smooth_frames(F, 270, 480, seed=2 + rank).pin_memory()
    frames = frames_host.to(dev)
    gathered = torch.empty((world, 1024), dtype=torch.float32, device=dev) if world > 1 else None
    def fn():
        flow = eng.flow(frames, iters=20, unpad=False)         # padded, as the I3D path consumes it
        y = i3d.forward_flow(flow[None])
        if world > 1:
            dist.all_gather_into_tensor(gathered, y)
        return y
    W, K = max(args.warmup, 3), max(args.steps, 1)
    if quick:
        W, K = 3, min(K, 4)
    def timed(f, steps, warm):
        for _ in range(warm):
            f()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            f()
        e1.record()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms)
    sampler = ClockSampler(local_rank) if rank == 0 else None
    ms = timed(fn, K, W)
    clocks = sampler.stop() if sampler else None
    ms_raft = timed(lambda: eng.flow(frames, iters=20, unpad=False), K, 1)
    def host_fn():
        flow = eng.flow(frames_host.to(dev, non_blocking=True), iters=20, unpad=False)
        y = i3d.forward_flow(flow[None])
        if world > 1:
            dist.all_gather_into_tensor(gathered, y)
        return y.cpu()
    ms_e2e = timed(host_fn, K, 1)
    roof = _gemm_roofline(lambda: eng.flow(frames, iters=20, unpad=False), min(K, 2), RAFT_GFLOP_272x480 * 1e9 * (F - 1), ms_raft / K)
    line = {"metric": "pairs/sec RAFT 480x270 (20 iters) -> I3D flow", "value": world * (F - 1) * K / (ms / 1e3), "unit": "pairs/s",
            "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f16", "data": "synthetic",
            "config": {"workload": "RAFT optical flow on 480x270 frame pairs -> I3D flow branch (BASELINE.json configs[3])",
                       "pairs_per_step_per_gpu": F - 1, "raft_only_pairs_per_sec": world * (F - 1) * K / (ms_raft / 1e3), "weights": wsrc,
                       "parallelism": f"dp{world}: one 64-pair stack per rank per step, all_gather of the (1,1024) features" if world > 1 else "dp1",
                       "note": "mask head + convex upsample run once (the reference runs them 20x and discards 19)"},
            "clocks": clocks,
            "e2e": {"value": world * (F - 1) * K / (ms_e2e / 1e3), "unit": "pairs/s", "h2d_bytes_per_step": int(frames_host.numel()) * world,
                    "d2h_bytes_per_step": 1024 * 4 * world},
            "gpu_launches": int(eng.launch_count + i3d.launch_count), "roofline": roof}
    if not args.no_cpu and not quick and rank == 0:
        from oracle import raft_net
        cores = usable_cores()
        torch.set_num_threads(cores)
        x = raft_net.pad(frames_host[:3].permute(0, 3, 1, 2).float())
        raft_net.forward(sd, x[:1], x[1:2], 2)
        t0 = time.perf_counter(); raft_net.forward(sd, x[:-1], x[1:], 20); dt = time.perf_counter() - t0
        line["cpu_baseline"] = {"value": 2.0 / dt, "unit": "pairs/s", "cores": cores, "kind": "port",
                                "sample": f"2 pairs 272x480, 20 iterations, oracle port of RAFT fp32, torch threads={cores}, {cpu_model_name()}"}
    if args.torch_gpu and not quick and rank == 0:
        from oracle import raft_net
        sdg = {k: v.cuda() for k, v in sd.items()}
        xg = raft_net.pad(frames_host[:9].permute(0, 3, 1, 2).float()).cuda()
        line["torch_gpu_baseline"] = _torch_gpu_leg(lambda: raft_net.forward(sdg, xg[:-1], xg[1:], 20), 8, "pairs/s",
                                                    "oracle port of RAFT (torch conv2d / cuDNN, eager), 8 pairs per call, 20 iterations")
    eng.close(); i3d.close()
    del eng, i3d, frames
    torch.cuda.empty_cache()
    return line


# ----------------------------------------------------------------------------------------- the video-list product path
def run_b16(args, quick: bool = False):
    """The reference's other ViT-B feature type ('CLIP-ViT-B/16', SURVEY 8 f4): same step as the headline (1000 synthetic
    224x224 uint8 frames), 16-pixel patches -> 197 tokens per frame, 4.4x the FLOPs of ViT-B/32."""
    import torch
    from video_features_b200 import synthetic_weights
    from video_features_b200.clip_engine import ClipEngine
    torch.cuda.set_device(0)
    eng = ClipEngine(synthetic_weights.clip_vit_b16_state_dict(0), device=0)
    n = FRAMES_PER_STEP
    frames_host = synth_frames_host(n, 500).pin_memory()
    frames_host_b = synth_frames_host(n, 501).pin_memory()
    outs = [torch.empty((n, 512), dtype=torch.float32).pin_memory() for _ in range(2)]
    frames = frames_host.cuda()
    W, K = max(args.warmup, 3), max(args.steps, 1)
    if quick:
        W, K = 3, min(K, 10)
    sampler = ClockSampler(0)
    launches0 = eng.launch_count
    ms = _timed_loop(lambda: eng.encode_frames_u8(frames), K, W)
    launches = (eng.launch_count - launches0) // (K + W)
    clocks = sampler.stop()
    pending = []

    def host_fn():                                     # as the headline's e2e: own H2D / D2H every step, two steps in flight
        k = len(pending) and pending[-1][1] == 0
        pending.append((eng.encode_frames_u8_host_async(frames_host_b if k else frames_host, outs[int(k)])[0], int(k)))
        while len(pending) > 1:
            eng.wait(pending.pop(0)[0])
    for _ in range(2):
        host_fn()
    while pending:
        eng.wait(pending.pop(0)[0])
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(K):
        host_fn()
    while pending:
        eng.wait(pending.pop(0)[0])
    e1.record()
    torch.cuda.synchronize()
    ms_e2e = e0.elapsed_time(e1)
    eng.profile(True)
    eng.encode_frames_u8(frames)
    gemm_ms, gemm_launches, gemm_flops = eng.profile_read()
    cats = eng.profile_categories()
    eng.profile(False)
    peaks = load_peaks()
    line = {"metric": "frames/sec CLIP-ViT-B/16 @224px", "value": n * K / (ms / 1e3), "unit": UNIT, "n_gpus": 1, "steps": K,
            "warmup": W, "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f16",
            "data": "synthetic",
            "config": {"workload": "1000 synthetic 224x224x3 uint8 frames per step, CLIP ViT-B/16 tower (197 tokens per frame)",
                       "frames_per_step": n, "weights": "synthetic (seeded, openai initialisation scales)"},
            "clocks": clocks,
            "e2e": {"value": n * K / (ms_e2e / 1e3), "unit": UNIT, "h2d_bytes_per_step": int(frames_host.numel()),
                    "d2h_bytes_per_step": n * 512 * 4},
            "gpu_launches": int(launches),
            "roofline": {"bound": "tensor", "kernel": "vf::gemm_f16_pair_kernel (QKV GEMM + attention_long_kernel: the fused kernel is 50-token only)",
                         "achieved": gemm_flops / (gemm_ms / 1e3) / 1e12 if gemm_ms > 0 else 0.0,
                         "peak": peaks["tflops_sustained"], "unit": "TFLOP/s",
                         "frac": (gemm_flops / (gemm_ms / 1e3) / 1e12 / peaks["tflops_sustained"]) if gemm_ms > 0 else 0.0,
                         "peak_source": peaks["source"] + ", bf16 dense sustained", "traffic": None,
                         "eager_ms_per_step_by_kernel": cats}}
    eng.close()
    torch.cuda.empty_cache()
    return line


def run_c5(args, rank: int, world: int, local_rank: int, quick: bool = False):
    """BASELINE.json configs[4]: a 10k-video list through the product's own list path -- ExtractCLIP.forward (decode
    pool -> pinned staging -> one engine call per 1024 frames -> per-video feature blocks) under the --device_ids
    dispatch (`dispatch.run_shard`: the rank's torch.chunk of the list, then ONE NCCL all-gather of every video's
    (12,512) block).  Decode is stubbed: list entry i maps to a deterministic synthetic 12-frame 224x224 clip, a function
    of i alone; the sink is the all-gather (nothing is written to disk).  Timed with CUDA events around the whole shard
    (they bracket the host work too), max over ranks."""
    import argparse as ap
    import numpy as np
    import torch
    import torch.distributed as dist
    from tqdm import tqdm
    from video_features_b200 import dispatch
    from video_features_b200.extract.extract_clip import ExtractCLIP
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1 and not dist.is_initialized():
        dist.init_process_group("nccl", device_id=dev)
    n_videos = int(os.environ.get("VF_BENCH_C5_VIDEOS", "10000"))
    per = 12
    pool_n = 64
    pool = np.random.default_rng(77).integers(0, 256, (pool_n, per, 224, 224, 3), dtype=np.uint8)

    class SynthStream:                                     # the two-step source interface of utils.FrameStream
        def __init__(self, path, method):
            self.clip = pool[int(path.rsplit("/", 1)[1]) % pool_n]
            self.count, self.hw, self.fps, self.timestamps_ms = per, (224, 224), 25.0, [0.0] * per

        def read_into(self, dst):                          # "decode": the clip's pixels land in the staging rows
            np.copyto(dst, self.clip)
            return per

    os.environ["VF_CLIP_SYNTHETIC"] = "0"
    ns = ap.Namespace(feature_type="CLIP-ViT-B/32", video_paths=[os.path.abspath(__file__)], flow_paths=None,
                      file_with_video_paths=None, video_dir=None, flow_dir=None, extraction_fps=None,
                      extract_method=f"uni_{per}", on_extraction="print", output_path="./output", output_direct=True,
                      tmp_path="./tmp")
    ex = ExtractCLIP(ns, external_call=True)
    ex.progress.close()
    ex.progress = tqdm(total=0, disable=True)
    ex.frame_stream = SynthStream
    ex.path_list = [f"synthetic://{i}" for i in range(n_videos)]
    # warm-up: engine creation, graph capture for the chunk sizes in use, pinned buffers, thread pools
    # (through the same run_shard, so the communicator has carried an all-gather of this kind before the timed pass)
    # twice: a tower chunk size is captured into a CUDA graph the second time it is seen
    for _ in range(2):
        warm = dispatch.run_shard(ex, min(n_videos, world * 3 * 86), rank, world, dev, gather_key="CLIP-ViT-B/32")
        del warm
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    trace = {} if os.environ.get("VF_C5_TRACE") == "1" else None     # host timeline of the shard (diagnostics)
    if trace is not None:
        inner_gather, inner_forward = dispatch.gather_feature_blocks, ExtractCLIP.forward

        def traced_gather(*a_, **k_):
            torch.cuda.synchronize()
            a = time.perf_counter()
            r = inner_gather(*a_, **k_)
            torch.cuda.synchronize()
            trace["gather"] = (a, time.perf_counter())
            return r

        def traced_forward(self, indices):
            a = time.perf_counter()
            r = inner_forward(self, indices)
            trace["forward"] = (a, time.perf_counter())
            return r
        dispatch.gather_feature_blocks = traced_gather
        ExtractCLIP.forward = traced_forward
        # device timeline of the engine calls: an event pair on the calling stream around every asynchronous call (the
        # stream waits for the call's tower, so consecutive end events are one call apart on the device)
        eng0 = ex._engines[local_rank]
        inner_async = eng0.encode_frames_u8_host_async
        trace["calls"] = []

        def traced_async(frames, out_host=None, out_dev=False):
            torch.cuda.set_device(local_rank)          # the engine thread's own current device (per-thread state)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            r = inner_async(frames, out_host, out_dev)
            b.record()
            trace["calls"].append((a, b, int(frames.shape[0])))
            return r
        eng0.encode_frames_u8_host_async = traced_async
    t0 = time.perf_counter()
    e0.record()
    blocks = dispatch.run_shard(ex, n_videos, rank, world, dev, gather_key="CLIP-ViT-B/32")
    e1.record()
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    if trace:
        dispatch.gather_feature_blocks, ExtractCLIP.forward = inner_gather, inner_forward
        f, g = trace.get("forward", (t0, t0)), trace.get("gather", (t0, t0))
        calls = trace.get("calls", [])
        if len(calls) > 2:
            gaps_ms = [calls[i][1].elapsed_time(calls[i + 1][1]) for i in range(len(calls) - 1)]   # spacing of call ends
            own = [a.elapsed_time(b) for a, b, _ in calls]
            print(f"[c5 trace rank {rank}] {len(calls)} engine calls of {calls[0][2]} frames: spacing of call ends median "
                  f"{sorted(gaps_ms)[len(gaps_ms) // 2]:.2f} ms (min {min(gaps_ms):.2f}, max {max(gaps_ms):.2f}); start->end on the calling stream "
                  f"median {sorted(own)[len(own) // 2]:.2f} ms; first end at {e0.elapsed_time(calls[0][1]):.1f} ms, last end at "
                  f"{e0.elapsed_time(calls[-1][1]):.1f} ms", file=sys.stderr, flush=True)
        print(f"[c5 trace rank {rank}] wall {wall:.3f} s: before forward {f[0] - t0:.3f}, forward {f[1] - f[0]:.3f}, "
              f"forward -> gather {g[0] - f[1]:.3f}, gather {g[1] - g[0]:.3f}, after {t0 + wall - g[1]:.3f}; stage waits "
              f"{ {k: round(v, 3) for k, v in ex.stage_wait.items()} }", file=sys.stderr, flush=True)
    clocks = sampler.stop() if sampler else None
    ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms = float(ms)
    # every rank holds every video's block, in list order: entries i and i + 64 are the same clip
    if len(blocks) != n_videos or not all(tuple(b.shape) == (per, 512) for b in blocks[:: max(1, n_videos // 50)]):
        raise AssertionError(f"list path returned {len(blocks)} blocks for {n_videos} videos; shapes "
                             f"{sorted({tuple(b.shape) for b in blocks})[:4]}")
    for i in (0, 1, pool_n - 1, n_videos // 2, n_videos - pool_n - 1):
        if 0 <= i and i + pool_n < n_videos:
            assert torch.equal(blocks[i], blocks[i + pool_n]), f"gathered block {i} != block {i + pool_n}"
    engine = ex._engines[local_rank]
    line = {"metric": "frames/sec CLIP-ViT-B/32 @224px, 10k-video list", "value": n_videos * per / (ms / 1e3), "unit": UNIT,
            "videos_per_sec": n_videos / (ms / 1e3), "n_gpus": world, "steps": 1, "warmup": 1, "ms_per_step": ms,
            "host_wall_s_rank0": wall, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f16",
            "data": "synthetic",
            "config": {"workload": "10k-video synthetic list, CLIP-ViT-B/32, sharded across --device_ids (BASELINE.json configs[4])",
                       "videos": n_videos, "frames_per_video": per, "frames_per_engine_call": ex.batch_frames,
                       "decode": "stubbed (clip = f(list index)); staging copy into pinned memory, H2D, tower, D2H, per-video "
                                 "blocks and the final all-gather are inside the timed region",
                       "host_threads_per_rank": ex.decode_workers, "host_cores_usable": usable_cores(),
                       "parallelism": f"dp{world}: torch.chunk of the list per rank + one all_gather of the feature blocks"},
            "clocks": clocks,
            "e2e": {"value": n_videos * per / (ms / 1e3), "unit": UNIT, "h2d_bytes_per_step": n_videos * per * 150528,
                    "d2h_bytes_per_step": n_videos * per * 2048,
                    "api": "ExtractCLIP.forward under dispatch.run_shard (main.py --device_ids path)",
                    "note": "this workload is host-to-host by construction (frames start in host memory, feature blocks end in "
                            "the gathered list): `value` and `e2e` are the same measurement, not a device-resident number repeated"},
            "gpu_launches": int(engine.launch_count)}
    for e in ex._engines.values():
        e.close()
    ex._engines.clear()
    del blocks
    torch.cuda.empty_cache()
    return line


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="engine", choices=["engine", "reference"])
    ap.add_argument("--chunk", type=int, default=0, help="frames per tower chunk (0 = library default)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--torch-gpu", action="store_true", dest="torch_gpu",
                    help="also time the oracle's fp32 torch modules on the same GPU (library-call bar), key torch_gpu_baseline")
    ap.add_argument("--workload", default="clip", choices=["clip", "i3d", "raft", "c5", "b16"],
                    help="clip = the headline (BASELINE.json configs[1], with the other configs as `secondary`); i3d / raft "
                         "/ c5 = configs[2] / configs[3] / configs[4] alone")
    ap.add_argument("--no-secondary", action="store_true", dest="no_secondary",
                    help="headline only: skip the secondary workloads (c5 video list, I3D, RAFT -> I3D flow)")
    ap.add_argument("--dump-outputs", metavar="DIR", dest="dump_outputs",
                    help="write the timed path's outputs of its last timed step to DIR/<name>.npy (clip workload)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.workload != "clip":
        ap.error("--dump-outputs writes the headline path's outputs: use it with --workload clip")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    if world != args.gpus and world == 1 and args.gpus > 1:
        # launched without torchrun: re-exec under torch.distributed.run on this node
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", os.environ.get("MASTER_PORT", "29541"),
               os.path.abspath(__file__)] + sys.argv[1:]
        raise SystemExit(subprocess.call(cmd, stdout=_REAL_STDOUT))     # the ranks inherit the REAL stdout for the JSON line
    if args.workload == "clip":
        return run_engine(args, rank, world, local_rank)
    line = {"i3d": lambda: run_i3d(args), "raft": lambda: run_raft(args, rank, world, local_rank),
            "c5": lambda: run_c5(args, rank, world, local_rank), "b16": lambda: run_b16(args)}[args.workload]()
    if rank == 0:
        emit(line)
    try:
        import torch.distributed as dist
        if dist.is_initialized():
            dist.destroy_process_group()
    except Exception:
        pass


if __name__ == "__main__":
    main()
