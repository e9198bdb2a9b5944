"""bench.py contract checks that need no GPU: the reference arm (the oracle port of the reference's --cpu flow) prints ONE
JSON line with the keys the driver reads, and rank != 0 leaves without work under a multi-rank launch."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(env_extra=None, extra_args=()):
    env = dict(os.environ, **(env_extra or {}))
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                        *extra_args],
                       capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-2000:]
    return [l for l in p.stdout.splitlines() if l.strip()]


def test_reference_arm_prints_one_contract_line():
    lines = _run()
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "frames/sec CLIP-ViT-B/32 @224px" and d["unit"] == "frames/s"
    assert d["higher_is_better"] is True and d["n_gpus"] == 1 and d["steps"] == 1 and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"]


def test_reference_arm_other_ranks_exit_without_work():
    lines = _run({"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"})
    assert lines == []


def test_reference_arm_dumps_the_last_step(tmp_path):
    """--dump-outputs DIR: the features the timed path computed, float32, one row per frame of its fixed sample -- the
    first 32 of the headline step's seeded frames (rank 0) -- equal to the oracle port run on those frames."""
    import numpy as np
    import torch
    from oracle import clip_preprocess, clip_tower
    from video_features_b200 import synthetic_weights
    _run(extra_args=("--dump-outputs", str(tmp_path)))
    y = np.load(tmp_path / "features.npy")
    assert y.dtype == np.float32 and y.shape == (32, 512)
    frames = torch.randint(0, 256, (1000, 224, 224, 3), dtype=torch.uint8, generator=torch.Generator().manual_seed(100))
    with torch.no_grad():
        ref = clip_tower.encode_image(synthetic_weights.clip_vit_b32_state_dict(0),
                                      clip_preprocess.preprocess_batch(frames[:32].numpy())).numpy()
    assert np.linalg.norm(y - ref) <= 1e-5 * np.linalg.norm(ref)


def test_steps_below_one_are_rejected():
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True, text=True,
                       timeout=600, cwd=ROOT)
    assert p.returncode != 0 and "--steps" in p.stderr


def test_engine_arm_fails_loudly_without_a_gpu():
    """No CPU fallback: on a machine without a CUDA device the engine arm exits non-zero with a clear message and prints
    no JSON line (a number must never come from a silent fallback)."""
    import torch
    if torch.cuda.is_available():
        import pytest
        pytest.skip("this check is for GPU-less machines")
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "3", "--no-cpu", "--no-secondary"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert p.returncode != 0
    assert "no CUDA device" in (p.stderr + p.stdout)
    assert not [l for l in p.stdout.splitlines() if l.startswith("{")]
