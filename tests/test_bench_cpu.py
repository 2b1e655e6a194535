"""bench.py contract checks that need no GPU: the reference arm prints ONE JSON line with the keys the driver reads, and the CUDA arm
fails loudly (non-zero exit, nothing on stdout) when there is no device instead of falling back to a CPU path."""
import json
import os
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*args, env=None):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, timeout=600,
                          env=dict(os.environ, **(env or {})), cwd=ROOT)


def test_reference_arm_prints_one_json_line_with_the_contract_keys():
    r = _run("--impl", "reference", "--steps", "1", "--warmup", "0", "--cpu-sample", "2")
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, r.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "scenes/s" and d["higher_is_better"] is True and d["n_gpus"] == 1
    assert d["value"] > 0 and d["steps"] == 1 and d["vs_baseline"] is None and d["gpu_launches"] == 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "scenes/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "model" not in d["config"]


def test_reference_arm_is_rank0_only_under_torchrun():
    r = _run("--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0", "--cpu-sample", "2", env={"RANK": "1", "WORLD_SIZE": "2"})
    assert r.returncode == 0 and r.stdout.strip() == "", (r.stdout, r.stderr[-1000:])


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-device failure mode")
def test_cuda_arm_fails_loudly_without_a_device():
    r = _run("--steps", "1")
    assert r.returncode != 0
    assert not any(l.lstrip().startswith("{") for l in r.stdout.splitlines()), "no bench line may be printed without a GPU"



def test_dump_outputs_is_rejected_on_the_reference_arm(tmp_path):
    r = _run("--impl", "reference", "--steps", "1", "--warmup", "0", "--cpu-sample", "2", "--dump-outputs", str(tmp_path / "d"))
    assert r.returncode != 0 and "--dump-outputs" in r.stderr and r.stdout.strip() == ""
    assert not (tmp_path / "d").exists()


def test_dump_outputs_writes_float_arrays_and_samples_scenes_above_64_mb(tmp_path):
    import numpy as np
    import bench
    small = {"decoded": torch.randn(5, 2, 7).to(torch.bfloat16), "metrics": torch.arange(8, dtype=torch.float64), "loss": torch.tensor(3.5)}
    bench.dump_outputs(str(tmp_path / "small"), small, 5)
    for k, v in small.items():
        a = np.load(tmp_path / "small" / f"{k}.npy")
        assert a.dtype == (np.float64 if v.dtype == torch.float64 else np.float32) and a.shape == tuple(v.shape), k
        assert np.array_equal(a, v.double().numpy()), k
    # 80 MB of per-scene rows numbered by their scene: one seeded sample of scenes, the same in every per-scene array and on every
    # call, 64 MB at most in all; arrays that are not per scene (metrics, here also of leading length > 1) stay whole
    scenes = 163840
    big = {"decoded": torch.arange(scenes, dtype=torch.float32)[:, None].repeat(1, 128),
           "per_scene": torch.arange(scenes, dtype=torch.float32)[:, None].repeat(1, 2),
           "metrics": torch.arange(8, dtype=torch.float32), "loss": torch.tensor(1.0)}
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), big, scenes)
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == ["decoded.npy", "loss.npy", "metrics.npy", "per_scene.npy"]
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= bench.DUMP_LIMIT_BYTES
    dec, per = np.load(tmp_path / "a" / "decoded.npy"), np.load(tmp_path / "a" / "per_scene.npy")
    assert 0.5 * scenes < dec.shape[0] < scenes and dec.shape[1] == 128
    assert (dec == dec[:, :1]).all() and np.array_equal(dec[:, 0], per[:, 0]) and (np.diff(dec[:, 0]) > 0).all()
    assert np.array_equal(np.load(tmp_path / "a" / "metrics.npy"), np.arange(8, dtype=np.float32))
    for f in files:
        assert np.array_equal(np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)), f
