"""bench.py's CUDA arm end to end at a small scene count: one JSON line on stdout, and the outputs of the last timed step written by
--dump-outputs for the inference, fine-tune and stage-1 paths — for inference the same on every run with the same inputs."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(dump, *args):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--warmup", "1", "--dump-outputs", str(dump), *args],
                       capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-3000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, r.stdout[-3000:]
    return json.loads(lines[0])


def test_bench_dumps_the_outputs_of_its_last_timed_inference_step(tmp_path):
    for steps in (2, 3):
        line = _bench(tmp_path / str(steps), "--steps", str(steps), "--scenes", "64", "--no-secondary", "--no-cpu-baseline")
        assert line["steps"] == steps and line["value"] > 0
        d = {n: np.load(tmp_path / str(steps) / f"{n}.npy") for n in ("decoded", "metrics", "per_scene", "sum_ade", "ade")}
        assert d["decoded"].shape == (64, 2, 25) and d["decoded"].dtype == np.float32 and np.isfinite(d["decoded"]).all()
        assert d["per_scene"].shape == (64, 2) and d["metrics"].shape == (8,) and np.array_equal(d["ade"], d["per_scene"][:, 0])
        assert abs(float(d["sum_ade"]) / 64 - line["config"]["ade_px"]) <= 1e-3 * max(1.0, line["config"]["ade_px"])
    # inference is stateless and the inputs are seeded: the outputs agree whatever the number of steps
    for n in ("decoded", "per_scene", "metrics"):
        np.testing.assert_allclose(np.load(tmp_path / "2" / f"{n}.npy"), np.load(tmp_path / "3" / f"{n}.npy"), rtol=1e-3, atol=1e-3)


@pytest.mark.parametrize("mode", ["train", "stage1"])
def test_bench_dumps_the_loss_of_its_last_timed_training_step(tmp_path, mode):
    line = _bench(tmp_path, "--mode", mode, "--steps", "2", "--scenes", "8")
    loss = np.load(tmp_path / "loss.npy")
    assert loss.shape == () and loss.dtype == np.float32 and np.isfinite(loss)
    assert abs(float(loss) - line["config"]["loss_first_last"][1]) <= 1e-3 * max(1.0, abs(float(loss)))
    if mode == "train":
        dec = np.load(tmp_path / "decoded.npy")
        assert dec.shape == (8, 2, 25) and dec.dtype == np.float32 and np.isfinite(dec).all()
    else:
        assert sorted(os.listdir(tmp_path)) == ["loss.npy"]
