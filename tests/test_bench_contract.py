"""The CPU-runnable part of bench.py's contract: `--impl reference` (the CPU port of the reference step, rank 0 only)
prints ONE JSON line with the keys the driver reads, for the metric / unit / workload of the GPU arm."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT


def test_reference_arm_prints_the_contract_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                        "--size", "64"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "our_unet_512_train_images_per_sec" and d["unit"] == "img/s"
    for k in ("value", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype",
              "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["value"] > 0 and d["higher_is_better"] is True and d["vs_baseline"] is None and d["data"] == "synthetic"
    assert "workload" in d["config"] and "model" not in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "sample" in cb
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_other_ranks_of_the_reference_arm_exit_quietly():
    env = dict(os.environ, RANK="1", LOCAL_RANK="1", WORLD_SIZE="2")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
                        "--size", "64"], capture_output=True, text=True, timeout=300, cwd=ROOT, env=env)
    assert r.returncode == 0 and not [ln for ln in r.stdout.splitlines() if ln.startswith("{")]


@pytest.mark.gpu
def test_dump_outputs_are_the_same_from_run_to_run(tmp_path):
    """--dump-outputs writes the loss, model output and every parameter gradient of the last timed step as float32
    .npy files, at most 64 MB in all, and two runs with the same arguments write the same arrays."""
    dumps = []
    for run in ("a", "b"):
        d = tmp_path / run
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "3", "--warmup", "1", "--batch", "2",
                            "--size", "64", "--no-cpu-baseline", "--no-profile", "--no-e2e", "--dump-outputs", str(d)],
                           capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert r.returncode == 0, r.stderr[-2000:]
        assert len([ln for ln in r.stdout.splitlines() if ln.startswith("{")]) == 1
        dumps.append({f: np.load(d / f) for f in sorted(os.listdir(d))})
    a, b = dumps
    assert len(a) == 2 + 90 and a["loss.npy"].shape == () and a["output.npy"].shape == (2, 3, 64, 64)
    assert sum(v.nbytes for v in a.values()) <= 64 << 20
    assert a.keys() == b.keys()
    for k in a:
        assert a[k].dtype == np.float32 and np.isfinite(a[k]).all(), k
        assert np.array_equal(a[k], b[k]), k
