"""bench.py contract (CPU part): the reference arm runs without a GPU and prints ONE JSON line with the keys
the driver reads; non-zero ranks of a torchrun launch of that arm exit silently."""
import json
import os
import subprocess
import sys

import pytest

from conftest import ROOT


def _run(extra_env=None, *args):
    env = dict(os.environ)
    env.update(extra_env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gib", "0.03",
                           "--steps", "2", "--warmup", "1", *args], capture_output=True, text=True, env=env, timeout=300)


def test_reference_arm_prints_one_contract_line():
    r = _run()
    assert r.returncode == 0, r.stderr
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "GB/s" and d["higher_is_better"] is True
    assert d["steps"] == 2 and d["warmup"] == 1 and d["n_gpus"] == 1 and d["value"] > 0
    assert d["dtype"] == "u8" and d["data"] == "synthetic" and d["vs_baseline"] is None and d["scaling"] == "weak"
    assert "workload" in d["config"] and 1.5 < d["config"]["ratio"] < 1.75
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["gpu_launches"] == 0


def test_reference_arm_other_ranks_stay_silent():
    r = _run({"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"}, "--gpus", "2")
    assert r.returncode == 0 and r.stdout.strip() == ""


def _check_dump(d, oracle, n_blocks):
    """--dump-outputs: float arrays under 64 MB in all, holding the decoded input of the sampled blocks"""
    import numpy as np
    files = {f: np.load(os.path.join(d, f)) for f in os.listdir(d)}
    assert set(files) == {"decoded_blocks.npy", "decoded_block_ids.npy", "decoded_sizes.npy"}
    assert all(a.dtype in (np.float32, np.float64) for a in files.values())
    assert sum(os.path.getsize(os.path.join(d, f)) for f in files) <= 64 << 20
    ids = files["decoded_block_ids.npy"].astype(np.int64)
    blocks = files["decoded_blocks.npy"]
    assert blocks.shape == (len(ids), 65536) and len(set(ids.tolist())) == len(ids) and ids.max() < n_blocks
    src = oracle.datagen_mt(n_blocks * 65536, 64 << 20, 0.5, 0).reshape(n_blocks, 65536)
    assert (blocks == src[ids]).all()
    assert (files["decoded_sizes.npy"] == 65536).all() and len(files["decoded_sizes.npy"]) == n_blocks


def test_reference_arm_dumps_outputs(tmp_path, oracle):
    r = _run(None, "--dump-outputs", str(tmp_path / "a"))
    assert r.returncode == 0, r.stderr
    _check_dump(str(tmp_path / "a"), oracle, int(0.03 * (1 << 30)) // 65536)


@pytest.mark.gpu
def test_gpu_arm_dumps_outputs_and_runs_the_steps_asked(tmp_path, oracle):
    launches = []
    for steps, name in ((1, "a"), (3, "b")):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gib", "0.0625", "--steps", str(steps),
                            "--warmup", "1", "--no-e2e", "--no-cpu", "--dump-outputs", str(tmp_path / name)],
                           capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr
        d = json.loads([l for l in r.stdout.splitlines() if l.strip()][-1])
        assert d["steps"] == steps and d["gpu_launches"] > 0
        launches.append(d["gpu_launches"])
        _check_dump(str(tmp_path / name), oracle, 1024)
    assert launches[1] == 3 * launches[0]                # the launches of the timed region scale with --steps
