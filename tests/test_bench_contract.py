"""bench.py's command line.  The reference arm (`--impl reference`) needs no GPU: one JSON line with the agreed keys on
rank 0, nothing (exit 0) on the other ranks.  `--dump-outputs` writes a bounded, fixed sample of what the last timed
step computed; its GPU test runs the engine arm at a small workload."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(extra_env, *args):
    env = dict(os.environ, **extra_env)
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], env=env, capture_output=True,
                          text=True, timeout=600)


def test_reference_arm_prints_one_contract_line():
    r = _run({"RANK": "0", "WORLD_SIZE": "1"}, "--impl", "reference", "--workload", "det5", "--steps", "1",
             "--warmup", "1")
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "DeformConv2d fwd+bwd images/sec" and d["unit"] == "images/s"
    for key in ("value", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
                "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in d, key
    assert d["value"] > 0 and d["higher_is_better"] is True and d["vs_baseline"] is None and d["data"] == "synthetic"
    assert d["config"]["workload"].startswith("det5")
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    e = d["e2e"]
    assert e["value"] == d["value"] and e["unit"] == d["unit"]
    assert e["h2d_bytes_per_step"] == 0 and e["d2h_bytes_per_step"] == 0


def test_reference_arm_is_silent_on_other_ranks():
    r = _run({"RANK": "1", "WORLD_SIZE": "2"}, "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "1")
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_steps_below_one_are_refused():
    r = _run({}, "--impl", "reference", "--steps", "0")
    assert r.returncode != 0 and "--steps" in r.stderr


def test_dump_outputs_stores_a_fixed_sample_within_the_budget(tmp_path):
    import torch
    import bench
    g = torch.Generator().manual_seed(0)
    arrays = {"out": torch.randn(8, 1000, 1000, generator=g), "grad_bias": torch.randn(64, generator=g).bfloat16()}
    share = (bench.DUMP_BUDGET_BYTES // 2 - 256) // 4
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), arrays)
    files = {f: np.load(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")}
    assert sorted(files) == ["grad_bias.npy", "out.npy"]
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= bench.DUMP_BUDGET_BYTES
    assert all(v.dtype == np.float32 for v in files.values())
    # small arrays whole, in their shape; large ones as the documented sample of the flattened array
    assert np.array_equal(files["grad_bias.npy"], arrays["grad_bias"].float().numpy())
    idx = np.sort(np.random.default_rng(0).choice(8_000_000, share, replace=False))
    assert np.array_equal(files["out.npy"], arrays["out"].reshape(-1).numpy()[idx])
    for f in files:
        assert np.array_equal(files[f], np.load(tmp_path / "b" / f))


@pytest.mark.gpu
def test_engine_arm_dumps_the_last_step(tmp_path):
    r = _run({}, "--workload", "det5", "--steps", "2", "--warmup", "1", "--no-cpu-baseline", "--no-e2e",
             "--dump-outputs", str(tmp_path))
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads(r.stdout.strip().splitlines()[-1])
    assert d["steps"] == 2
    files = {f[:-4]: np.load(tmp_path / f) for f in os.listdir(tmp_path)}
    assert sorted(files) == ["grad_bias", "grad_offset", "grad_weight", "grad_x", "out"]
    assert all(v.dtype == np.float32 and np.isfinite(v).all() for v in files.values())
    # det5: O = 256, C = 128, 3 x 3; out [1024, 256, 8, 8] is sampled
    assert files["grad_bias"].shape == (256,) and files["grad_weight"].shape == (256, 128, 3, 3)
    assert files["out"].ndim == 1 and np.abs(files["out"]).max() > 0
