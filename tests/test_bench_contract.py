"""bench.py's reference arm (`--impl reference`: the reference's own CPU pipeline -- the unmodified classes when a copy
of the reference is present, else the oracle port -- timed for whole epochs on the host cores) prints ONE JSON line
with the contract's keys.  CPU-only; a reduced env count keeps it at a few seconds."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "1",
                        "--envs-per-gpu", "64", "--cpu-procs", "4"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, r.stdout[-2000:]
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "env_steps_per_sec" and d["unit"] == "env-steps/s"
    assert d["higher_is_better"] is True and d["scaling"] == "weak" and d["data"] == "synthetic"
    assert d["n_gpus"] == 1 and d["steps"] == 2 and d["warmup"] == 1 and d["vs_baseline"] is None
    assert d["value"] > 0 and d["ms_per_step"] > 0
    assert "64 envs/GPU" in d["config"]["workload"] and "horizon 128" in d["config"]["workload"]
    cb = d["cpu_baseline"]
    from oracle import reference_loader
    assert cb["kind"] == ("reference" if reference_loader.available() else "port")
    assert cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    # every step is a whole epoch timed for real: the per-epoch times add up to steps * ms_per_step
    assert len(cb["detail"]["epoch_s"]) == 2
    assert abs(sum(cb["detail"]["epoch_s"]) * 1e3 - d["steps"] * d["ms_per_step"]) < 1e-6 * d["ms_per_step"] + 1e-3
    e2e = d["e2e"]
    assert e2e["value"] == d["value"] and e2e["h2d_bytes_per_step"] == 0 and e2e["d2h_bytes_per_step"] == 0


@pytest.mark.gpu
def test_dump_outputs_of_the_last_timed_step(tmp_path):
    """`--dump-outputs DIR`: float32 / float64 .npy files of the last timed epoch (rollout, advantages, returns,
    parameters, logged scalars), 64 MB at most; `--steps` sets the number of timed steps."""
    import numpy as np
    out = tmp_path / "dump"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1", "--envs-per-gpu",
                        "256", "--skip-cpu-baseline", "--skip-roofline", "--skip-secondary", "--dump-outputs", str(out)],
                       capture_output=True, text=True, timeout=900, cwd=str(tmp_path))
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, r.stdout[-2000:]
    d = json.loads(lines[0])
    assert d["steps"] == 2 and len(d["step_ms"]) == 2 and len(d["e2e_step_ms"]) == 2
    files = {f[:-4]: np.load(out / f) for f in os.listdir(out)}
    assert all(f.endswith(".npy") for f in os.listdir(out))
    assert sum(os.path.getsize(out / f) for f in os.listdir(out)) <= 64 << 20
    for name in ("obs", "next_obs", "acts", "rewards", "values", "advs", "estimate_returns", "params",
                 "obs_norm_mean", "env_sample"):
        assert name in files, sorted(files)
    assert any(n.startswith("info_") for n in files)
    for name, a in files.items():
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        assert np.isfinite(a).all(), name
    assert files["obs"].shape == (128, 256, 17) and files["advs"].shape[:2] == (128, 256)
    assert np.abs(files["advs"]).max() > 0 and np.abs(files["params"]).max() > 0
