"""bench.py's output contract.  On the CPU, through the reference arm (the only arm that runs without a GPU): exactly
one JSON line on stdout with the keys its readers use; ranks other than 0 stay silent.  --dump-outputs: the format and
row sample on the CPU, the CUDA arm's arrays on the GPU."""
import importlib.util
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(env_extra):
    env = dict(os.environ, **env_extra)
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "1", "--steps", "1",
                           "--warmup", "1"], capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)


def test_reference_arm_prints_one_json_line_with_the_contract_keys():
    res = _run({})
    assert res.returncode == 0, res.stderr[-2000:]
    lines = [l for l in res.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, res.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "learned-dynamics env-steps/sec" and d["unit"] == "env-steps/s"
    assert d["higher_is_better"] is True and d["scaling"] == "weak" and d["n_gpus"] == 1 and d["warmup"] >= 3
    assert d["value"] > 0 and d["vs_baseline"] is None and d["data"] == "synthetic"
    assert "workload" in d["config"] and "model" not in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("port", "reference") and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_is_silent_on_other_ranks():
    res = _run({"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"})
    assert res.returncode == 0 and res.stdout.strip() == ""


def _bench_module():
    spec = importlib.util.spec_from_file_location("bench", os.path.join(ROOT, "bench.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_dump_outputs_keeps_a_fixed_row_sample_under_the_limit(tmp_path):
    bench = _bench_module()
    E = 5000
    g = torch.Generator().manual_seed(4)
    per_env = {"next_state": torch.randn(E, 226, generator=g),
               "done": (torch.rand(E, generator=g) < 0.1).to(torch.uint8),
               "num_steps": torch.randint(0, 300, (E,), generator=g, dtype=torch.int32)}
    limit = 1 << 20   # about a fifth of what these arrays take
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), per_env, {"disc_quantile": 0.25}, limit=limit)
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == ["disc_quantile.npy", "done.npy", "next_state.npy", "num_steps.npy", "rows.npy"]
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= limit
    rows = np.load(tmp_path / "a" / "rows.npy").astype(np.int64)
    assert rows.size > 1000 and np.all(np.diff(rows) > 0) and rows[-1] < E
    for f in files:
        a, b = np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)
        assert a.dtype in (np.float32, np.float64) and np.array_equal(a, b), f
    np.testing.assert_array_equal(np.load(tmp_path / "a" / "next_state.npy"), per_env["next_state"].numpy()[rows])
    np.testing.assert_array_equal(np.load(tmp_path / "a" / "num_steps.npy"), per_env["num_steps"].numpy()[rows])
    assert float(np.load(tmp_path / "a" / "disc_quantile.npy")[0]) == 0.25
    bench.dump_outputs(str(tmp_path / "c"), per_env)   # under the default 64 MB: every row, no index file
    assert sorted(os.listdir(tmp_path / "c")) == ["done.npy", "next_state.npy", "num_steps.npy"]
    np.testing.assert_array_equal(np.load(tmp_path / "c" / "next_state.npy"), per_env["next_state"].numpy())
    np.testing.assert_array_equal(np.load(tmp_path / "c" / "done.npy"), per_env["done"].numpy())


def test_dump_outputs_is_refused_for_the_reference_arm(tmp_path):
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--dump-outputs",
                          str(tmp_path / "d")], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert res.returncode == 2 and "--dump-outputs" in res.stderr and not os.path.exists(tmp_path / "d")


@pytest.mark.gpu
def test_cuda_arm_times_the_steps_asked_for_and_dumps_its_last_step(tmp_path):
    """--steps is the number of timed steps for every workload, the long-step configs included.  The dump is the last
    timed step's: every env's counter has counted warmup + steps calls, the ring-buffered cost and disc agree with that
    step's single-buffer ipm and bonus (cost = ipm - bonus, bonus = lambda_b * c_min * min(disc / threshold, 1)), and
    disc_quantile is the 0.9 quantile of the dumped disc.  Two runs with the same arguments dump identical arrays."""
    warmup, steps, lambda_b, c_min = 3, 500, 0.0025, -1.0
    lines = []
    for d in ("a", "b"):
        res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--config", "4", "--envs", "4096",
                              "--steps", str(steps), "--warmup", str(warmup), "--skip-cpu-baseline", "--skip-sustained",
                              "--skip-extras", "--dump-outputs", str(tmp_path / d)],
                             capture_output=True, text=True, timeout=900, cwd=ROOT)
        assert res.returncode == 0, res.stderr[-3000:]
        lines.append(json.loads(res.stdout.strip().splitlines()[-1]))
    assert [l["steps"] for l in lines] == [steps, steps] and lines[0]["config"]["envs_per_gpu"] == 4096
    names = sorted(os.listdir(tmp_path / "a"))
    assert names == sorted(f"{n}.npy" for n in ("next_state", "disc", "done", "cost", "ipm", "bonus", "num_steps",
                                                 "imitation_reward", "disc_quantile"))
    for n in names:
        a, b = np.load(tmp_path / "a" / n), np.load(tmp_path / "b" / n)
        assert a.dtype in (np.float32, np.float64) and np.array_equal(a, b, equal_nan=True), n
    out = {n[:-4]: np.load(tmp_path / "a" / n) for n in names}
    assert out["next_state"].shape == (4096, 226) and np.all(out["num_steps"] == warmup + steps)
    ipm, bonus, disc = out["ipm"], out["bonus"], out["disc"]
    assert np.abs(out["cost"] - (ipm - bonus)).max() <= 1e-6 * np.abs(ipm).max()
    thr = np.float32(lines[0]["config"]["threshold"])
    assert (disc < thr).mean() > 0.5   # the bonus follows disc rather than sitting at its cap
    want = np.float32(lambda_b) * (np.minimum(disc / thr, np.float32(1.0)) * np.float32(c_min))
    np.testing.assert_allclose(bonus, want, rtol=1e-6, atol=0)
    q = np.quantile(disc.astype(np.float64), 0.9)
    assert abs(float(out["disc_quantile"][0]) - q) <= 1e-5 * max(abs(q), float(disc.max() - disc.min()))
