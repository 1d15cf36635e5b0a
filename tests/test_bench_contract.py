"""bench.py --impl reference (the CPU arm run next to the GPU arm): one JSON line with the contract's keys; the
outputs --dump-outputs writes."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DUMPED = ("obs", "rew4", "covered", "env_index")


def test_reference_arm_prints_the_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "1",
                          "--cpu-seconds", "0.5", "--workload", "default4096"], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    line = [l for l in out.stdout.splitlines() if l.startswith("{")][-1]
    d = json.loads(line)
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e", "gpu_launches"):
        assert k in d, k
    assert d["impl"] == "reference" and d["metric"] == "agent-steps/s" and d["value"] > 0 and d["steps"] == 2
    assert d["config"]["workload"] == "default4096" and d["gpu_launches"] == 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "agent-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_native_arm_refuses_to_run_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        return
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1"], capture_output=True, text=True, timeout=300)
    assert out.returncode != 0 and "no CPU fallback" in (out.stderr + out.stdout)


def _load_dump(d):
    out = {k: np.load(os.path.join(d, k + ".npy")) for k in DUMPED}
    assert all(a.dtype in (np.float32, np.float64) for a in out.values())
    assert sum(os.path.getsize(os.path.join(d, k + ".npy")) for k in DUMPED) <= 64 << 20
    return out


def test_dump_outputs_samples_large_outputs_by_a_fixed_seed(tmp_path):
    """Outputs above the dump budget are cut to the same seeded, sorted set of environments every time, and every
    written row belongs to the environment env_index names."""
    import torch
    import bench
    E, n = 16384, 64   # 67 MB of outputs
    env = torch.arange(E, dtype=torch.float32)
    obs = env.reshape(E, 1, 1).expand(E, n, 12).contiguous()
    rew4 = (env.reshape(1, E, 1) + torch.arange(4.0).reshape(4, 1, 1)).expand(4, E, n).contiguous()
    covered = torch.arange(E, dtype=torch.int32)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), obs, rew4, covered)
    a, b = _load_dump(tmp_path / "a"), _load_dump(tmp_path / "b")
    idx = a["env_index"]
    assert 0 < idx.size < E and np.all(np.diff(idx) > 0) and np.array_equal(idx, b["env_index"])
    assert a["obs"].shape == (idx.size, n, 12) and a["rew4"].shape == (4, idx.size, n)
    assert np.all(a["obs"] == idx[:, None, None]) and np.all(a["covered"] == idx)
    assert np.all(a["rew4"] == idx[None, :, None] + np.arange(4.0)[:, None, None])


@pytest.mark.gpu
def test_dump_outputs_of_the_native_arm_are_reproducible(tmp_path):
    """Two runs with the same arguments dump identical outputs of the last timed step; one more timed step changes
    them, and the JSON line reports the --steps it was given."""
    dumps = {}
    for tag, steps in (("a", 3), ("b", 3), ("c", 4)):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "default4096", "--steps", str(steps),
                              "--warmup", "2", "--no-extras", "--e2e-steps", "1", "--dump-outputs", str(tmp_path / tag)],
                             capture_output=True, text=True, timeout=600)
        assert out.returncode == 0, out.stderr[-2000:]
        line = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
        assert line["steps"] == steps
        dumps[tag] = _load_dump(tmp_path / tag)
    a, b, c = dumps["a"], dumps["b"], dumps["c"]
    assert a["obs"].shape == (4096, 10, 12) and a["rew4"].shape == (4, 4096, 10) and a["covered"].shape == (4096,)
    assert np.array_equal(a["env_index"], np.arange(4096))
    for k in DUMPED:
        assert np.array_equal(a[k], b[k]), k
    assert not np.array_equal(a["obs"], c["obs"]) and not np.array_equal(a["rew4"], c["rew4"])
