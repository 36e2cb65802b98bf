"""CPU tier: bench.py's JSON contract on the arm that runs without a GPU (`--impl reference`, the CPU oracle port)."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))


@pytest.mark.parametrize("variant", ["v0", "v5"])
def test_reference_arm_prints_one_contract_line(variant):
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                          "--variant", variant], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600)
    assert res.returncode == 0, res.stderr[-2000:]
    lines = [l for l in res.stdout.splitlines() if l.strip()]
    assert len(lines) == 1                                   # ONE JSON line on stdout, nothing else
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "env_steps_per_sec" and d["unit"] == "env-steps/s"
    assert d["higher_is_better"] is True and d["scaling"] == "weak" and d["vs_baseline"] is None
    assert d["value"] > 0 and d["steps"] == 1 and d["warmup"] == 1 and d["n_gpus"] == 1 and d["gpu_launches"] == 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "model" not in d["config"]


def test_reference_arm_other_ranks_stay_silent():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
                          "--warmup", "1"], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=120, env=env)
    assert res.returncode == 0 and res.stdout.strip() == ""


@pytest.mark.gpu
@pytest.mark.parametrize("variant", ["v0", "v5"])
def test_dump_outputs_repeat_exactly(variant, tmp_path):
    """--dump-outputs writes the last timed step's outputs; two runs with the same arguments write the same bits, and
    --steps is the number of timed steps."""
    import numpy as np
    names = ["obs", "reward", "done", "env_index", "obs_env_index"]
    if variant == "v5":
        names += ["local_obs", "local_reward", "local_done", "foveal_goal"]
    runs = []
    for k in range(2):
        out = tmp_path / ("run%d" % k)
        res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--variant", variant, "--envs", "3000",
                              "--steps", "4", "--warmup", "3", "--no-extras", "--no-cpu-baseline", "--dump-outputs", str(out)],
                             stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600)
        assert res.returncode == 0, res.stderr[-2000:]
        d = json.loads(res.stdout)
        assert d["steps"] == 4 and d["warmup"] == 3
        if variant == "v0":
            assert d["gpu_launches"] == 4                       # one fused launch per timed step
        assert sorted(p.name for p in out.iterdir()) == sorted(n + ".npy" for n in names)
        runs.append({n: np.load(str(out / (n + ".npy"))) for n in names})
    a, b = runs
    assert sum(x.nbytes for x in a.values()) <= 64 << 20
    assert a["reward"].shape == (3000,) and a["obs"].shape[0] == 256 and a["obs_env_index"].shape == (256,)
    for n in names:
        assert a[n].dtype in (np.float32, np.float64)
        assert np.array_equal(a[n].view(np.uint8), b[n].view(np.uint8)), n
    assert set(np.unique(a["reward"].view(np.uint32)).tolist()) <= {0x80000000, 0xBF800000, 0xBC23D70A, 0x42C80000}


def test_default_warmup_puts_the_foveal_variants_in_steady_state(monkeypatch):
    """bench.py's own arm warms v2 / v4 / v5 for 1,000 steps unless told otherwise (their episodes start together and need
    that long to de-synchronise, DESIGN.md 3.5); everything else, and the CPU arm, keeps the short default."""
    sys.path.insert(0, ROOT)
    import bench

    def parsed(*argv):
        monkeypatch.setattr(sys, "argv", ["bench.py", *argv])
        return bench.parse_args()
    assert parsed().warmup == 5 and parsed("--variant", "v3").warmup == 5
    for v in ("v2", "v4", "v5"):
        assert parsed("--variant", v).warmup == 1000
        assert parsed("--variant", v, "--impl", "reference").warmup == 5
        assert parsed("--variant", v, "--warmup", "7").warmup == 7
    assert "steady_state" in bench.workload_config(parsed("--variant", "v4"))
    assert "steady_state" not in bench.workload_config(parsed())
