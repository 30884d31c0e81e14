"""bench.py contract on the CPU: the reference arm (`--impl reference`: the oracle's simplex over a process pool)
prints one JSON line with the documented keys, and under a multi-rank launch only rank 0 works.  Also
`--dump-outputs`: the arrays of the last timed step, on both arms (ours needs a GPU)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(env_extra=None, args=("--impl", "reference", "--case", "case9", "--steps", "2", "--warmup", "1",
                               "--ref-sample", "2")):
    env = dict(os.environ)
    env.update(env_extra or {})
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True,
                         timeout=300, env=env, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    return out.stdout.strip()


def _load_dump(d):
    arrays = {f[:-4]: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d))}
    assert all(f.endswith(".npy") for f in os.listdir(d))
    assert all(v.dtype == np.float64 for v in arrays.values())
    assert sum(v.nbytes for v in arrays.values()) <= 64 * 10**6
    return arrays


def test_reference_arm_json_line():
    line = _run().splitlines()[-1]
    d = json.loads(line)
    assert d["impl"] == "reference" and d["unit"] == "scenarios/s" and d["higher_is_better"] is True
    assert d["steps"] == 2 and d["warmup"] == 1 and d["value"] > 0 and d["ms_per_step"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["config"]["optimal"] == 4 and "workload" in d["config"] and d["scaling"] == "strong" and d["dtype"] == "f64"


def test_reference_arm_other_ranks_exit_quietly():
    assert _run({"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"}) == ""


def test_reference_arm_dumps_its_last_step(tmp_path):
    """One warm-up and two timed steps of two scenarios each: the dump holds scenarios 5 and 6, as solved again here."""
    import bench
    _run(args=("--impl", "reference", "--case", "case9", "--steps", "2", "--warmup", "1", "--ref-sample", "2",
               "--dump-outputs", str(tmp_path)))
    d = _load_dump(tmp_path)
    assert set(d) == {"scenario_id", "status", "objective"}
    assert d["scenario_id"].tolist() == [5.0, 6.0] and d["status"].tolist() == [0.0, 0.0]
    bench._cpu_init("case9")
    assert np.allclose(d["objective"], [bench._cpu_solve((s, 1000.0))[2] for s in (5, 6)], rtol=1e-12, atol=0)


@pytest.mark.gpu
def test_our_arm_dumps_its_last_step(gpu, tmp_path):
    """The batch arm at a small size: every scenario's status, objective and violation, the full vectors of all of them
    (8 fit the sample), and objective = f + df'p for each, on the inputs bench.py builds."""
    import bench
    line = _run(args=("--case", "case9", "--scenarios", "8", "--steps", "2", "--warmup", "2", "--single-case", "none",
                      "--cpu-sample", "0", "--dump-outputs", str(tmp_path))).splitlines()[-1]
    assert json.loads(line)["config"]["optimal"] == 8
    d = _load_dump(tmp_path)
    assert set(d) == {"scenario_id", "status", "objective", "violation", "sample_scenario_id", "p", "lambda",
                      "mult_x_U", "mult_x_L", "p_slack"}
    ids = list(range(1, 9))
    assert d["scenario_id"].tolist() == ids and d["sample_scenario_id"].tolist() == ids
    assert np.all(d["status"] == 0) and d["violation"].shape == (8,)
    mdl, inp = bench.linearise(bench.network("case9"), ids)
    assert d["p"].shape == (8, mdl.n) and d["lambda"].shape == (8, mdl.m) and d["p_slack"].shape == (8, mdl.m, 2)
    assert np.all(np.abs(d["p"]) <= 1000.0 + 1e-9)
    pobj = inp["f"] + np.einsum("sn,sn->s", inp["df"], d["p"])
    assert np.allclose(pobj, d["objective"], rtol=1e-9, atol=1e-9)
