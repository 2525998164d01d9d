"""The bench line committed from the GPU box (profiles/r01_bench_final_cfg3.json) carries every key the measurement
contract names, and bench.py's reference arm prints exactly one JSON line with its own keys (run here on the CPU).
On a GPU: --dump-outputs writes the last timed learn step's outputs."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_committed_bench_line_has_the_contract_keys():
    j = json.load(open(os.path.join(ROOT, "profiles", "r01_bench_final_cfg3.json")))
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
              "dtype", "data", "config", "e2e", "gpu_launches", "clocks", "roofline", "cpu_baseline"):
        assert k in j, k
    assert j["metric"] == "agent-updates/sec" and j["higher_is_better"] is True and j["scaling"] == "weak" and j["vs_baseline"] is None
    assert "workload" in j["config"] and j["config"]["workload"].startswith("cfg3")
    assert set(("value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step")) <= set(j["e2e"]) and j["e2e"]["h2d_bytes_per_step"] > 0
    assert set(("bound", "achieved", "peak", "unit", "frac", "traffic")) <= set(j["roofline"])
    assert abs(j["roofline"]["frac"] - j["roofline"]["achieved"] / j["roofline"]["peak"]) < 1e-9 and j["roofline"]["traffic"] > 0
    assert set(("value", "unit", "cores", "kind", "sample")) <= set(j["cpu_baseline"]) and j["cpu_baseline"]["kind"] == "port"
    assert j["gpu_launches"] == 4 * j["steps"] and j["warmup"] >= 3
    assert set(("sm_mhz", "sm_max_mhz", "reasons")) <= set(j["clocks"])
    assert not set(j["clocks"]["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}


def test_reference_arm_prints_one_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, cwd=ROOT, timeout=600)
    assert out.returncode == 0, out.stderr[-500:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    j = json.loads(lines[0])
    assert j["impl"] == "reference" and j["metric"] == "agent-updates/sec" and j["higher_is_better"] is True
    assert j["e2e"]["h2d_bytes_per_step"] == 0 and j["e2e"]["value"] == j["value"] == j["cpu_baseline"]["value"]
    assert j["config"]["workload"].startswith("cfg3")


@pytest.mark.gpu
def test_dump_outputs_writes_the_last_timed_learn_step(tmp_path):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "3", "--blocks", "none",
                          "--no-cpu-baseline", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, cwd=ROOT, timeout=900)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1 and json.loads(lines[0])["steps"] == 2
    names = ("metrics", "theta_sample", "theta_target_sample", "adam_m_sample", "adam_v_sample")
    assert sorted(os.listdir(tmp_path)) == sorted(f"{n}.npy" for n in names)
    a = {n: np.load(os.path.join(tmp_path, f"{n}.npy")) for n in names}
    assert all(v.dtype == np.float32 and np.isfinite(v).all() for v in a.values())
    assert sum(v.nbytes for v in a.values()) <= 64 << 20
    m = a["metrics"]
    assert m.shape == (256, 8) and (m[:, 7] == 1).all() and (m[:, 0] > 0).all()      # every ring full: every network learned
    assert (m[:, 3:7].sum(1) == 256).all()                                               # action histogram over the batch
    assert all(a[n].shape == (1 << 20,) for n in names[1:])
    # five learn steps from zero moments, no target sync yet (frequency 1000)
    assert (a["adam_v_sample"] >= 0).all() and (a["adam_v_sample"] > 0).any() and (a["adam_m_sample"] != 0).any()
    assert not np.array_equal(a["theta_sample"], a["theta_target_sample"])
