"""The JSON line bench.py prints, checked key by key against the driver's contract: on the lines committed under profiles/ (GPU runs of
this round) and on a live run of the CPU reference arm."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE = {"metric": str, "value": (int, float), "unit": str, "n_gpus": int, "steps": int, "warmup": int, "ms_per_step": (int, float),
        "higher_is_better": bool, "scaling": str, "dtype": str, "data": str, "config": dict}


def _line(path):
    return json.loads([l for l in open(path) if l.startswith("{")][-1])


def _check_common(j):
    for k, t in BASE.items():
        assert k in j and isinstance(j[k], t), (k, j.get(k))
    assert "vs_baseline" in j and j["vs_baseline"] is None           # BASELINE.md holds no published number for this metric
    assert "workload" in j["config"] and not ({"model", "seq_len", "global_batch"} & set(j["config"]))
    e = j["e2e"]
    assert set(e) >= {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"} and e["unit"] == j["unit"]


@pytest.mark.parametrize("name", ["r02_bench_1gpu_lv.json", "r02_bench_8gpu_lv.json", "r02_bench_hjb.json", "r02_bench_1gpu_seir.json"])
def test_committed_gpu_lines(name):
    j = _line(os.path.join(ROOT, "profiles", name))
    _check_common(j)
    assert j["value"] > 0 and j["gpu_launches"] > 0 and j["e2e"]["value"] > 0
    assert j["e2e"]["h2d_bytes_per_step"] > 0 and j["e2e"]["d2h_bytes_per_step"] > 0 and abs(j["e2e"]["value"] - j["value"]) > 0
    r = j["roofline"]
    assert r["bound"] in ("hbm", "tensor") and r["unit"] in ("GB/s", "TFLOP/s") and set(r) >= {"achieved", "peak", "frac", "traffic"}
    assert abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9 and 0 < r["frac"] <= 1
    c = j["clocks"]
    assert set(c) >= {"sm_mhz", "sm_max_mhz", "reasons"} and not ({"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"} & set(c["reasons"]))
    if j["n_gpus"] == 1:
        b = j["cpu_baseline"]
        assert set(b) >= {"value", "unit", "cores", "kind", "sample"} and b["kind"] in ("port", "reference") and b["cores"] >= 1
    else:
        assert j["scaling"] == "weak" and j["allreduce_check"]["bitwise_identical_on_all_ranks"]


@pytest.mark.parametrize("extra", [["--n-per-gpu", "1024"], ["--config", "hjb", "--n-per-gpu", "200"]])
def test_reference_arm_live(extra):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "3", "--warmup", "1"] + extra,
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    j = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
    _check_common(j)
    assert j["impl"] == "reference" and j["value"] > 0 and j["steps"] == 3
    assert j["e2e"]["value"] == j["value"] and j["e2e"]["h2d_bytes_per_step"] == 0 and j["e2e"]["d2h_bytes_per_step"] == 0
    b = j["cpu_baseline"]
    assert b["kind"] == "port" and b["value"] == j["value"] and b["cores"] >= 1 and isinstance(b["sample"], str)


@pytest.mark.gpu
def test_dump_outputs_hold_the_last_timed_step(tmp_path, O):
    """--dump-outputs writes what the timed step returns -- the saved states, loss and grad_theta of the seeded LV ensemble -- and they
    agree with the CPU oracle on the same inputs."""
    import numpy as np
    from helpers import glorot_theta, synthetic_ensemble
    n = 1024
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1", "--n-per-gpu", str(n),
                          "--no-strong", "--no-cpu-baseline", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    assert json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])["steps"] == 2
    got = {k: np.load(tmp_path / f"{k}.npy") for k in ("out", "grad_theta", "loss")}
    assert {k: (v.shape, v.dtype) for k, v in got.items()} == {"out": ((31, 2, n), np.float32), "grad_theta": ((1218,), np.float32),
                                                                 "loss": ((1,), np.float32)}
    theta = glorot_theta((2, 32, 32, 2), seed=1)
    u0, y = synthetic_ensemble(n, seed=0)
    l64, g64, _, out64 = O.ensemble_loss_grad(O.lv_model(), theta.astype(np.float64), u0, y, np.ones(2), 0.1, 30, want_out=True)
    assert np.all(np.abs(got["out"] - out64) <= 3e-4 * (1 + np.abs(out64)))
    assert abs(got["loss"][0] - l64) <= 1e-4 * abs(l64)
    assert np.linalg.norm(got["grad_theta"] - g64) <= 2e-3 * np.linalg.norm(g64)


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--n-per-gpu", "512"],
                         capture_output=True, text=True, timeout=300, env=env)
    assert out.returncode == 0 and not [l for l in out.stdout.splitlines() if l.startswith("{")]
