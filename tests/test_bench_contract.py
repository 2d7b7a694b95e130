"""CPU: bench.py's contract -- the reference arm runs on host cores and prints one JSON line with the agreed
keys; the committed B200 bench lines carry every key the driver / judge read."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT

REQUIRED = ["metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
            "vs_baseline", "dtype", "data", "config", "e2e", "gpu_launches", "cpu_baseline"]


def test_reference_arm_prints_contract_line():
    env = dict(os.environ, GPB200_CPU_SAMPLE_N="768")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                       capture_output=True, text=True, timeout=300, env=env, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    j = json.loads(lines[0])
    for k in REQUIRED:
        assert k in j, k
    assert j["impl"] == "reference" and j["unit"] == "GFLOP/s" and j["higher_is_better"] is True
    assert j["cpu_baseline"]["kind"] == "port" and j["cpu_baseline"]["cores"] >= 1
    assert j["e2e"]["h2d_bytes_per_step"] == 0 and j["gpu_launches"] == 0
    assert j["value"] > 0 and "workload" in j["config"]
    # same config string as our arm; the value is the phase-extrapolated full-config rate, the raw sample rate sits beside it
    assert "N=32768" in j["config"]["workload"] and j["config"]["value_kind"] == "extrapolated_to_full_config"
    assert j["config"]["rate_at_sample_gflops"] > 0 and "N_sample=768" in j["cpu_baseline"]["sample"]


def test_reference_arm_ignores_torchrun_thread_pinning():
    """torchrun exports OMP_NUM_THREADS=1; the CPU arm must still use every host core and say how many."""
    env = dict(os.environ, GPB200_CPU_SAMPLE_N="512", OMP_NUM_THREADS="1", RANK="0", LOCAL_RANK="0", WORLD_SIZE="2")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=300, env=env, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    j = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][0])
    assert j["cpu_baseline"]["cores"] == (os.cpu_count() or 1)


def test_phase_extrapolation_model():
    import bench
    sec = {"cov_loop": 1.0, "dmll_loop": 2.0, "solve_mll": 0.5, "dpotrf": 3.0, "potrs_identity_ger": 10.0}
    assert abs(bench.extrapolate_full(sec, 8192, 32768) - (3.5 * 16 + 13.0 * 64)) < 1e-9
    assert abs(bench.extrapolate_full(sec, 32768, 32768) - 16.5) < 1e-9


def test_reference_arm_other_ranks_stay_silent():
    env = dict(os.environ, GPB200_CPU_SAMPLE_N="256", RANK="1", LOCAL_RANK="1", WORLD_SIZE="2")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=120, env=env, cwd=ROOT)
    assert r.returncode == 0 and r.stdout.strip() == ""


@pytest.mark.gpu
def test_dump_outputs_hold_what_the_timed_steps_returned(tmp_path):
    """--dump-outputs writes float64 arrays of the last timed steps; on bench.py's own seeded inputs they equal the oracle
    (tolerances of the parity tests)."""
    import bench
    from oracle import gp_oracle as orc
    n = 1536
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--n", str(n), "--steps", "2", "--warmup", "1",
                        "--no-cpu-baseline", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    j = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][0])
    assert j["steps"] == 2
    out = {p.name[:-4]: np.load(p) for p in tmp_path.glob("*.npy")}
    assert set(out) == {"alpha", "mll", "dmll_kernel", "trace_A", "e2e_alpha", "e2e_mll", "e2e_dmll", "predict_mu",
                        "predict_var"}
    assert all(v.dtype == np.float64 for v in out.values())
    assert sum(v.nbytes for v in out.values()) <= 64 << 20
    X, y = bench.synth(n, bench.D, seed=1)
    spec = ("SEIso", [bench.LL, bench.LSIG])
    o = orc.mll_and_dmll(spec, X, y, bench.LNOISE, ("MeanConst", 0.0))
    rel = lambda a, b: float(np.max(np.abs(a - b)) / np.max(np.abs(b)))
    for m in (out["mll"], out["e2e_mll"]):
        assert m.shape == (1,) and abs(m[0] - o["mll"]) <= 1e-10 * abs(o["mll"])
    assert rel(out["alpha"], o["alpha"]) < 1e-10 and rel(out["e2e_alpha"], o["alpha"]) < 1e-10
    assert rel(out["dmll_kernel"], o["dmll_kernel"]) < 1e-8 and rel(out["e2e_dmll"], o["dmll"]) < 1e-8
    assert abs(out["trace_A"][0] - o["trA"]) <= 1e-8 * abs(o["trA"])
    mo, vo = orc.predict_f(spec, X, o, np.random.default_rng(2).standard_normal((4096, bench.D)), ("MeanConst", 0.0))
    assert rel(out["predict_mu"], mo) < 1e-10
    assert np.max(np.abs(out["predict_var"] - vo)) <= 1e-10 * np.max(np.abs(vo)) + 1e-13


@pytest.mark.parametrize("name", ["r01_final_bench_1gpu.json", "r01_final_bench_2gpu.json", "r01_final_bench_8gpu.json"])
def test_committed_bench_lines_have_every_key(name):
    j = json.load(open(os.path.join(ROOT, "profiles", name)))
    for k in REQUIRED + ["clocks", "roofline"]:
        assert k in j, (name, k)
    assert j["dtype"] == "f64" and j["scaling"] == "strong" and j["data"] == "synthetic"
    assert j["gpu_launches"] > 0 and j["e2e"]["h2d_bytes_per_step"] > 0
    assert not set(j["clocks"]["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}
    if j["n_gpus"] == 1:
        rf = j["roofline"]
        assert rf["bound"] == "tensor" and rf["unit"] == "TFLOP/s" and 0.5 < rf["frac"] <= 1.05
        assert abs(rf["frac"] - rf["achieved"] / rf["peak"]) < 1e-9
        assert j["cpu_baseline"]["kind"] == "port"
        # value == F_alg / time
        assert abs(j["value"] - (32768.0 ** 3 + 2 * 32768.0 ** 2) / (j["ms_per_step"] * 1e-3) * 1e-9) < 1e-6 * j["value"]
