"""Latent-GP (GPA) target + gradient step at the full-size config on one GPU: N = 32768, d = 8, Bernoulli likelihood,
SEIso + Noise kernel (numerically PD at GPA's exp(-40) nugget).  Usage: python profiles/tools/gpa_bench.py [out.json] [N]

One step is update_target_and_dtarget: Gram + Cholesky, f = L v, and gpb200_gpa_grad (L' g, the triangular-inverse
merges, the row scan, the two GEMMs of P + P', the kernel-gradient trace).  Per-phase times are the engine's CUDA
events (Engine.timings()); the step time is a host clock around the step, whose calls all end in a stream synchronise.

Algorithmic flops of a step: F = N^3/3 (Cholesky) + N^3/3 (triangular inverse) + 2 N^3/3 (P + P' as two triangular
NT GEMMs); the rate is F over the step time.  The in-run DMMA peak (gpb200_fp64_peak) and the card's name and power
limit are read in the same run."""
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.join(ROOT, "gaussianprocesses.jl_b200"))
import gpb200                                       # noqa: E402
from scipy.special import expit                     # noqa: E402

WARMUP, STEPS = 3, 5


def device_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power, clock = [s.strip() for s in q.split(",")]
    return dict(name=name, power_limit=power, max_sm_clock=clock)


def main():
    out = sys.argv[1] if len(sys.argv) > 1 else None
    N = int(sys.argv[2]) if len(sys.argv) > 2 else 32768
    d = 8
    rng = np.random.default_rng(0)
    X = rng.standard_normal((N, d))
    y = rng.random(N) < expit(np.sin(X).sum(axis=1))
    gp = gpb200.GPA(X.T, y, gpb200.MeanZero(), gpb200.SEIso(0.0, 0.0) + gpb200.Noise(-2.0), gpb200.BernLik())
    gp.set_params(np.concatenate([0.5 * rng.standard_normal(N), gp.get_params()[N:]]))
    steps, phases = [], []
    for it in range(WARMUP + STEPS):
        t0 = time.perf_counter()
        gp.update_target_and_dtarget()
        t1 = time.perf_counter()
        if it >= WARMUP:
            tm = gp._eng.timings()
            steps.append((t1 - t0) * 1e3)
            phases.append(dict(gram=tm["gram"], cholesky=tm["cholesky"], unwhiten=tm["gpa_unwhiten"], lt_g=tm["gpa_trmv_t"],
                               inverse_merges=tm["gpa_merges"], scan=tm["gpa_scan"], gemms_P_plus_Pt=tm["gpa_gemms"],
                               trace=tm["trace"]))
    F = N ** 3 / 3 + N ** 3 / 3 + 2 * N ** 3 / 3
    ms = float(np.median(steps))
    ph = {k: float(np.median([p[k] for p in phases])) for k in phases[0]}
    res = dict(config=dict(N=N, d=d, likelihood="BernLik", kernel="SEIso(0,0) + Noise(-2)", warmup=WARMUP, steps=STEPS),
               device=device_info(), step_ms=ms, step_ms_all=steps, phase_ms=ph,
               flops_formula="N^3/3 + N^3/3 + 2N^3/3", flops=F, tflops_step=F / (ms * 1e-3) * 1e-12,
               tflops_gemms=(2 * N ** 3 / 3) / (ph["gemms_P_plus_Pt"] * 1e-3) * 1e-12,
               fp64_peak=gp._eng.fp64_peak(), target=gp.target, dtarget_kernel=gp.dtarget[N:].tolist())
    line = json.dumps(res)
    print(line)
    if out:
        with open(out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
