#!/usr/bin/env python
"""bench.py -- the headline metric of BASELINE.json on B200:

    log-mll + gradient (update_mll_and_dmll!, src/GPE.jl:332-335) for GPE SEIso, N=32768, d=8, FP64
    reported as algorithmic GFLOP/s (F_alg = N^3 + 2 N^2, SURVEY.md §8(d)) and ms per evaluation.

A "step" is one evaluation of the hot path (Gram build -> Cholesky -> alpha/mll -> K_y^-1 ->
fused gradient trace) on synthetic inputs (x, y ~ N(0,1), seed 1; SEIso(0.3,0.3), logNoise 0.3,
MeanConst(0) -- config C2 of SURVEY.md §8(d)).

  value        inputs resident in HBM, timed with CUDA events on the engine's stream
  e2e          same step through the public GPE API with HOST buffers: x, y uploaded from pinned host
               memory and alpha / mll / dmll read back inside the timed region
  roofline     the dominant kernel (FP64 DMMA NT GEMM): algorithmic flops / sum of its launch
               durations (CUDA events around every launch in one extra profiled step) vs the DMMA
               issue rate measured in the same run (MEASURED_PEAKS.json has no FP64 figure)
  cpu_baseline the reference's algorithm (oracle port: scalar loops in C + LAPACK via OpenBLAS, all
               host cores) on a bounded sample (N=8192) of the same workload
  --impl reference   times only that CPU path (Julia is not installed in this image).
  --dump-outputs DIR after the timed steps, writes what the last timed step of each GPU path returned to its caller
                     as DIR/<name>.npy (float64): alpha, mll, dmll_kernel, trace_A (resident step), e2e_alpha, e2e_mll,
                     e2e_dmll (e2e step), predict_mu, predict_var (predict_f).  Inputs are seeded, so two builds run
                     with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import time

if "reference" in sys.argv[1:] or "--impl=reference" in sys.argv[1:]:
    # torchrun exports OMP_NUM_THREADS=1; the CPU arm must use every host core, so set the BLAS pool size before
    # numpy/scipy load OpenBLAS (threadpoolctl re-asserts it at run time and the line records the count used)
    for _k in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[_k] = str(os.cpu_count() or 1)

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "gaussianprocesses.jl_b200"))

N_FULL, D = 32768, 8
LL, LSIG, LNOISE = 0.3, 0.3, 0.3
N_CPU_SAMPLE = int(os.environ.get("GPB200_CPU_SAMPLE_N", "8192"))      # bounded CPU sample of our arm's cpu_baseline leg
METRIC = "log-mll+grad GFLOP/s, GPE SEIso N=32768 d=8 FP64 (update_mll_and_dmll!)"
WORKLOAD = ("C2: GPE SEIso(0.3,0.3) logNoise 0.3 MeanConst(0), N=%d d=8 FP64: Gram + Cholesky + alpha/mll + K^-1 + "
            "gradient trace per step")
CPU_BUDGET_S = float(os.environ.get("GPB200_CPU_BUDGET_S", "200"))    # wall-clock budget of the whole reference arm


def falg(n):
    return float(n) ** 3 + 2.0 * float(n) ** 2


def synth(n, d, seed=1):
    rng = np.random.default_rng(seed)
    return rng.standard_normal((n, d)), rng.standard_normal(n)


class StdoutToStderr:
    """NCCL prints its version banner on the process's C stdout when the first communicator is created; route fd 1 to
    stderr for that stretch so that rank 0's stdout carries nothing but the one JSON line."""

    def __enter__(self):
        sys.stdout.flush()
        self._saved = os.dup(1)
        os.dup2(2, 1)
        return self

    def __exit__(self, *exc):
        try:
            sys.stdout.flush()
        finally:
            os.dup2(self._saved, 1)
            os.close(self._saved)
        return False


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            out = self.proc.communicate(timeout=5)[0]
        except Exception:
            out = ""
        sm, mx, reasons = [], [], set()
        for line in out.strip().splitlines():
            f = [t.strip() for t in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        busy = [s for s in sm if s > 0.5 * (max(mx) if mx else 1)] or sm
        return {"sm_mhz": float(np.median(busy)) if busy else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def pin_blas_threads():
    """All host cores for OpenBLAS, whatever OMP_NUM_THREADS says (torchrun sets it to 1).  Returns the count in use."""
    want = os.cpu_count() or 1
    try:
        import threadpoolctl
        threadpoolctl.threadpool_limits(limits=want)
        import scipy.linalg  # noqa: F401  (loads the OpenBLAS that LAPACK calls go to)
        threadpoolctl.threadpool_limits(limits=want)
        got = [p.get("num_threads", 1) for p in threadpoolctl.threadpool_info() if p.get("user_api") == "blas"]
        return max(got) if got else want
    except Exception:
        return want


def extrapolate_full(seconds, n, n_full=N_FULL):
    """Phase-wise extrapolation of one CPU evaluation from the sample size n to the metric's N: the scalar cov! /
    dmll_kern! loops and the alpha solve are O(N^2), dpotrf and dpotrs(-I) are O(N^3) (BLAS efficiency assumed
    unchanged).  Returns seconds at n_full."""
    r = float(n_full) / float(n)
    t2 = seconds["cov_loop"] + seconds["dmll_loop"] + seconds["solve_mll"]
    t3 = seconds["dpotrf"] + seconds["potrs_identity_ger"]
    return t2 * r ** 2 + t3 * r ** 3


def full_size_record():
    """One full-size (N=32768) CPU evaluation measured on a pool box and committed (profiles/): validates the extrapolation."""
    pth = os.path.join(ROOT, "profiles", "r02_cpu_full_size.json")
    try:
        return json.load(open(pth))
    except Exception:
        return None


def cpu_baseline_run(n, steps=1):
    from oracle import cpu_baseline as cb
    cores = pin_blas_threads()
    X, y = synth(n, D, seed=1)
    best, last = None, None
    for _ in range(steps):
        r = cb.seiso_mll_and_dmll(X, y, LL, LSIG, LNOISE, 0.0)
        t = r["seconds"]["total"]
        if best is None or t < best:
            best, last = t, r
    return best, last, cores


def run_reference(args, rank, world):
    """Reference arm: the reference's own CPU algorithm (oracle port; Julia is absent from the image) on ALL host cores.
    Each step is a bounded sample of the C2 workload (same kernel, d, distribution; N_sample < 32768 chosen so that
    the warm-up plus the K timed steps fit CPU_BUDGET_S); `value` is the metric at the metric's own N=32768, obtained
    by extrapolating every phase of the measured step with its complexity, the raw sample rate is reported beside it."""
    if rank != 0:
        return
    from oracle import cpu_baseline as cb
    cores = pin_blas_threads()
    per_step = CPU_BUDGET_S / (args.steps + 1)
    # ~8.5 s per evaluation at N=8192 on the pool's 64 host cores (round-1 records); time ~ N^3
    n = int(8192 * (per_step / 8.5) ** (1.0 / 3.0)) // 1024 * 1024
    n = max(2048, min(N_FULL, n))
    if os.environ.get("GPB200_CPU_SAMPLE_N"):
        n = int(os.environ["GPB200_CPU_SAMPLE_N"])
    X, y = synth(n, D, seed=1)
    if args.warmup > 0:
        cb.seiso_mll_and_dmll(X, y, LL, LSIG, LNOISE, 0.0)      # one warm-up is enough for a CPU path (thread pools, page faults)
    ts, phases = [], None
    for _ in range(args.steps):
        r = cb.seiso_mll_and_dmll(X, y, LL, LSIG, LNOISE, 0.0)
        ts.append(r["seconds"]["total"])
        phases = r["seconds"] if phases is None else {k: phases[k] + v for k, v in r["seconds"].items()}
    phases = {k: v / args.steps for k, v in phases.items()}
    t_sample = float(np.mean(ts))
    rate_sample = falg(n) / t_sample * 1e-9
    t_full = extrapolate_full(phases, n) if n != N_FULL else t_sample
    val = falg(N_FULL) / t_full * 1e-9
    rec = full_size_record()
    sample = ("each step = one full update_mll_and_dmll! with the reference's algorithm (scalar cov!/dmll_kern! loops in C, "
              "1 thread, as the reference; dpotrf + dpotrs(-I) + dger via OpenBLAS on %d threads) at N_sample=%d of 32768, d=8: "
              "%.2f s/step = %.1f GFLOP/s at N_sample; value = F_alg(32768) / t(32768) with t extrapolated per phase "
              "(O(N^2): cov %.2f s, dmll %.2f s, solve %.2f s; O(N^3): dpotrf %.2f s, potrs(-I)+ger %.2f s) -> %.0f s"
              % (cores, n, t_sample, rate_sample, phases["cov_loop"], phases["dmll_loop"], phases["solve_mll"],
                 phases["dpotrf"], phases["potrs_identity_ger"], t_full))
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": "GFLOP/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": t_sample * 1e3, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOAD % N_FULL,
                   "sample": "N_sample=%d per step (bounded CPU sample); value is the phase-extrapolated rate at N=32768" % n,
                   "value_kind": "extrapolated_to_full_config" if n != N_FULL else "measured_full_config",
                   "rate_at_sample_gflops": rate_sample, "seconds_full_config_extrapolated": t_full,
                   "full_size_measured_once": rec},
        "cpu_baseline": {"value": val, "unit": "GFLOP/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": "GFLOP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--n", type=int, default=N_FULL, help="override N (debug only; the metric is N=32768)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed steps as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    import gpb200

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback in libgpb200)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        with StdoutToStderr():
            dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
            dist.barrier()

    N = args.n
    X, y = synth(N, D, seed=1)
    # pinned host staging for the e2e leg
    xp = torch.empty((N, D), dtype=torch.float64).pin_memory(); xp.numpy()[:] = X
    yp = torch.empty((N,), dtype=torch.float64).pin_memory(); yp.numpy()[:] = y
    Xh, yh = xp.numpy(), yp.numpy()

    gp = gpb200.GPE(Xh.T, yh, gpb200.MeanConst(0.0), gpb200.SEIso(LL, LSIG), LNOISE, device=local_rank)
    eng = gp._eng
    if world > 1:
        # strong scaling: the SAME N=32768 problem, work partitioned over the ranks (block-column
        # Cholesky with NCCL panel broadcasts, split inverse, row-cyclic W'W + trace)
        with StdoutToStderr():
            gp.init_distributed()
    if os.environ.get("GPB200_SHARD") is not None:          # storage-mode override (replicated 0 / row-sharded 1) for A/B runs
        eng.set_option("shard", int(os.environ["GPB200_SHARD"]))
    stream = torch.cuda.current_stream()
    eng.set_stream(stream.cuda_stream)
    theta = np.array([LL, LSIG])
    r = yh - 0.0

    def step_resident():
        eng.factorize(theta, LNOISE)
        alpha, mll = eng.mll(r)
        eng.grad_prepare()
        gk, tr_a = eng.grad_kernel()
        return {"alpha": alpha, "mll": mll, "dmll_kernel": gk, "trace_A": tr_a}

    def step_e2e():
        gp.reload_data(Xh.T, yh)            # H2D of x and (inside update_mll) y
        gp.update_mll_and_dmll()            # D2H alpha, mll, dmll
        return gp.mll

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        step_resident()
    sampler = ClockSampler(local_rank)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    l0 = eng.launch_count()
    sampler.start()
    e0.record(stream)
    for _ in range(args.steps):
        outputs = step_resident()
    e1.record(stream)
    barrier()
    clocks = sampler.stop()
    launches = eng.launch_count() - l0
    ms_total = e0.elapsed_time(e1)
    tmr = eng.timings()
    if world > 1:
        t = torch.tensor([ms_total], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total = float(t.item())
    ms_step = ms_total / args.steps

    # ---- e2e: host buffers in, host results out, through the public GPE API -------------------
    step_e2e()
    check = {"mll": float(gp.mll), "dmll": [float(v) for v in gp.dmll], "alpha_l1": float(np.sum(np.abs(gp.alpha))),
             "note": "results of one e2e step (host copies of mll, dmll=[noise,beta,ll,lsigma], sum|alpha|); identical "
                     "inputs at every n_gpus, so the lines of a scaling run must agree to ~1e-10 relative"}
    barrier()
    t0 = time.perf_counter()
    e0.record(stream)
    for _ in range(args.steps):
        step_e2e()
    e1.record(stream)
    barrier()
    e2e_wall = (time.perf_counter() - t0) * 1e3 / args.steps
    outputs.update(e2e_alpha=gp.alpha.copy(), e2e_mll=gp.mll, e2e_dmll=gp.dmll.copy())
    e2e_ms = max(e0.elapsed_time(e1) / args.steps, e2e_wall)
    if world > 1:
        t = torch.tensor([e2e_ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_ms = float(t.item())
    h2d = X.nbytes + y.nbytes + theta.nbytes + 8
    d2h = 8 * N + 8 + 8 * (theta.size + 1)

    # ---- roofline of the dominant kernel: one profiled step (events around every GEMM launch) ----
    roof = None
    pk = eng.fp64_peak()
    eng.set_option("profile", 1)
    step_resident()
    torch.cuda.synchronize()
    tp = eng.timings()
    eng.set_option("profile", 0)
    if tp["gemm_ms"] > 0:
        alg = float(N) ** 3 / world                             # N^3/3 Cholesky + 2N^3/3 inverse, all in this kernel (per rank)
        achieved = alg / (tp["gemm_ms"] * 1e-3) * 1e-12
        traffic = None
        tj = os.path.join(ROOT, "profiles", "gemm_traffic.json")
        if os.path.exists(tj):
            try:
                traffic = json.load(open(tj)).get("dram_bytes_per_launch")
            except Exception:
                traffic = None
        roof = {"bound": "tensor", "kernel": "gpb200_dgemm_nt_tma (FP64 DMMA.8x8x4 fed by TMA)",
                "achieved": achieved, "peak": pk["dmma_tflops"], "unit": "TFLOP/s", "frac": achieved / pk["dmma_tflops"],
                "traffic": traffic,
                "traffic_source": "dram__bytes_read+write of the largest launch (W'W) in the committed ncu --set full capture "
                                  "(profiles/gemm_traffic.json); not re-measured in this run",
                "peak_source": "DMMA.8x8x4 issue rate measured in this run (gpb200_fp64_peak); MEASURED_PEAKS.json "
                               "carries no FP64 figure -- its HBM/bf16 numbers do not bound this kernel; DFMA rate "
                               "%.1f TFLOP/s, cuBLAS DGEMM on this pool 36.5 TFLOP/s (profiles/r01_cublas_dgemm.txt)" % pk["dfma_tflops"],
                "launches_per_step": int(tp["gemm_launches"]), "kernel_ms_per_step": tp["gemm_ms"],
                "kernel_share_of_step": tp["gemm_ms"] / ms_step,
                "algorithmic_flops_per_step": alg, "executed_flops_per_step": tp["gemm_flops"]}

    # predict_f (batched, M = 4096 test points, mean + variance), device-timed inside the library (CUDA events)
    Xs = np.random.default_rng(2).standard_normal((4096, D))
    eng.predict(Xs)                        # warm-up: sizes the cross-Gram workspace
    pms = []
    for _ in range(3):
        mu_p, var_p, _ = eng.predict(Xs)
        pms.append(eng.timings()["predict"])
    predict_ms = float(np.median(pms))
    outputs.update(predict_mu=mu_p, predict_var=var_p)
    check["predict_mu_l1"] = float(np.sum(np.abs(mu_p)))
    check["predict_var_sum"] = float(np.sum(var_p))
    hbm_peak = None
    try:
        hbm_peak = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"])
    except Exception:
        hbm_peak = 6574.5                  # B200_PROFILING.md fallback == the pool's measured copy bandwidth
    Npad = (N + 127) // 128 * 128
    T = Npad // 128
    tri_bytes = 8.0 * 128 * 128 * (T * (T + 1) // 2)            # lower tiles of the N x N matrix
    own = 1.0 / world                                          # Gram / trace tiles are dealt over the ranks
    roof_other = {
        "gram_lower_kernel": {"bound": "hbm", "unit": "GB/s", "peak": hbm_peak,
                              "achieved": (tri_bytes * own + 8.0 * N * D) / (tmr["gram"] * 1e-3) * 1e-9,
                              "bytes": "lower 128x128 tiles written once (%.3f GB per rank) + x read" % (tri_bytes * own * 1e-9),
                              "ms": tmr["gram"]},
        "trace_kernel": {"bound": "hbm", "unit": "GB/s", "peak": hbm_peak,
                         "achieved": (tri_bytes * own + 8.0 * N * D) / (tmr["trace"] * 1e-3) * 1e-9,
                         "bytes": "lower tiles of K^-1 read once + x", "ms": tmr["trace"]},
        "predict_f_M4096": {"bound": "tensor", "unit": "TFLOP/s", "peak": pk["dmma_tflops"],
                            "achieved": (float(N) ** 2 * 4096 + 2.0 * N * 4096) / (predict_ms * 1e-3) * 1e-12,
                            "flops": "N^2 M (TRSM) + 2 N M (mean), SURVEY 8(d); includes H2D of x*, cross-Gram, D2H of mu, var",
                            "ms": predict_ms},
    }
    for v in roof_other.values():
        v["frac"] = v["achieved"] / v["peak"]

    if rank == 0:
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            tcpu, res, cores = cpu_baseline_run(N_CPU_SAMPLE, steps=1)
            t_full = extrapolate_full(res["seconds"], N_CPU_SAMPLE)
            cpu = {"value": falg(N_FULL) / t_full * 1e-9, "unit": "GFLOP/s", "cores": cores, "kind": "port",
                   "rate_at_sample": falg(N_CPU_SAMPLE) / tcpu * 1e-9,
                   "sample": "N_sample=%d d=8 (of 32768): one full update_mll_and_dmll! with the reference's algorithm -- scalar "
                             "cov!/dmll_kern! loops (C, 1 thread, as the reference) + dpotrf + dpotrs(-I) (OpenBLAS, %d threads); "
                             "%.1f s; phases %s; value = F_alg(32768)/t(32768), t extrapolated per phase (O(N^2) loops, "
                             "O(N^3) LAPACK) = %.0f s"
                             % (N_CPU_SAMPLE, cores, tcpu, {k: round(v, 2) for k, v in res["seconds"].items()}, t_full),
                   "full_size_measured_once": full_size_record()}
        val = falg(N) / (ms_step * 1e-3) * 1e-9
        line = {
            "metric": METRIC, "value": val, "unit": "GFLOP/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": WORKLOAD % N,
                       "l2": "working set (two 8.6 GB N x N FP64 matrices) exceeds the 126 MB L2; no flush needed",
                       "parallelism": "1 GPU" if world == 1 else
                       "%d GPUs: 1-D block-cyclic block columns (NCCL panel broadcast over NVLink, look-ahead), "
                       "split level-parallel inverse + all-gather, tile-row-cyclic W'W/trace + all-reduce of P+1 sums; "
                       "F/G %s" % (world, "row-sharded over the GPUs (own block rows mapped)" if eng.storage_info()["sharded"] else "replicated per GPU"),
                       "phases_ms": {k: round(v, 3) for k, v in tmr.items() if k in ("gram", "cholesky", "solve_mll", "inverse", "trace")},
                       "predict_f_ms_M4096": predict_ms},
            "clocks": clocks,
            "e2e": {"value": falg(N) / (e2e_ms * 1e-3) * 1e-9, "unit": "GFLOP/s", "ms_per_step": e2e_ms,
                    "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h)},
            "gpu_launches": int(launches),
            "roofline": roof,
            "roofline_other": roof_other,
            "check": check,
            "cpu_baseline": cpu,
        }
        if args.dump_outputs:
            os.makedirs(args.dump_outputs, exist_ok=True)
            for name, v in outputs.items():
                np.save(os.path.join(args.dump_outputs, name + ".npy"), np.atleast_1d(np.asarray(v, dtype=np.float64)))
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
