#!/usr/bin/env python
"""bench.py -- headline benchmark: BASELINE.json configs[1], batched Levenberg-Marquardt fits.

    python bench.py --gpus N --steps K --warmup W            # this engine (CUDA, sm_100a)
    python bench.py --impl reference --gpus N --steps K ...  # the reference algorithm on the host CPUs

A "step" is one pass of the hot path over one batch: `batch` independent 4-parameter
Gaussian-peak fits (m = 64 samples, double, box bounds, analytic Jacobian, reference default
settings), every fit run to the reference's own termination.  Metric: LM problems solved / s.

Own arm, three measurements in one run:
  value      device-resident: inputs already in HBM, CUDA events on the launching stream,
             barrier + synchronize on both sides, max over ranks.
  e2e        through the host-pointer C-ABI call (mir_optimize_least_squares_batched_d) with
             pinned HOST buffers: H2D of samples/guesses/bounds and D2H of parameters/results are
             inside the timed region.
  roofline   achieved FP64 FMA-pipe TFLOP/s (algorithmic flops counted from on-device work
             counters, SURVEY 8d convention) against the DFMA peak measured on this GPU, plus
             the algorithmic-bytes HBM figure against MEASURED_PEAKS.json.
  cpu_baseline   the CPU oracle (restated reference + real LAPACK posvx) on all host cores, on a
             bounded sample of the same workload (rank 0, N=1 only).

Reference arm (`--impl reference`): the oracle on all host cores, bounded sample per step.

`--dump-outputs DIR` writes what the last timed step of the device-resident arm computed (rank 0) as float64 .npy
files, so that two builds run with the same arguments (hence the same seeded inputs) can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.dont_write_bytecode = True          # the benchmark writes nothing into the tree it runs from
sys.path.insert(0, ROOT)

M, N = 64, 4
C_F, C_G = 8, 6          # model flops per row for f, and for the analytic Jacobian given f's intermediates (SURVEY 8d)
WORKLOAD = ("configs[1]: batched independent 4-parameter Gaussian-peak fits, m=64 samples each, double, box bounds, "
            "analytic Jacobian, reference default settings (BASELINE names it 'one warp per problem'; at this batch size the "
            "library runs one THREAD per problem, see roofline.kernel)")


def algorithmic_flops(stats, m=M, n=N):
    """SURVEY 8d convention (FMA = 2 flops, exp/sqrt/div = 1 flop; the reference's redundant SYRK on
    rejected passes is NOT counted)."""
    jac = stats["fresh_jacobians"] + stats["broyden_updates"]
    return (stats["model_evals"] * m * (C_F + 2)
            + stats["qp_solves"] * (n ** 3 / 3 + 2 * n * n)
            + stats["passes"] * 2 * n * n
            + jac * (2 * m * n + m * n * (n + 1))
            + stats["broyden_updates"] * 4 * m * n
            + stats["fresh_jacobians"] * m * C_G)


ALGO_BYTES_PER_FIT = M * 8 + N * 8 + N * 8 + 32      # samples + guess + solution + Result = 608 B (shared grid/bounds)
DUMP_BYTES = 64_000_000


def dump_outputs(out_dir, x, results):
    """Writes x.npy (batch x n parameters), one file per Result field and rows.npy (the row numbers written), all float64.
    When every row does not fit in DUMP_BYTES, the rows are a fixed seeded sample, the same in every run of one batch size.
    +-inf is written as the largest finite double of that sign: a fit that stops because lambda exceeded maxLambda
    (furtherImprovement) returns lambda = +inf whenever the last increase overflowed, as the reference does, and every lambda
    above maxLambda is the same state of the algorithm.  NaN is written as NaN."""
    arrays = {"x": x, **{f: results[f] for f in results.dtype.names}}
    row_bytes = 8 * (1 + sum(a[0].size for a in arrays.values()))
    batch = len(x)
    keep = min(batch, (DUMP_BYTES - 4096) // row_bytes)          # (4096: room for the .npy headers)
    rows = np.arange(batch) if keep == batch else np.sort(np.random.default_rng(0).choice(batch, keep, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "rows.npy"), rows.astype(np.float64))
    big = np.finfo(np.float64).max
    for name, a in arrays.items():
        a = np.nan_to_num(np.asarray(a[rows], dtype=np.float64), nan=np.nan, posinf=big, neginf=-big)
        np.save(os.path.join(out_dir, f"{name}.npy"), np.ascontiguousarray(a))


class ClockSampler:
    """Samples nvidia-smi SM clocks / throttle reasons while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index, self.samples, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for s in self.samples:
            f = [v.strip() for v in s.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0])); mx = float(f[1])
            except ValueError:
                continue
            for nme, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(nme)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f), "measured (MEASURED_PEAKS.json)"
    return {"hbm_gbs": 6650.0}, "fallback (B200_PROFILING.md: 6.65 TB/s)"


def cpu_oracle_rate(wl, sample, nthreads=0):
    """fits/s of the CPU oracle on the first `sample` problems, all host cores."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from conftest import load_oracle
    from oracle_util import oracle_batched_mp
    import mir_optim_b200._abi as abi
    import ctypes as C
    lib = load_oracle()
    s = abi.LeastSquaresSettingsD()
    abi.bind_reference_abi(lib)
    lib.mir_least_squares_init_d(C.byref(s))
    t0 = time.perf_counter()
    _, res, threads = oracle_batched_mp(lib, s, wl.model, wl.x0[:sample], wl.l, wl.u, t=wl.t, y=wl.y[:sample], procs=nthreads)
    dt = time.perf_counter() - t0
    return sample / dt, threads, dt, res


def _timed(torch, fn, reps):
    """mean CUDA-event time (ms) of `reps` calls after one warm-up call."""
    fn(); torch.cuda.synchronize()
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def secondary_batched(torch, eng, dev, workloads, rank):
    """configs[2] (8-parameter sum of exponentials, FD Jacobian, double and float) and configs[4]a (batched n=64 BoxQP):
    device-resident throughput of THIS rank's GPU (the batched paths shard without communication)."""
    out = {}
    for name, dt in (("c3_sumexp8_f64", np.float64), ("c3_sumexp8_f32", np.float32)):
        B = 1 << 20                    # BASELINE configs[2]: 1M fits
        wl = workloads.c3_sumexp8(B, dtype=dt, seed=3 + rank)
        st = eng.settings(dt)
        T = lambda v: torch.from_numpy(v).to(dev)
        t, y, x0, l, u = T(wl.t), T(wl.y), T(wl.x0), T(wl.l), T(wl.u)
        x = torch.empty_like(x0)
        res = torch.empty(B * (32 if dt == np.float64 else 24), dtype=torch.uint8, device=dev)

        def step():
            x.copy_(x0)
            eng.optimize_batched_device(st, wl.model, x, l, u, t=t, y=y, fd_jacobian=True, results=res)
        ms = _timed(torch, step, 2)
        ok = float(np.mean(eng.results_from_bytes(res, dt)["status"] >= 0))
        # roofline of this config: SURVEY 8d's conservative algorithmic count, 1.6e6 flop per fit (exp = 1 flop), against the
        # FP64 / FP32 FMA peak measured live; the kernel is lm_mux_kernel (four fits per warp, J^T J on the FP64 tensor pipe)
        peak = eng.lib.mir_b200_measure_peak_tflops(0 if dt == np.float64 else 2, 3)
        ach = 1.6e6 * B / (ms * 1e-3) / 1e12
        out[name] = {"value": B / ms * 1e3, "unit": "fits/s per GPU", "batch": B, "m": 128, "n": 8, "jacobian": "finite differences",
                     "ms": ms, "frac_status_ok": ok,
                     "roofline": {"bound": "fp64_fma" if dt == np.float64 else "fp32_fma", "kernel": "lm_mux_kernel<ModelSumExp<T,8>, T, finite differences>",
                                  "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak if peak > 0 else None,
                                  "algorithmic_flops_per_fit": 1.6e6,
                                  "hbm_GBps_algorithmic": (1184 if dt == np.float64 else 600) * B / (ms * 1e-3) / 1e9}}
    # configs[4]b: configs[1] with bounds tightened so that at least one is active at the solution (every pass runs BOXCQP's
    # active-set loop), 2^20 fits, thread-per-problem kernel
    B = 1 << 20
    wl = workloads.c2_gauss4(B, noise=0.05, tight_bounds=True, seed=7 + rank)
    st = eng.settings(np.float64)
    T = lambda v: torch.from_numpy(v).to(dev)
    t, y, x0, l, u = T(wl.t), T(wl.y), T(wl.x0), T(wl.l), T(wl.u)
    x = torch.empty_like(x0)
    res = torch.empty(B * 32, dtype=torch.uint8, device=dev)

    def step_b():
        x.copy_(x0)
        eng.optimize_batched_device(st, wl.model, x, l, u, t=t, y=y, results=res)
    ms = _timed(torch, step_b, 2)
    xh = x.cpu().numpy()
    out["c5b_gauss4_active_bounds_f64"] = {"value": B / ms * 1e3, "unit": "fits/s per GPU", "batch": B, "m": 64, "n": 4, "ms": ms,
                                           "frac_status_ok": float(np.mean(eng.results_from_bytes(res, np.float64)["status"] >= 0)),
                                           "frac_on_a_bound": float(np.mean(np.any((xh == wl.l) | (xh == wl.u), axis=1)))}
    del t, y, x0, x, res
    B, n = 100000, 64
    g = torch.Generator(device=dev); g.manual_seed(5 + rank)
    P = torch.empty(B, n, n, dtype=torch.float64, device=dev)
    eye = 0.1 * torch.eye(n, dtype=torch.float64, device=dev)
    for s0 in range(0, B, 4096):
        e = min(B, s0 + 4096)
        A = torch.randn(e - s0, 256, n, dtype=torch.float64, device=dev, generator=g)
        P[s0:e] = torch.bmm(A.transpose(1, 2), A) / 256 + eye
    q = torch.randn(B, n, dtype=torch.float64, device=dev, generator=g)
    l = -2.0 * torch.rand(B, n, dtype=torch.float64, device=dev, generator=g)
    u = 2.0 * torch.rand(B, n, dtype=torch.float64, device=dev, generator=g)
    x = torch.zeros(B, n, dtype=torch.float64, device=dev)
    status = torch.empty(B, dtype=torch.int32, device=dev); iters = torch.empty(B, dtype=torch.int32, device=dev)
    ms = _timed(torch, lambda: eng.solve_box_qp_batched_device(P, q, l, u, x, status, iters), 3)
    lower = n * (n + 1) // 2 * 8 + 4 * n * 8 + 4
    out["c5a_boxqp_n64_f64"] = {"value": B / ms * 1e3, "unit": "QP/s per GPU", "batch": B, "n": n, "ms": ms,
                                "frac_solved": float((status == 0).double().mean().item()),
                                "mean_boxcqp_iterations": float(iters.double().mean().item()),
                                "active_fraction": float(((x == l) | (x == u)).double().mean().item()),
                                "algorithmic_GBps": B * lower / ms / 1e6}
    del P
    return out


def secondary_c4(torch, dist, eng, dev, workloads, sharding, rank, world, m=4_000_000):
    """configs[3]: ONE problem, m = 4M residuals, n = 128, analytic Jacobian, rows sharded over all ranks; per accepted
    step one NCCL all-reduce of [lower(J'J) | J'r] (8,384 doubles), per pass one 1-double all-reduce.  Strong scaling."""
    comm = None
    if world > 1:
        comm = eng.nccl_comm_init(world, sharding.exchange_unique_id(eng, dist, rank), rank)
    lo, hi = sharding.row_shard(m, rank, world)
    wl = workloads.c4_gaussmix(m=m, row_slice=(lo, hi))
    t = torch.from_numpy(wl.t).to(dev); y = torch.from_numpy(wl.y).to(dev)
    st = eng.settings(np.float64)
    best = None
    for rep in range(3):
        x = wl.x0[0].copy()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(); t0 = time.perf_counter()
        r, stats = eng.optimize_sharded(st, wl.model, x, wl.l, wl.u, t, y, comm=comm, want_stats=True)
        torch.cuda.synchronize(); dt = time.perf_counter() - t0
        if world > 1:
            tt = torch.tensor([dt], dtype=torch.float64, device=dev)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            dt = float(tt.item())
        if rep > 0 and (best is None or dt < best[0]):
            best = (dt, r, stats, x)
    dt, r, stats, x = best
    out = {"value": r.iterations / dt, "unit": "LM iterations/s (whole job)", "m": m, "n": wl.n, "rows_per_rank": hi - lo,
           "solve_s": dt, "iterations": int(r.iterations), "passes": int(stats["passes"]), "passes_per_s": stats["passes"] / dt,
           "ms_per_pass": dt / max(int(stats["passes"]), 1) * 1e3, "ms_per_accepted_iteration": dt / max(int(r.iterations), 1) * 1e3,
           "allreduces_per_pass": 0 if world == 1 else 2,
           "status": int(r.status), "fCalls": int(r.fCalls), "gCalls": int(r.gCalls), "residual": float(r.residual),
           "max_rel_err_vs_truth": float(np.max(np.abs(x - wl.truth[0]) / np.abs(wl.truth[0]))),
           "timing": "wall clock around the blocking C-ABI call, device-synchronised, max over ranks, best of 2 after 1 warm-up",
           "collective": "none (1 GPU)" if world == 1 else f"NCCL all-reduce over {world} ranks, 67 KB per accepted step + 8 B per pass"}
    del t, y
    if comm is not None:
        eng.nccl_comm_destroy(comm)
    if rank == 0:
        # the dominant kernel of this path alone: J'J of this rank's rows on the FP64 tensor pipe (DMMA), J >> L2
        rows = ((hi - lo) + 31) // 32 * 32
        n = wl.n
        J = torch.randn(rows, n + (n & 1), dtype=torch.float64, device=dev)
        packed = torch.empty(n * (n + 1) // 2, dtype=torch.float64, device=dev)
        ms = _timed(torch, lambda: eng.syrk_lower_device(J, n, packed), 5)
        dmma = eng.lib.mir_b200_measure_peak_tflops(1, 5)
        ach = rows * n * (n + 1) / ms / 1e9
        out["roofline"] = {"bound": "tensor", "kernel": "syrk_dmma_kernel (FP64 mma.sync m8n8k4, TMA-fed)", "achieved": ach, "peak": dmma,
                           "unit": "TFLOP/s", "frac": ach / dmma if dmma > 0 else None,
                           "peak_source": "FP64 DMMA pipe measured live by mir_b200_measure_peak_tflops(1)",
                           "algorithmic_flops_per_launch": rows * n * (n + 1), "kernel_ms": ms, "rows": rows,
                           "J_read_GBps": rows * J.shape[1] * 8 / ms / 1e6}
        del J
    return out


def secondary_cpu_baselines(workloads, c4_m=4_000_000):
    """The CPU oracle (restated reference + real LAPACK/CBLAS from OpenBLAS) on bounded samples of the secondary configs,
    all host cores, timed on this box in the same run (rank 0, N = 1 only).  Reported baselines, not targets."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from conftest import load_oracle
    from oracle_util import oracle_batched, oracle_batched_mp, oracle_box_qp_batched_mp
    from mir_optim_b200.api import ReferenceAPI
    lib = load_oracle(); api = ReferenceAPI(lib)
    cores = os.cpu_count() or 1
    out = {}
    for name, dt in (("c3_sumexp8_f64", np.float64), ("c3_sumexp8_f32", np.float32)):
        n_s = 2048
        wl = workloads.c3_sumexp8(n_s, dtype=dt, seed=3)
        t0 = time.perf_counter()
        _, res, procs = oracle_batched_mp(lib, api.settings(dt), wl.model, wl.x0, wl.l, wl.u, t=wl.t, y=wl.y, fd_jacobian=True)
        secs = time.perf_counter() - t0
        out[name] = {"value": n_s / secs, "unit": "fits/s", "cores": procs, "kind": "port",
                     "sample": f"{n_s} fits of the same generator ({secs:.1f} s), one forked single-threaded-OpenBLAS worker per core",
                     "frac_status_ok": float(np.mean(res["status"] >= 0))}
    n_b = 16384
    wl = workloads.c2_gauss4(n_b, noise=0.05, tight_bounds=True, seed=7)
    t0 = time.perf_counter()
    _, res, procs = oracle_batched_mp(lib, api.settings(np.float64), wl.model, wl.x0, wl.l, wl.u, t=wl.t, y=wl.y)
    secs = time.perf_counter() - t0
    out["c5b_gauss4_active_bounds_f64"] = {"value": n_b / secs, "unit": "fits/s", "cores": procs, "kind": "port",
                                           "sample": f"{n_b} fits of the same generator ({secs:.1f} s), one forked single-threaded-OpenBLAS worker per core",
                                           "frac_status_ok": float(np.mean(res["status"] >= 0))}
    n_q = 8192
    wl = workloads.c5_boxqp(n_q, bound_scale=2.0)
    t0 = time.perf_counter()
    _, st, it, procs = oracle_box_qp_batched_mp(lib, wl.P, wl.q, wl.l, wl.u)
    secs = time.perf_counter() - t0
    out["c5a_boxqp_n64_f64"] = {"value": n_q / secs, "unit": "QP/s", "cores": procs, "kind": "port",
                                "sample": f"{n_q} QPs (n = 64, P = A'A/256 + 0.1 I, bounds +-U(0,2)) ({secs:.1f} s), one forked worker per core",
                                "mean_boxcqp_iterations": float(it.mean()), "frac_solved": float(np.mean(st == 0))}
    # configs[3]: ONE problem at the full size; OpenBLAS and the model callbacks use all cores.  Bounded by
    # maxIterations = 2 (the per-pass cost does not depend on the pass index: same J^T J, same rank-1 update, same evaluation)
    wl = workloads.c4_gaussmix(m=c4_m)
    s = api.settings(np.float64); s.maxIterations = 2
    lib.oracle_set_blas_threads(cores)
    lib.oracle_counters_reset()
    t0 = time.perf_counter()
    _, res, _ = oracle_batched(lib, s, wl.model, wl.x0, wl.l, wl.u, t=wl.t, y=wl.y.reshape(1, -1))
    secs = time.perf_counter() - t0
    lib.oracle_set_blas_threads(1)
    import ctypes as C
    p_ = C.c_ulonglong(); q_ = C.c_ulonglong()
    lib.oracle_counters(C.byref(p_), C.byref(q_))
    passes = max(int(p_.value), 1)
    out["c4_gaussmix_4Mx128_f64"] = {"value": int(res["iterations"][0]) / secs, "unit": "LM iterations/s", "cores": cores, "kind": "port",
                                     "passes_per_s": passes / secs, "passes": passes, "iterations": int(res["iterations"][0]),
                                     "sample": f"the same {c4_m} x 128 problem, first 2 accepted steps ({passes} passes, {secs:.1f} s): "
                                               f"OpenBLAS dsyrk/dgemv/dger with {cores} threads, model callbacks OpenMP over rows"}
    return out


def run_reference(args, rank, world):
    """`--impl reference`: the reference algorithm (CPU oracle: restated LM/BOXCQP + real LAPACK ?posvx from
    OpenBLAS; the D reference itself cannot be built here -- no D compiler) on all host cores."""
    if rank != 0:
        return
    from mir_optim_b200 import workloads
    cores = os.cpu_count() or 1
    wl = workloads.c2_gauss4(max(args.ref_sample, 1024), noise=0.05)
    rate, threads, _, _ = cpu_oracle_rate(wl, 4096)                      # calibration (untimed)
    sample = int(min(len(wl.x0), max(1024, rate * args.ref_step_seconds)))
    for _ in range(args.warmup):
        cpu_oracle_rate(wl, sample)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        cpu_oracle_rate(wl, sample)
    dt = time.perf_counter() - t0
    value = sample * args.steps / dt
    line = {"impl": "reference", "metric": "LM problems solved/sec (batched)", "value": value, "unit": "fits/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": WORKLOAD, "batch_per_step": sample, "m": M, "n": N},
            "cpu_baseline": {"value": value, "unit": "fits/s", "cores": threads, "kind": "port",
                             "sample": f"{sample} of the 2^20 fits per step, one forked worker process per core over problems, OpenBLAS 1 thread/worker; host has {cores} logical cores"},
            "e2e": {"value": value, "unit": "fits/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    _emit(line)


_REAL_STDOUT = None


def _own_stdout():
    """stdout carries exactly ONE JSON line: anything libraries print to fd 1 meanwhile (e.g. NCCL's version banner)
    is sent to stderr instead."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def _emit(line):
    sys.stdout.flush()
    os.write(_REAL_STDOUT if _REAL_STDOUT is not None else 1, (json.dumps(line) + "\n").encode())


def main():
    _own_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=1 << 20, help="fits per GPU per step (weak scaling)")
    ap.add_argument("--noise", type=float, default=0.05)
    ap.add_argument("--cpu-sample", type=int, default=32768)
    ap.add_argument("--ref-sample", type=int, default=65536)
    ap.add_argument("--ref-step-seconds", type=float, default=3.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip the configs[2]/[3]/[4] measurements")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the parameters and Result fields of the last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 0)

    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    import mir_optim_b200 as mo
    from mir_optim_b200 import workloads

    if not torch.cuda.is_available() or mo.engine.device_count() == 0:
        raise SystemExit("bench.py: no CUDA device; this engine has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(v):
        if world == 1:
            return v
        t = torch.tensor([v], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    eng = mo.engine
    B = args.batch
    wl = workloads.c2_gauss4(B, noise=args.noise, seed=2 + rank)          # independent problems: no data-path collective
    settings = eng.settings(np.float64)

    # ---------------- device-resident arm ----------------
    t_d = torch.from_numpy(wl.t).to(dev); y_d = torch.from_numpy(wl.y).to(dev)
    x0_d = torch.from_numpy(wl.x0).to(dev); x_d = torch.empty_like(x0_d)
    l_d = torch.from_numpy(wl.l).to(dev); u_d = torch.from_numpy(wl.u).to(dev)
    res_d = torch.empty(B * 32, dtype=torch.uint8, device=dev)
    stats_d = torch.zeros(8, dtype=torch.int64, device=dev)

    def step_resident():
        x_d.copy_(x0_d)
        eng.optimize_batched_device(settings, wl.model, x_d, l_d, u_d, t=t_d, y=y_d, results=res_d, stats=stats_d)

    for _ in range(args.warmup):
        step_resident()
    barrier()
    stats_d.zero_()
    launches0 = eng.kernel_launches()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ev0 = torch.cuda.Event(enable_timing=True); ev1 = torch.cuda.Event(enable_timing=True)
    kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    ev0.record()
    for i in range(args.steps):
        x_d.copy_(x0_d)
        kev[i][0].record()
        eng.optimize_batched_device(settings, wl.model, x_d, l_d, u_d, t=t_d, y=y_d, results=res_d, stats=stats_d)
        kev[i][1].record()
    ev1.record()
    barrier()
    elapsed_ms = max_over_ranks(ev0.elapsed_time(ev1))
    kernel_ms = float(np.mean([a.elapsed_time(b) for a, b in kev]))
    launches = eng.kernel_launches() - launches0
    clocks = sampler.stop() if rank == 0 else None
    stats = dict(zip(("problems", "passes", "accepted", "fresh_jacobians", "broyden_updates", "model_evals", "qp_solves",
                      "qp_iterations"), (int(v) for v in stats_d.cpu().tolist())))
    value = world * B * args.steps / (elapsed_ms * 1e-3)
    res_host = eng.results_from_bytes(res_d, np.float64)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, x_d.cpu().numpy(), res_host)
    assert np.all(res_host["status"] >= 0), "a fit failed"

    # ---------------- end-to-end arm: pinned host buffers through the host-pointer C ABI ----------------
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
    t_h, y_h, x0_h, l_h, u_h = pin(wl.t), pin(wl.y), pin(wl.x0), pin(wl.l), pin(wl.u)
    x_h = torch.empty_like(x0_h).pin_memory()
    from mir_optim_b200.engine import RESULT_DTYPES
    res_pin = torch.empty(B * 32, dtype=torch.uint8).pin_memory()              # the Result PODs land in pinned memory too
    res_view = res_pin.numpy().view(RESULT_DTYPES[np.dtype(np.float64)])
    e2e_t = 0.0
    res_e2e = None
    for i in range(2 + args.steps):
        x_h.copy_(x0_h)
        barrier()
        t0 = time.perf_counter()
        res_e2e, _ = eng.optimize_batched(settings, wl.model, x_h.numpy(), l_h.numpy(), u_h.numpy(), t=t_h.numpy(), y=y_h.numpy(),
                                          device=local_rank, results=res_view)
        dt = time.perf_counter() - t0
        if i >= 2:
            e2e_t += max_over_ranks(dt)
    e2e_value = world * B * args.steps / e2e_t
    h2d = wl.t.nbytes + wl.y.nbytes + wl.x0.nbytes + wl.l.nbytes + wl.u.nbytes
    d2h = wl.x0.nbytes + res_e2e.nbytes
    assert np.array_equal(res_e2e, res_host) and np.array_equal(x_h.numpy(), x_d.cpu().numpy()), "e2e and resident paths disagree"

    # ---------------- the other named configs (reported under "secondary"; every rank takes part) ----------------
    secondary = None
    if not args.no_secondary:
        del t_d, y_d, x0_d, x_d, res_d
        torch.cuda.empty_cache()
        secondary = {}
        try:
            sec = secondary_batched(torch, eng, dev, workloads, rank)
            for k, v in sec.items():                 # whole-job value = sum over ranks (independent problems, no collective)
                tot = v["value"]
                if world > 1:
                    tt = torch.tensor([tot], dtype=torch.float64, device=dev)
                    dist.all_reduce(tt)
                    tot = float(tt.item())
                v["value_per_gpu_rank0"] = v["value"]; v["value"] = tot; v["unit"] = v["unit"].replace(" per GPU", " (whole job)")
            secondary.update(sec)
        except Exception as e:                       # noqa: BLE001 -- the headline line must still be printed
            secondary["batched_error"] = repr(e)
        try:
            from mir_optim_b200 import sharding
            secondary["c4_gaussmix_4Mx128_f64"] = secondary_c4(torch, dist if world > 1 else None, eng, dev, workloads, sharding, rank, world)
        except Exception as e:                       # noqa: BLE001
            secondary["c4_error"] = repr(e)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---------------- roofline ----------------
    peaks, peak_src = measured_peaks()
    dfma_peak = eng.lib.mir_b200_measure_peak_tflops(0, 5)
    flops_per_launch = algorithmic_flops(stats) / args.steps
    ach_tf = flops_per_launch / (kernel_ms * 1e-3) / 1e12
    ach_gbs = ALGO_BYTES_PER_FIT * B / (kernel_ms * 1e-3) / 1e9
    roofline = {
        "bound": "fp64_fma",
        "kernel": ("lm_tpp_kernel<ModelGauss4<double>, double, analytic J, v-list> (one thread per fit)" if B >= 16384
                   else "lm_small_kernel<ModelGauss4<double>, double, 8 lanes per fit>"),
        "achieved": ach_tf, "peak": dfma_peak, "unit": "TFLOP/s", "frac": ach_tf / dfma_peak if dfma_peak > 0 else None,
        "peak_source": "DFMA pipe measured live by mir_b200_measure_peak_tflops(0)",
        "traffic": None,
        "algorithmic_flops_per_launch": flops_per_launch, "kernel_ms": kernel_ms,
        "hbm": {"bound": "hbm", "achieved": ach_gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": ach_gbs / peaks["hbm_gbs"],
                "algorithmic_bytes_per_fit": ALGO_BYTES_PER_FIT, "peak_source": peak_src,
                "note": "608 B/fit against ~1e5 flop/fit: the path is FP64-pipe/latency bound, not HBM bound (SURVEY 8d)"},
        "work_per_fit": {k: v / (B * args.steps) for k, v in stats.items() if k != "problems"},
    }
    prof = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.exists(prof):
        with open(prof) as f:
            roofline["traffic"] = json.load(f).get("lm_tpp_gauss4_1Mfits_dram_bytes_per_launch")
            roofline["traffic_note"] = "dram__bytes_read.sum + dram__bytes_write.sum of one 2^20-fit launch (ncu --set full), profiles/"

    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        sample = min(args.cpu_sample, B)
        rate, threads, secs, ro = cpu_oracle_rate(wl, sample)
        cpu = {"value": rate, "unit": "fits/s", "cores": threads, "kind": "port",
               "sample": f"first {sample} of the {B} fits of one step ({secs:.1f} s), one forked worker process per core over problems, OpenBLAS 1 thread/worker, "
                         f"host has {os.cpu_count()} logical cores; oracle = restated least_squares.d:877-1176 + real LAPACK dposvx"}

    if secondary is not None and world == 1 and not args.no_cpu_baseline:
        try:
            for k, v in secondary_cpu_baselines(workloads).items():
                if k in secondary:
                    secondary[k]["cpu_baseline"] = v
        except Exception as e:                       # noqa: BLE001
            secondary["cpu_baseline_error"] = repr(e)

    line = {"metric": "LM problems solved/sec (batched)", "value": value, "unit": "fits/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": elapsed_ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": WORKLOAD, "batch_per_gpu": B, "m": M, "n": N, "noise_sigma": args.noise,
                       "l2": f"inputs larger than L2: {wl.y.nbytes / 2**20:.0f} MiB of samples per GPU per step vs 126 MB L2",
                       "parallelism": f"{world} GPU(s), problems split evenly, no collective"},
            "e2e": {"value": e2e_value, "unit": "fits/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "ms_per_step": e2e_t / args.steps * 1e3},
            "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu, "secondary": secondary}
    _emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
