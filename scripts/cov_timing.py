"""Time of the resident covariance (mir_b200_covariance_batched_dev_*) next to the resident fit it follows, on the
shapes of configs[1] (2^20 Gauss4 fits, double), configs[2] (2^20 sum-of-4-exponentials fits, FD, double and float) and
a Gaussian mixture with n = 11 (3 peaks + linear baseline, 2^16 problems).  CUDA events around each call; the fit and
the covariance alternate for --reps repetitions after a warm-up of every shape.  Writes one JSON document (stdout and
--out) with the card's name and power limit.  Needs a CUDA device.

usage: python scripts/cov_timing.py [--reps 5] [--out cov_timing.json]"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = [s.strip() for s in q.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:                                  # (the name from torch is still recorded)
        import torch
        return {"name": torch.cuda.get_device_name(0), "power_limit": f"unknown ({e})", "max_sm_clock": "unknown"}


def tiled(wl, batch):
    """The workload's problems repeated up to `batch` (every problem does the same work as in a fresh draw)."""
    k = -(-batch // len(wl.y))
    out = dict(wl)
    out["y"] = np.tile(wl.y, (k, 1))[:batch]; out["x0"] = np.tile(wl.x0, (k, 1))[:batch]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    import mir_optim_b200 as mo
    from mir_optim_b200 import ModelId, workloads
    assert torch.cuda.is_available(), "cov_timing.py needs a CUDA device"
    eng = mo.engine
    dev = torch.device("cuda:0")
    T = lambda v: torch.from_numpy(np.ascontiguousarray(v)).to(dev)

    rng = np.random.default_rng(21)
    tg = np.linspace(0.0, 1.0, 200)
    base = np.array([1.0, 0.25, 0.06, 0.7, 0.5, 0.05, 1.2, 0.75, 0.07, 0.2, -0.1])
    xm = np.tile(base, (4096, 1)); xm[:, 0:9:3] *= rng.uniform(0.8, 1.2, (4096, 3))
    ym = xm[:, 9:10] + xm[:, 10:11] * tg
    for k in range(3):
        ym = ym + xm[:, 3 * k:3 * k + 1] * np.exp(-0.5 * ((tg - xm[:, 3 * k + 1:3 * k + 2]) / xm[:, 3 * k + 2:3 * k + 3]) ** 2)
    ym = ym + 0.01 * rng.standard_normal(ym.shape)
    gm = workloads.Workload(model=ModelId.GAUSSMIX, t=tg, y=ym, x0=xm * 1.03, l=np.full(11, -np.inf), u=np.full(11, np.inf), fd_jacobian=False)

    shapes = [
        ("configs[1] gauss4 f64", tiled(workloads.c2_gauss4(65536), 1 << 20), np.float64),
        ("configs[2] sumexp8 f64", tiled(workloads.c3_sumexp8(65536), 1 << 20), np.float64),
        ("configs[2] sumexp8 f32", tiled(workloads.c3_sumexp8(65536), 1 << 20), np.float32),
        ("gaussmix n=11 f64", tiled(gm, 1 << 16), np.float64),
    ]
    out = {"card": card(), "reps": a.reps, "timing": "CUDA events around one resident call each, fit and covariance alternating",
           "shapes": []}
    for name, wl, dt in shapes:
        wl = workloads.Workload(wl)
        s = eng.settings(dt)
        t, y, l, u = T(wl.t.astype(dt)), T(wl.y.astype(dt)), T(wl.l.astype(dt)), T(wl.u.astype(dt))
        x0 = T(wl.x0.astype(dt))
        batch, n = wl.x0.shape
        x = x0.clone()
        cov = torch.empty((batch, n, n), dtype=x.dtype, device=dev)
        sd = torch.empty((batch, n), dtype=x.dtype, device=dev)
        info = torch.empty(batch, dtype=torch.int32, device=dev)

        def run_fit():
            x.copy_(x0)
            eng.optimize_batched_device(s, wl.model, x, l, u, t=t, y=y, fd_jacobian=wl.fd_jacobian)

        def run_cov():
            eng.covariance_batched_device(s, wl.model, x, l, u, t=t, y=y, fd_jacobian=wl.fd_jacobian, cov=cov, stddev=sd, info=info)

        run_fit(); run_cov(); torch.cuda.synchronize()                       # warm-up: modules, pools
        fit_ms, cov_ms = [], []
        for _ in range(a.reps):
            for fn, acc in ((run_fit, fit_ms), (run_cov, cov_ms)):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(); fn(); e1.record(); torch.cuda.synchronize()
                acc.append(e0.elapsed_time(e1))
        inf = info.cpu().numpy()
        rec = {"shape": name, "batch": batch, "m": int(wl.y.shape[1]), "n": n, "dtype": np.dtype(dt).name, "fd": bool(wl.fd_jacobian),
               "fit_ms": fit_ms, "cov_ms": cov_ms, "fit_ms_median": float(np.median(fit_ms)), "cov_ms_median": float(np.median(cov_ms)),
               "cov_over_fit": float(np.median(cov_ms) / np.median(fit_ms)),
               "info_counts": {str(k): int(v) for k, v in zip(*np.unique(inf, return_counts=True))}}
        out["shapes"].append(rec)
        print(json.dumps(rec), flush=True)
    text = json.dumps(out, indent=1)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        open(a.out, "w").write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
