"""Time of the resident prediction (mir_b200_predict_batched_dev_*) next to the resident fit and covariance it follows,
on the shape of configs[1] (2^20 Gauss4 fits, m = 64, double; prediction at k = 64 and k = 256 abscissae) and a Gaussian
mixture with n = 11 (3 peaks + linear baseline, 2^16 problems, k = 200).  CUDA events around each call; the arms
(fit, covariance, each prediction) alternate for --reps repetitions after a warm-up of every shape.  Writes one JSON
document (stdout and --out) with the card's name and power limit.  Needs a CUDA device.

usage: python scripts/predict_timing.py [--reps 5] [--out predict_timing.json]"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

from cov_timing import card, tiled  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    import mir_optim_b200 as mo
    from mir_optim_b200 import ModelId, workloads
    assert torch.cuda.is_available(), "predict_timing.py needs a CUDA device"
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
        ("configs[1] gauss4 f64", tiled(workloads.c2_gauss4(65536), 1 << 20), np.float64, (64, 256), (-4.0, 4.0)),
        ("gaussmix n=11 f64", tiled(gm, 1 << 16), np.float64, (200,), (0.0, 1.0)),
    ]
    out = {"card": card(), "reps": a.reps,
           "timing": "CUDA events around one resident call each; fit, covariance and the predictions alternating", "shapes": []}
    for name, wl, dt, ks, span in shapes:
        wl = workloads.Workload(wl)
        s = eng.settings(dt)
        t, y, l, u = T(wl.t.astype(dt)), T(wl.y.astype(dt)), T(wl.l.astype(dt)), T(wl.u.astype(dt))
        x0 = T(wl.x0.astype(dt))
        batch, n = wl.x0.shape
        x = x0.clone()
        cov = torch.empty((batch, n, n), dtype=x.dtype, device=dev)
        sd = torch.empty((batch, n), dtype=x.dtype, device=dev)
        info = torch.empty(batch, dtype=torch.int32, device=dev)
        ts = {k: T(np.linspace(span[0], span[1], k).astype(dt)) for k in ks}
        val = {k: torch.empty((batch, k), dtype=x.dtype, device=dev) for k in ks}
        se = {k: torch.empty((batch, k), dtype=x.dtype, device=dev) for k in ks}

        def run_fit():
            x.copy_(x0)
            eng.optimize_batched_device(s, wl.model, x, l, u, t=t, y=y, fd_jacobian=wl.fd_jacobian)

        def run_cov():
            eng.covariance_batched_device(s, wl.model, x, l, u, t=t, y=y, fd_jacobian=wl.fd_jacobian, cov=cov, stddev=sd, info=info)

        def run_pred(k):
            return lambda: eng.predict_batched_device(s, wl.model, x, l, u, t=ts[k], cov=cov, fd_jacobian=wl.fd_jacobian,
                                                      value=val[k], se=se[k])

        arms = [("fit", run_fit), ("cov", run_cov)] + [(f"predict_k{k}", run_pred(k)) for k in ks]
        for _, fn in arms:                                                   # warm-up: modules, pools
            fn()
        torch.cuda.synchronize()
        ms = {nm: [] for nm, _ in arms}
        for _ in range(a.reps):
            for nm, fn in arms:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(); fn(); e1.record(); torch.cuda.synchronize()
                ms[nm].append(e0.elapsed_time(e1))
        inf = info.cpu().numpy()
        rec = {"shape": name, "batch": batch, "m": int(wl.y.shape[1]), "n": n, "dtype": np.dtype(dt).name, "fd": bool(wl.fd_jacobian),
               "ms": ms, "ms_median": {nm: float(np.median(v)) for nm, v in ms.items()},
               "predict_over_fit": {nm: float(np.median(v) / np.median(ms["fit"])) for nm, v in ms.items() if nm.startswith("predict")},
               "info_counts": {str(k): int(v) for k, v in zip(*np.unique(inf, return_counts=True))},
               "se_finite": {f"k{k}": bool(torch.isfinite(se[k][torch.from_numpy(inf == 0).to(dev)]).all()) for k in ks}}
        out["shapes"].append(rec)
        print(json.dumps(rec), flush=True)
    text = json.dumps(out, indent=1)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        open(a.out, "w").write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
