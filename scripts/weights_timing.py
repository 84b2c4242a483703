"""Cost of per-observation weights (MIR_MODEL_WEIGHTED) in the resident entry points, with CUDA events around one call each:
  * configs[1] (2^20 Gauss4 fits, m = 64, double) in three arms that alternate: unweighted (the thread-per-problem
    kernel), all-ones weights and weights 1/sigma_i (both on the general CTA-per-problem kernel, where weights run);
  * a Gaussian mixture with n = 11 (3 peaks + linear baseline, 2^16 problems, m = 200), weighted against unweighted --
    both on the general kernel, so the difference is the cost of the multiply and the weight loads alone;
  * the resident weighted covariance against the unweighted one on the same two shapes.
Every shape is warmed up first.  Writes one JSON document (stdout and --out) with the card's name and power limit.
Needs a CUDA device.

usage: python scripts/weights_timing.py [--reps 5] [--out weights_timing.json]"""
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
    assert torch.cuda.is_available(), "weights_timing.py needs a CUDA device"
    eng = mo.engine
    dev = torch.device("cuda:0")
    T = lambda v: torch.from_numpy(np.ascontiguousarray(v)).to(dev)        # noqa: E731

    rng = np.random.default_rng(21)
    tg = np.linspace(0.0, 1.0, 200)
    base = np.array([1.0, 0.25, 0.06, 0.7, 0.5, 0.05, 1.2, 0.75, 0.07, 0.2, -0.1])
    xm = np.tile(base, (4096, 1)); xm[:, 0:9:3] *= rng.uniform(0.8, 1.2, (4096, 3))
    ym = xm[:, 9:10] + xm[:, 10:11] * tg
    for k in range(3):
        ym = ym + xm[:, 3 * k:3 * k + 1] * np.exp(-0.5 * ((tg - xm[:, 3 * k + 1:3 * k + 2]) / xm[:, 3 * k + 2:3 * k + 3]) ** 2)
    ym = ym + 0.01 * rng.standard_normal(ym.shape)
    gm = workloads.Workload(model=ModelId.GAUSSMIX, t=tg, y=ym, x0=xm * 1.03, l=np.full(11, -np.inf), u=np.full(11, np.inf), fd_jacobian=False)

    shapes = [("configs[1] gauss4 f64", tiled(workloads.c2_gauss4(65536), 1 << 20)), ("gaussmix n=11 f64", tiled(gm, 1 << 16))]
    out = {"card": card(), "reps": a.reps, "timing": "CUDA events around one resident call each, arms alternating", "shapes": []}
    for name, wl in shapes:
        wl = workloads.Workload(wl)
        s = eng.settings(np.float64)
        t, y, l, u, x0 = (T(v.astype(np.float64)) for v in (wl.t, wl.y, wl.l, wl.u, wl.x0))
        batch, n = wl.x0.shape
        m = wl.y.shape[1]
        sigma = 10.0 ** np.random.default_rng(5).uniform(-1.0, 0.0, (batch, m))
        arms = {"unweighted": None, "ones": T(np.ones((batch, m))), "inv_sigma": T(1.0 / sigma)}
        if "gaussmix" in name:
            del arms["ones"]
        x = x0.clone()
        cov = torch.empty((batch, n, n), dtype=x.dtype, device=dev)
        sd = torch.empty((batch, n), dtype=x.dtype, device=dev)
        info = torch.empty(batch, dtype=torch.int32, device=dev)
        res = torch.empty(batch * 32, dtype=torch.uint8, device=dev)
        calls = {}
        for arm, w in arms.items():
            def fit(w=w):
                x.copy_(x0)
                eng.optimize_batched_device(s, wl.model, x, l, u, t=t, y=y, w=w, results=res)
            calls[f"fit_{arm}"] = fit
            if arm != "ones":
                def covariance(w=w):
                    eng.covariance_batched_device(s, wl.model, x, l, u, t=t, y=y, w=w, cov=cov, stddev=sd, info=info)
                calls[f"cov_{arm}"] = covariance
        for fn in calls.values():                                              # warm-up: modules, pools
            fn()
        torch.cuda.synchronize()
        ms = {k: [] for k in calls}
        for _ in range(a.reps):
            for k, fn in calls.items():
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(); fn(); e1.record(); torch.cuda.synchronize()
                ms[k].append(e0.elapsed_time(e1))
        rec = {"shape": name, "batch": batch, "m": m, "n": n, "dtype": "float64", "ms": ms,
               "ms_median": {k: float(np.median(v)) for k, v in ms.items()},
               "fits_per_s_median": {k: batch / (float(np.median(v)) * 1e-3) for k, v in ms.items() if k.startswith("fit_")}}
        out["shapes"].append(rec)
        print(json.dumps(rec), flush=True)
    text = json.dumps(out, indent=1)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        open(a.out, "w").write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
