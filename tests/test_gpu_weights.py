"""Per-observation weights (MIR_MODEL_WEIGHTED) on the B200: weighted fits and covariances of the general kernel against
the weighted host reference (tests/weights_util.py: the oracle LM with f~ = w (.) f), weights of one against the
unweighted general kernel bit for bit, zero-weight padding, scipy's curve_fit(sigma=...), user models, and the host
form against the device form."""
import os
import subprocess
import sys

import numpy as np
import pytest

import mir_optim_b200 as mo
from mir_optim_b200 import ModelId, workloads
from cov_util import cov_bound, cov_error, cov_reference
from oracle_util import rel_err
from test_gpu_cta_general import same_counters, sumexp
from test_gpu_covariance import GAUSS4_USER
from weights_util import oracle_batched_weighted, sigma_weights, weighted_callbacks

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
eng = mo.engine


def gaussmix(B, m, seed):
    """n = 3 K + 2 = 11: three Gaussians on a linear baseline, amplitudes capped so that some bounds are active."""
    rng = np.random.default_rng(seed)
    K = 3
    t = np.linspace(0.0, 1.0, m)
    truth = np.empty((B, 3 * K + 2))
    truth[:, 0:3 * K:3] = rng.uniform(1.0, 3.0, (B, K)); truth[:, 1:3 * K:3] = np.array([0.25, 0.5, 0.75]) + rng.uniform(-0.03, 0.03, (B, K))
    truth[:, 2:3 * K:3] = rng.uniform(0.05, 0.09, (B, K)); truth[:, -2] = rng.uniform(0, 1, B); truth[:, -1] = rng.uniform(-1, 1, B)
    y = truth[:, -2, None] + truth[:, -1, None] * t[None, :]
    for k in range(K):
        y = y + truth[:, 3 * k, None] * np.exp(-0.5 * ((t[None, :] - truth[:, 3 * k + 1, None]) / truth[:, 3 * k + 2, None]) ** 2)
    y = y + 1e-2 * rng.normal(size=y.shape)
    l = np.full(3 * K + 2, -np.inf); u = np.full(3 * K + 2, np.inf)
    l[0:3 * K:3] = 0.0; u[0:3 * K:3] = 2.5
    x0 = np.clip(truth * rng.uniform(0.95, 1.05, truth.shape), l, u)
    return dict(t=t, y=y, x0=x0, l=l, u=u)


def expdecay3(B, m, seed):
    rng = np.random.default_rng(seed)
    t = np.linspace(0.0, 5.0, m)
    truth = np.stack([rng.uniform(1, 3, B), rng.uniform(0.5, 1.5, B), rng.uniform(-0.5, 0.5, B)], axis=1)
    y = truth[:, 0, None] * np.exp(-truth[:, 1, None] * t[None, :]) + truth[:, 2, None] + 0.02 * rng.normal(size=(B, m))
    return dict(t=t, y=y, x0=truth * rng.uniform(0.8, 1.2, truth.shape), l=np.full(3, -np.inf), u=np.full(3, np.inf))


def spline_case(B, seed, lam=1e-3):
    rng = np.random.default_rng(seed)
    n, P = 10, 50
    knots = np.cumsum(rng.uniform(0.5, 1.5, n))
    t = np.sort(rng.uniform(knots[0] - 0.3, knots[-1] + 0.3, (B, P)), axis=1)
    y = 3.0 * np.sin(0.7 * t) + 0.1 * t + 0.05 * rng.normal(size=(B, P))
    return dict(t=t, y=y, x0=np.zeros((B, n)), l=np.full(n, -np.inf), u=np.full(n, np.inf), aux=knots, param=lam)


def gauss4(B, seed, per_problem_grid=False):
    wl = workloads.c2_gauss4(B, noise=0.05, seed=seed)
    t = wl.t
    if per_problem_grid:
        t = np.sort(np.random.default_rng(seed).uniform(-4.0, 4.0, (B, wl.m)), axis=1)
    return dict(t=t, y=wl.y, x0=wl.x0, l=wl.l, u=wl.u)


CASES = {
    "gauss4": (ModelId.GAUSS4, lambda: gauss4(160, 21), False, np.float64),
    "gauss4_fd": (ModelId.GAUSS4, lambda: gauss4(160, 22), True, np.float64),
    "gauss4_grid_per_problem": (ModelId.GAUSS4, lambda: gauss4(160, 23, per_problem_grid=True), False, np.float64),
    "expdecay3": (ModelId.EXPDECAY3, lambda: expdecay3(160, 90, 24), False, np.float64),
    "sumexp10": (ModelId.SUMEXP, lambda: sumexp(128, 5, 120, seed=25), False, np.float64),
    "gaussmix11_bounds": (ModelId.GAUSSMIX, lambda: gaussmix(96, 150, 26), False, np.float64),
    "spline_fd": (ModelId.SPLINE, lambda: spline_case(96, 27), True, np.float64),
    "gauss4_float": (ModelId.GAUSS4, lambda: gauss4(256, 28), False, np.float32),
}


@pytest.mark.parametrize("case", list(CASES))
def test_k_step_trajectories_against_the_weighted_oracle(oracle_lib, case):
    """k = 1, 2, 3 accepted steps with w = 1/sigma (sigma over a decade within a problem) and some zero rows: the same
    statuses and counters as the weighted reference for >= 99 % of problems, x and lambda to rounding."""
    model, make, fd, dt = CASES[case]
    d = make()
    B, m = d["y"].shape
    w = sigma_weights(B, m, seed=list(CASES).index(case), zero_rows=max(1, m // 16))
    args = {k: (v.astype(dt) if isinstance(v, np.ndarray) else v) for k, v in d.items() if k in ("t", "y", "aux", "param")}
    x0, l, u = d["x0"].astype(dt), d["l"].astype(dt), d["u"].astype(dt)
    for k in (1, 2, 3):
        s = eng.settings(dt); s.maxIterations = k
        xg = x0.copy()
        rg, stats = eng.optimize_batched(s, model, xg, l, u, fd_jacobian=fd, want_stats=True, w=w, **args)
        xo, ro = oracle_batched_weighted(oracle_lib, s, model, x0, l, u, w=w.astype(dt), fd_jacobian=fd, **args)
        same = same_counters(rg, ro)
        if dt == np.float32:                       # float trajectories may fork on a rounding-level accept / reject
            assert same.mean() > 0.97, (k, float(same.mean()))
            assert np.max(rel_err(xg[same], xo[same])) < 1e-4
            continue
        assert same.mean() >= 0.99, (k, float(same.mean()))
        tol = (1e-8 if fd else 1e-10) * (1 if k < 3 else 10)
        assert np.max(rel_err(xg[same], xo[same])) < tol, (k, float(np.max(rel_err(xg[same], xo[same]))))
        assert np.max(rel_err(rg["lambda"][same], ro["lambda"][same])) < 1e-11
        assert np.max(rel_err(rg["residual"][same], ro["residual"][same])) < 1e-9
        assert stats["problems"] == B
        if model == ModelId.GAUSSMIX:
            assert np.all(xg >= l) and np.all(xg <= u) and np.any((xg == l) | (xg == u))


def test_unit_weights_are_bit_identical_to_the_unweighted_general_kernel():
    """w = 1 changes no bit: SUMEXP n = 10 (general kernel either way) in process; Gauss4 n = 4 against the unweighted
    general kernel (MIRB200_BATCH_KERNEL=cta) in a subprocess, since without weights that shape runs a specialised kernel."""
    d = sumexp(300, 5, 100, seed=31)
    s = eng.settings(np.float64); s.maxIterations = 6
    xa = d["x0"].copy(); ra, _ = eng.optimize_batched(s, ModelId.SUMEXP, xa, d["l"], d["u"], t=d["t"], y=d["y"])
    xb = d["x0"].copy(); rb, _ = eng.optimize_batched(s, ModelId.SUMEXP, xb, d["l"], d["u"], t=d["t"], y=d["y"], w=np.ones_like(d["y"]))
    assert xa.tobytes() == xb.tobytes() and ra.tobytes() == rb.tobytes()

    code = r'''
import sys, numpy as np
import mir_optim_b200 as mo
from mir_optim_b200 import workloads
eng = mo.engine
wl = workloads.c2_gauss4(2048, noise=0.05, seed=32)
out = {}
for dt in (np.float64, np.float32):
    s = eng.settings(dt); s.maxIterations = 8
    x = wl.x0.astype(dt).copy()
    kw = dict(w=np.ones(wl.y.shape)) if sys.argv[1] == "w" else {}
    r, _ = eng.optimize_batched(s, wl.model, x, wl.l.astype(dt), wl.u.astype(dt), t=wl.t.astype(dt), y=wl.y.astype(dt), **kw)
    out[dt.__name__] = (x.tobytes() + r.tobytes()).hex()
print(repr(out))
'''
    outs = {}
    for mode in ("w", "cta"):
        env = dict(os.environ, PYTHONPATH=ROOT)
        if mode == "cta":
            env["MIRB200_BATCH_KERNEL"] = "cta"
        p = subprocess.run([sys.executable, "-c", code, mode], capture_output=True, text=True, env=env, timeout=600)
        assert p.returncode == 0, p.stderr[-2000:]
        outs[mode] = p.stdout.strip().splitlines()[-1]
    assert outs["w"] == outs["cta"]


def test_zero_weight_padding_gives_the_unpadded_fit_and_covariance():
    """A problem padded from m to m + 37 rows with w = 0 (finite t, y on the padding) fits and has the covariance of the
    unpadded one, info = -1 at m_w <= n_F included."""
    wl = workloads.c2_gauss4(512, noise=0.05, seed=33)
    B, m, P = 512, wl.m, 37
    w = sigma_weights(B, m, seed=4)
    tp = np.concatenate([wl.t, np.linspace(5.0, 9.0, P)])
    yp = np.concatenate([wl.y, np.full((B, P), 1e3)], axis=1)
    wp = np.concatenate([w, np.zeros((B, P))], axis=1)
    for k in (3, 0):
        s = eng.settings(np.float64)
        if k:
            s.maxIterations = k
        xa = wl.x0.copy(); ra, _ = eng.optimize_batched(s, wl.model, xa, wl.l, wl.u, t=wl.t, y=wl.y, w=w)
        xb = wl.x0.copy(); rb, _ = eng.optimize_batched(s, wl.model, xb, wl.l, wl.u, t=tp, y=yp, w=wp)
        assert np.all(same_counters(ra, rb))
        assert np.max(rel_err(xa, xb)) < 1e-12 and np.max(rel_err(ra["residual"], rb["residual"])) < 1e-12
    for scaled in (True, False):
        ca, sa, ia = eng.covariance_batched(s, wl.model, xa, wl.l, wl.u, t=wl.t, y=wl.y, w=w, scaled=scaled)
        cb, sb, ib = eng.covariance_batched(s, wl.model, xa, wl.l, wl.u, t=tp, y=yp, w=wp, scaled=scaled)
        assert np.array_equal(ia, ib) and (ia == 0).mean() > 0.9
        assert cov_error(ca[ia == 0], cb[ia == 0]).max() < 1e-12
    # the degrees-of-freedom boundary: 4 informative rows and 4 free parameters -> -1; 5 -> 0, padded or not
    x = wl.truth[:8].copy(); big = np.full(4, 1e3)
    for rows, want in ((4, -1), (5, 0)):
        idx = np.linspace(10, 54, rows).astype(int)
        t1, y1, w1 = wl.t[idx], wl.y[:8, idx], w[:8, idx]
        tq = np.concatenate([t1, tp[m:]]); yq = np.concatenate([y1, yp[:8, m:]], axis=1); wq = np.concatenate([w1, wp[:8, m:]], axis=1)
        _, _, i1 = eng.covariance_batched(None, wl.model, x, -big, big, t=t1, y=y1, w=w1)
        c2, _, i2 = eng.covariance_batched(None, wl.model, x, -big, big, t=tq, y=yq, w=wq)
        assert np.all(i1 == want) and np.all(i2 == want), (rows, i1, i2)
        if want == -1:
            assert np.all(np.isinf(c2))


@pytest.mark.parametrize("dt", [np.float64, np.float32])
@pytest.mark.parametrize("fd", [False, True])
def test_weighted_covariance_against_the_reference(oracle_lib, dt, fd):
    """The definition with r~ and J~ over the rows with w != 0 (cov_util.cov_reference on the weighted callbacks, zero rows
    dropped: they add nothing to J^T J and ||r||^2 and leave m_w rows)."""
    wl = workloads.c2_gauss4(1024, noise=0.05, seed=34)
    w = sigma_weights(1024, wl.m, seed=5, zero_rows=6)
    s = eng.settings(dt)
    x = wl.x0.astype(dt).copy()
    eng.optimize_batched(s, wl.model, x, wl.l.astype(dt), wl.u.astype(dt), t=wl.t.astype(dt), y=wl.y.astype(dt), w=w, fd_jacobian=fd)
    for scaled in (True, False):
        cov, sd, info = eng.covariance_batched(s, wl.model, x, wl.l, wl.u, t=wl.t, y=wl.y, w=w, fd_jacobian=fd, scaled=scaled)
        fw, gw = weighted_callbacks(oracle_lib, wl.model, dt, wl.t, wl.y, w, fd=fd)
        keep = w != 0
        f = lambda b, p: fw(b, p)[keep[b]]                                                  # noqa: E731
        g = None if fd else (lambda b, p: gw(b, p)[keep[b]])
        ref, rinfo, kap = cov_reference(f, g, x, wl.l.astype(dt), wl.u.astype(dt), s.jacobianEpsilon, scaled=scaled)
        assert np.array_equal(info, rinfo)
        ok = rinfo == 0
        assert ok.mean() > 0.9
        bound = cov_bound(kap[ok], dt)
        assert np.all(cov_error(cov[ok], ref[ok]) <= bound), float(np.max(cov_error(cov[ok], ref[ok]) / bound))
        assert np.array_equal(cov, np.swapaxes(cov, 1, 2), equal_nan=True)


def test_weighted_covariance_matches_curve_fit_sigma():
    """With w = 1/sigma the scaled covariance is curve_fit(sigma=sigma, absolute_sigma=False)'s pcov and the unscaled one
    is absolute_sigma=True's, at the fitted point."""
    from scipy.optimize import curve_fit
    wl = workloads.c2_gauss4(6, noise=0.05, seed=35)
    w = sigma_weights(6, wl.m, seed=6, zero_rows=3)
    inf = np.full(4, np.inf)
    x = wl.x0.copy()
    eng.optimize_batched(eng.settings(), wl.model, x, -inf, inf, t=wl.t, y=wl.y, w=w)

    def f(t, A, mu, s, c):
        return A * np.exp(-0.5 * ((t - mu) / s) ** 2) + c

    def jac(t, A, mu, s, c):
        z = (t - mu) / s; e = np.exp(-0.5 * z * z)
        return np.stack([e, A * e * z / s, A * e * z * z / s, np.ones_like(t)], axis=1)

    for absolute in (False, True):
        cov, _, info = eng.covariance_batched(None, wl.model, x, -inf, inf, t=wl.t, y=wl.y, w=w, scaled=not absolute)
        assert np.all(info == 0)
        for b in range(6):
            k = w[b] != 0
            popt, pcov = curve_fit(f, wl.t[k], wl.y[b, k], p0=x[b], sigma=1.0 / w[b, k], absolute_sigma=absolute, jac=jac)
            np.testing.assert_allclose(popt, x[b], rtol=1e-6, atol=1e-9)
            np.testing.assert_allclose(cov[b], pcov, rtol=1e-6, atol=1e-6 * np.sqrt(np.outer(np.diag(pcov), np.diag(pcov))).max())


def test_weighted_user_model_matches_weighted_builtin():
    """A user model restating Gauss4 with the built-in operation sequence, weighted: the same k-step trajectories and
    covariance as the weighted built-in."""
    mid = eng.compile_model(GAUSS4_USER)
    try:
        wl = workloads.c2_gauss4(512, noise=0.05, seed=36)
        w = sigma_weights(512, wl.m, seed=7, zero_rows=4)
        for k in (1, 2, 3):
            s = eng.settings(np.float64); s.maxIterations = k
            xb = wl.x0.copy(); rb, _ = eng.optimize_batched(s, wl.model, xb, wl.l, wl.u, t=wl.t, y=wl.y, w=w)
            xu = wl.x0.copy(); ru, _ = eng.optimize_batched(s, mid, xu, wl.l, wl.u, t=wl.t, y=wl.y, w=w)
            assert np.array_equal(rb["status"], ru["status"]) and np.array_equal(rb["fCalls"], ru["fCalls"]) and np.array_equal(rb["iterations"], ru["iterations"])
            assert np.max(rel_err(xb, xu)) < 1e-12
        for scaled in (True, False):
            cb, _, ib = eng.covariance_batched(None, wl.model, xb, wl.l, wl.u, t=wl.t, y=wl.y, w=w, scaled=scaled)
            cu, _, iu = eng.covariance_batched(None, mid, xb, wl.l, wl.u, t=wl.t, y=wl.y, w=w, scaled=scaled)
            assert np.array_equal(ib, iu) and cov_error(cu[ib == 0], cb[ib == 0]).max() <= 1e-13
    finally:
        eng.release_model(mid)


# Declares CtaWeighted<CtaUser<UserModel<double>>> without defining it: every program of the model that instantiates the
# weighted adapter fails to compile, the unweighted ones are unaffected.
NO_WEIGHTED_DOUBLE = r"""
namespace mirb200 { template <> struct CtaWeighted<CtaUser<::UserModel<double>, double>, double>; }
"""


def test_weighted_user_programs_compile_at_first_weighted_use():
    """Registration and unweighted calls build no weighted program; a weighted fit and a weighted covariance build theirs
    at their first call (here they cannot compile, which makes the build visible), and the unweighted programs still run."""
    from mir_optim_b200.engine import B200Error
    mid = eng.compile_model(GAUSS4_USER + NO_WEIGHTED_DOUBLE)         # (the double fit program is built at registration)
    try:
        wl = workloads.c2_gauss4(64, noise=0.05, seed=38)
        w = sigma_weights(64, wl.m, seed=9)
        s = eng.settings(np.float64); s.maxIterations = 3
        x = wl.x0.copy(); eng.optimize_batched(s, mid, x, wl.l, wl.u, t=wl.t, y=wl.y)
        eng.covariance_batched(None, mid, x, wl.l, wl.u, t=wl.t, y=wl.y)
        for call in (lambda: eng.optimize_batched(s, mid, wl.x0.copy(), wl.l, wl.u, t=wl.t, y=wl.y, w=w),
                     lambda: eng.covariance_batched(None, mid, x, wl.l, wl.u, t=wl.t, y=wl.y, w=w)):
            with pytest.raises(B200Error) as e:
                call()
            assert e.value.code == 2 and "does not compile" in str(e.value)
        xf = wl.x0.astype(np.float32)                                 # float: the weighted programs are unaffected
        eng.optimize_batched(eng.settings(np.float32), mid, xf, wl.l, wl.u, t=wl.t, y=wl.y, w=w)
    finally:
        eng.release_model(mid)


def test_host_form_equals_device_form_over_several_staging_chunks():
    """2^17 + 123 weighted problems: the host form (staged in chunks of 65536 problems) and the device form give the same
    bits, for the fit and the covariance."""
    import torch
    B = (1 << 17) + 123
    wl = workloads.c2_gauss4(B, noise=0.05, seed=37)
    w = sigma_weights(B, wl.m, seed=8, zero_rows=2)
    s = eng.settings(np.float64); s.maxIterations = 6
    xh = wl.x0.copy(); rh, _ = eng.optimize_batched(s, wl.model, xh, wl.l, wl.u, t=wl.t, y=wl.y, w=w)
    dev = torch.device("cuda")
    T = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)                            # noqa: E731
    xd = T(wl.x0)
    rd = eng.optimize_batched_device(s, wl.model, xd, T(wl.l), T(wl.u), t=T(wl.t), y=T(wl.y), w=T(w))
    torch.cuda.synchronize()
    assert xd.cpu().numpy().tobytes() == xh.tobytes()
    assert eng.results_from_bytes(rd, np.float64).tobytes() == rh.tobytes()
    ch, sh, ih = eng.covariance_batched(None, wl.model, xh, wl.l, wl.u, t=wl.t, y=wl.y, w=w)
    cd, sd, idv = eng.covariance_batched_device(None, wl.model, T(xh), T(wl.l), T(wl.u), t=T(wl.t), y=T(wl.y), w=T(w))
    torch.cuda.synchronize()
    assert cd.cpu().numpy().tobytes() == ch.tobytes() and idv.cpu().numpy().tobytes() == ih.tobytes()
