"""Batched prediction on the B200 (mir_b200_predict_batched_*): values bit for bit against the oracle's callbacks, the
standard error against the host reference of its definition (tests/predict_util.py) under its stated bound, identities
that need no host reference (the hat matrix, a linear model, the spread of refits), what is never read, determinism,
the host and device forms, resident chains, and user models."""
import ctypes as C

import numpy as np
import pytest

import mir_optim_b200 as mo
from mir_optim_b200 import ModelId, workloads
from mir_optim_b200._abi import ModelDesc, MODEL_WEIGHTED
from mir_optim_b200.engine import B200Error
from cov_util import fd_jacobian, oracle_callbacks
from predict_util import predict_callbacks, predict_reference, se_within_bound
from test_gpu_covariance import GAUSS4_USER, fit, gaussmix_workload
from user_models import LOGISTIC

pytestmark = pytest.mark.gpu

eng = mo.engine
DT = [np.float64, np.float32]

# p0 + p1 t + p2 t^2: a model linear in its parameters, with its Jacobian
POLY3 = r'''
template <class REAL> struct UserModel {
    static constexpr bool kAnalytic = true;
    __device__ static REAL residual(const REAL* p, int n, int m, int row, REAL t, REAL y, const REAL* aux, REAL param) {
        return (p[0] + p[1] * t + p[2] * t * t) - y;
    }
    __device__ static void jacobian(const REAL* p, int n, int m, int row, REAL t, REAL y, const REAL* aux, REAL param, REAL* J) {
        J[0] = 1; J[1] = t; J[2] = t * t;
    }
};
'''


def spd(rng, batch, n, scale=1e-2):
    A = rng.standard_normal((batch, n, n))
    return scale * (A @ np.swapaxes(A, 1, 2) + 0.1 * np.eye(n))


def value_cases(batch, seed):
    """model -> (x (batch, n), t* shared (k,), t* per problem (batch, k), aux or None)"""
    rng = np.random.default_rng(seed)
    k = 37
    out = {}
    g = workloads.c2_gauss4(batch, seed=seed)
    out["gauss4"] = (ModelId.GAUSS4, g.truth, np.linspace(-5.0, 5.0, k), rng.uniform(-5, 5, (batch, k)), None)
    x = np.column_stack([rng.uniform(1, 5, batch), rng.uniform(0.2, 2, batch), rng.uniform(-1, 1, batch)])
    out["expdecay3"] = (ModelId.EXPDECAY3, x, np.linspace(0.0, 10.0, k), rng.uniform(0, 10, (batch, k)), None)
    x = np.empty((batch, 10)); x[:, 0::2] = rng.uniform(1, 5, (batch, 5)); x[:, 1::2] = np.array([0.2, 0.6, 1.5, 4.0, 10.0]) * rng.uniform(0.8, 1.2, (batch, 5))
    out["sumexp10"] = (ModelId.SUMEXP, x, np.linspace(0.0, 5.0, k), rng.uniform(0, 5, (batch, k)), None)
    gm = gaussmix_workload(batch, seed=seed)
    out["gaussmix11"] = (ModelId.GAUSSMIX, gm.x0, np.linspace(-0.2, 1.2, k), rng.uniform(-0.2, 1.2, (batch, k)), None)
    n = 8
    knots = np.linspace(0.0, 10.0, n)
    out["spline"] = (ModelId.SPLINE, rng.uniform(-1, 1, (batch, n)), np.linspace(-0.5, 10.5, k), rng.uniform(-0.5, 10.5, (batch, k)), knots)
    pk = np.sort(knots[None, :] + np.concatenate([np.zeros((batch, 1)), rng.uniform(-0.3, 0.3, (batch, n - 2)), np.zeros((batch, 1))], axis=1), axis=1)
    out["spline_per_problem_knots"] = (ModelId.SPLINE, rng.uniform(-1, 1, (batch, n)), np.linspace(-0.5, 10.5, k), rng.uniform(-0.5, 10.5, (batch, k)), pk)
    return out


@pytest.mark.parametrize("dt", DT)
@pytest.mark.parametrize("per_problem_t", [False, True])
@pytest.mark.parametrize("case", ["gauss4", "expdecay3", "sumexp10", "gaussmix11", "spline", "spline_per_problem_knots", "gauss4_user"])
def test_values_bit_for_bit(oracle_lib, dt, per_problem_t, case):
    batch = 64
    cases = value_cases(batch, seed=41)
    model, x, ts, tp, aux = cases["gauss4" if case == "gauss4_user" else case]
    t = (tp if per_problem_t else ts).astype(dt)
    x = x.astype(dt)
    n = x.shape[1]
    inf = np.full(n, np.inf, dt)
    f, _, k = predict_callbacks(oracle_lib, model, dt, t, batch, aux=aux)
    ref, _, _ = predict_reference(f, None, x, -inf, inf, 0.0, None, k)
    mid = eng.compile_model(GAUSS4_USER) if case == "gauss4_user" else model
    try:
        v, se = eng.predict_batched(None, mid, x, -inf, inf, t=t, aux=aux)
        assert se is None
        assert v.dtype == dt and v.tobytes() == ref.tobytes(), np.max(np.abs(v - ref))
        if model == ModelId.SPLINE:                     # the smoothing weight does not enter the values
            v2, _ = eng.predict_batched(None, mid, x, -inf, inf, t=t, aux=aux, param=1e-3)
            assert v2.tobytes() == v.tobytes()
    finally:
        if case == "gauss4_user":
            eng.release_model(mid)


def own_grid_case(name, batch, rng):
    """(model, t (m,), y (batch, m), x0, l, u, aux) with y drawn from the model at a known truth"""
    m = 48
    if name == "expdecay2":
        t = np.linspace(0, 5, m); tr = np.column_stack([rng.uniform(1, 3, batch), rng.uniform(0.3, 1.5, batch)])
        clean = tr[:, :1] * np.exp(-t * tr[:, 1:2]); model = ModelId.EXPDECAY2
    elif name == "exptau3":
        t = np.linspace(0, 5, m); tr = np.column_stack([rng.uniform(1, 3, batch), rng.uniform(0.5, 2, batch), rng.uniform(-1, 1, batch)])
        clean = tr[:, :1] * np.exp(-t / tr[:, 1:2]) + tr[:, 2:3]; model = ModelId.EXPTAU3
    elif name == "expdecay3":
        t = np.linspace(0, 5, m); tr = np.column_stack([rng.uniform(1, 3, batch), rng.uniform(0.3, 1.5, batch), rng.uniform(-1, 1, batch)])
        clean = tr[:, :1] * np.exp(-tr[:, 1:2] * t) + tr[:, 2:3]; model = ModelId.EXPDECAY3
    elif name == "gauss4":
        g = workloads.c2_gauss4(batch, m=m, seed=int(rng.integers(1000)))
        return g.model, g.t, g.y, g.x0, g.l, g.u, None
    elif name == "sumexp":
        t = np.linspace(0, 5, m); tr = np.empty((batch, 6)); tr[:, 0::2] = rng.uniform(1, 3, (batch, 3)); tr[:, 1::2] = np.array([0.3, 1.0, 3.0]) * rng.uniform(0.9, 1.1, (batch, 3))
        clean = np.einsum("bk,bkm->bm", tr[:, 0::2], np.exp(-tr[:, 1::2, None] * t)); model = ModelId.SUMEXP
    else:
        g = gaussmix_workload(batch, m=m, seed=int(rng.integers(1000)))
        return g.model, g.t, g.y, g.x0, g.l, g.u, None
    y = clean + 0.01 * rng.standard_normal(clean.shape)
    inf = np.full(tr.shape[1], np.inf)
    return model, t, y, tr * 1.05, -inf, inf, None


@pytest.mark.parametrize("dt", DT)
@pytest.mark.parametrize("name", ["expdecay2", "exptau3", "expdecay3", "gauss4", "sumexp", "gaussmix", "spline"])
def test_values_on_the_fits_own_grid_are_its_residuals_plus_y(oracle_lib, dt, name):
    rng = np.random.default_rng(52)
    batch = 32
    if name == "spline":
        P, n = 40, 7
        px = np.sort(rng.uniform(0.0, 6.0, P)).astype(dt); knots = np.linspace(0.0, 6.0, n)
        py = (np.cos(px)[None, :] + 0.05 * rng.standard_normal((batch, P))).astype(dt)
        l = np.full(n, -5.0); u = np.full(n, 5.0)
        x, _ = eng.fit_spline_batched(eng.settings(dt), px, py, knots, l, u, 0.0)
        t = np.zeros(P + 1, dt); t[:P] = px
        y = np.zeros((batch, P + 1), dt); y[:, :P] = py
        f, _ = oracle_callbacks(oracle_lib, ModelId.SPLINE, dt, t, y, aux=knots, param=0.0, fd=True)
        v, _ = eng.predict_batched(None, ModelId.SPLINE, x, l, u, t=px, aux=knots)
        r = np.stack([f(b, x[b])[:P] for b in range(batch)])
        assert (v - py).astype(dt).tobytes() == r.tobytes()
        return
    model, t, y, x0, l, u, aux = own_grid_case(name, batch, rng)
    wl = workloads.Workload(model=model, t=t, y=y, x0=x0, l=l, u=u)
    s, x, _ = fit(wl, dt)
    f, _ = oracle_callbacks(oracle_lib, model, dt, t, y, fd=True)
    v, _ = eng.predict_batched(None, model, x, l, u, t=t.astype(dt))
    r = np.stack([f(b, x[b]) for b in range(batch)])
    assert (v - y.astype(dt)).astype(dt).tobytes() == r.tobytes()


def check_se(se, q, bound, dt):
    ok, worst = se_within_bound(se, q, bound, dt)
    assert ok, worst


@pytest.mark.parametrize("dt", DT)
@pytest.mark.parametrize("fd", [False, True])
def test_se_parity_gauss4(oracle_lib, dt, fd):
    wl = workloads.c2_gauss4(1024, dtype=dt)
    s, x, _ = fit(wl, dt, fd=fd)
    cov, _, info = eng.covariance_batched(s, wl.model, x, wl.l, wl.u, t=wl.t, y=wl.y, fd_jacobian=fd)
    ts = np.linspace(-4.5, 4.5, 41).astype(dt)
    v, se = eng.predict_batched(s, wl.model, x, wl.l, wl.u, t=ts, cov=cov, fd_jacobian=fd)
    f, g, k = predict_callbacks(oracle_lib, wl.model, dt, ts, 1024, fd=fd)
    ref, q, bound = predict_reference(f, g, x, wl.l.astype(dt), wl.u.astype(dt), s.jacobianEpsilon, cov, k)
    assert v.tobytes() == ref.tobytes()
    ok = info == 0
    assert ok.mean() > 0.99
    check_se(se[ok], q[ok], bound[ok], dt)


def test_se_parity_fd_near_a_bound(oracle_lib):
    # a free parameter within h of its bound: the central difference is clamped there, as in the fit (LS:1030-1047)
    wl = workloads.c2_gauss4(256)
    s, x, _ = fit(wl, np.float64, fd=True)
    eps = s.jacobianEpsilon
    l = np.tile(wl.l, (256, 1)); u = np.tile(wl.u, (256, 1))
    l[:, 3] = x[:, 3] - 0.25 * eps; u[:, 0] = x[:, 0] + 0.5 * eps
    cov, _, info = eng.covariance_batched(s, wl.model, x, l, u, t=wl.t, y=wl.y, fd_jacobian=True)
    assert np.all(info == 0)
    ts = np.linspace(-4.0, 4.0, 29)
    _, se = eng.predict_batched(s, wl.model, x, l, u, t=ts, cov=cov, fd_jacobian=True)
    f, _, k = predict_callbacks(oracle_lib, wl.model, np.float64, ts, 256, fd=True)
    _, q, bound = predict_reference(f, None, x, l, u, eps, cov, k)
    check_se(se, q, bound, np.float64)


def test_se_parity_gaussmix_n11_with_active_bounds(oracle_lib):
    wl = gaussmix_workload(128)
    s, x, _ = fit(wl, np.float64)
    cov, _, info = eng.covariance_batched(s, wl.model, x, wl.l, wl.u, t=wl.t, y=wl.y)
    fixed = (x == wl.u) | (x == wl.l)
    assert fixed[:, 3].mean() > 0.5
    ts = np.linspace(-0.1, 1.1, 45)
    for fd in (False, True):
        _, se = eng.predict_batched(s, wl.model, x, wl.l, wl.u, t=ts, cov=cov, fd_jacobian=fd)
        f, g, k = predict_callbacks(oracle_lib, wl.model, np.float64, ts, 128, fd=fd)
        _, q, bound = predict_reference(f, g, x, wl.l, wl.u, s.jacobianEpsilon, cov, k)
        ok = info == 0
        check_se(se[ok], q[ok], bound[ok], np.float64)


@pytest.mark.parametrize("per_problem_knots", [False, True])
def test_se_parity_spline_fd(oracle_lib, per_problem_knots):
    rng = np.random.default_rng(8)
    batch, P, n, lam = 32, 60, 8, 1e-3
    px = np.sort(rng.uniform(0.0, 10.0, P))
    py = np.sin(px)[None, :] + 0.05 * rng.standard_normal((batch, P))
    knots = np.linspace(0.0, 10.0, n)
    if per_problem_knots:
        knots = np.sort(knots[None, :] + np.concatenate([np.zeros((batch, 1)), rng.uniform(-0.2, 0.2, (batch, n - 2)), np.zeros((batch, 1))], axis=1), axis=1)
    l = np.full(n, -10.0); u = np.full(n, 10.0)
    s = eng.settings()
    vals, _ = eng.fit_spline_batched(s, px, py, knots, l, u, lam)
    cov, _, info = eng.covariance_batched(s, ModelId.SPLINE, vals, l, u, t=px, y=py, fd_jacobian=True, aux=knots, param=lam)
    assert np.all(info == 0)
    ts = np.linspace(-0.5, 10.5, 57)
    v, se = eng.predict_batched(s, ModelId.SPLINE, vals, l, u, t=ts, cov=cov, fd_jacobian=True, aux=knots, param=lam)
    f, g, k = predict_callbacks(oracle_lib, ModelId.SPLINE, np.float64, ts, batch, aux=knots)
    ref, q, bound = predict_reference(f, g, vals, l, u, s.jacobianEpsilon, cov, k)
    assert v.tobytes() == ref.tobytes()
    check_se(se, q, bound, np.float64)


def test_se_parity_user_model_without_jacobian():
    # LOGISTIC uses CUDA's exp, which numpy does not restate bit for bit: the reference's f is the device's own value
    # output at the (clamped) difference points, so the central difference and the quadratic form are checked exactly
    rng = np.random.default_rng(9)
    mid = eng.compile_model(LOGISTIC)
    try:
        t = np.linspace(0.0, 10.0, 80); batch = 16
        truth = np.column_stack([rng.uniform(4, 6, batch), rng.uniform(0.8, 1.2, batch), rng.uniform(4, 6, batch)])
        y = truth[:, :1] / (1 + np.exp(-truth[:, 1:2] * (t - truth[:, 2:3]))) + 0.02 * rng.standard_normal((batch, 80))
        l = np.array([0.0, 0.0, 0.0]); u = np.array([20.0, 5.0, 10.0])
        ts = np.linspace(-1.0, 11.0, 25)
        for dt in DT:
            s = eng.settings(dt)
            x = truth.astype(dt).copy()
            eng.optimize_batched(s, mid, x, l, u, t=t, y=y)
            cov, _, info = eng.covariance_batched(s, mid, x, l, u, t=t, y=y)
            assert np.all(info == 0)
            v, se = eng.predict_batched(s, mid, x, l, u, t=ts, cov=cov)
            fdev = lambda b, p: eng.predict_batched(s, mid, p[None, :].astype(dt), l, u, t=ts)[0][0]
            np.testing.assert_allclose(v, (x[:, :1] / (1 + np.exp(-x[:, 1:2] * (ts - x[:, 2:3])))).astype(dt),
                                       rtol=1e-12 if dt == np.float64 else 1e-5)
            _, q, bound = predict_reference(fdev, None, x, l.astype(dt), u.astype(dt), s.jacobianEpsilon, cov, len(ts))
            check_se(se, q, bound, dt)
    finally:
        eng.release_model(mid)


@pytest.mark.parametrize("weighted", [False, True])
def test_hat_matrix_identity(weighted):
    """At t* = t: sum_i w_i^2 se_i^2 = s^2 n_F with s^2 = Result.residual / (m_w - n_F) (w = 1 unweighted)."""
    batch = 512
    wl = workloads.c2_gauss4(batch, seed=61)
    rng = np.random.default_rng(62)
    w = None
    if weighted:
        w = 1.0 / rng.uniform(0.5, 2.0, (batch, wl.m)); w[:, ::9] = 0.0
    s = eng.settings()
    x = wl.x0.copy()
    res, _ = eng.optimize_batched(s, wl.model, x, wl.l, wl.u, t=wl.t, y=wl.y, w=w)
    cov, _, info = eng.covariance_batched(s, wl.model, x, wl.l, wl.u, t=wl.t, y=wl.y, w=w)
    _, se = eng.predict_batched(s, wl.model, x, wl.l, wl.u, t=wl.t, cov=cov)
    nf = ((wl.l < x) & (x < wl.u)).sum(axis=1)
    mw = wl.m if w is None else (w != 0).sum(axis=1)
    ww = np.ones((batch, wl.m)) if w is None else w
    lhs = (ww * ww * se * se).sum(axis=1)
    rhs = res["residual"] / (mw - nf) * nf
    ok = (info == 0) & (nf > 0)
    assert ok.mean() > 0.9
    rel = np.abs(lhs[ok] - rhs[ok]) / rhs[ok]
    assert rel.max() <= 1e-10, rel.max()


def test_coverage_of_the_band():
    N, m, sigma = 8192, 64, 0.05
    rng = np.random.default_rng(17)
    t = np.linspace(-4.0, 4.0, m)
    truth = np.array([5.0, 0.2, 0.8, 0.5])
    fm = lambda tt, p: p[0] * np.exp(-0.5 * ((tt - p[1]) / p[2]) ** 2) + p[3]
    y = fm(t, truth)[None, :] + sigma * rng.standard_normal((N, m))
    l = np.array([0.0, -2.0, 0.1, -5.0]); u = np.array([50.0, 2.0, 5.0, 5.0])
    x = np.tile(truth * 1.05, (N, 1))
    s = eng.settings()
    res, _ = eng.optimize_batched(s, ModelId.GAUSS4, x, l, u, t=t, y=y)
    assert np.all(res["status"] >= 0)
    cov, _, info = eng.covariance_batched(s, ModelId.GAUSS4, x, l, u, t=t, y=y)
    assert np.all(info == 0)
    ts = np.linspace(-4.0, 4.0, 33)
    v, se = eng.predict_batched(s, ModelId.GAUSS4, x, l, u, t=ts, cov=cov)
    z = (v - fm(ts, truth)[None, :]) / se
    zs = z.std(axis=0, ddof=1)
    assert np.all(np.abs(zs - 1) < 0.05), zs


@pytest.mark.parametrize("dt", DT)
def test_linear_model_is_exact(dt):
    rng = np.random.default_rng(71)
    batch, n = 64, 3
    mid = eng.compile_model(POLY3)
    try:
        x = rng.standard_normal((batch, n)); cov = spd(rng, batch, n)
        ts = np.linspace(-2.0, 3.0, 31)
        inf = np.full(n, np.inf)
        v, se = eng.predict_batched(None, mid, x.astype(dt), -inf, inf, t=ts, cov=cov.astype(dt))
        Phi = np.vander(ts.astype(dt).astype(np.float64), n, increasing=True)
        xd = x.astype(dt).astype(np.float64); cd = cov.astype(dt).astype(np.float64)
        exact = np.sqrt(np.einsum("ia,bac,ic->bi", Phi, cd, Phi))
        tol = 1e-13 if dt == np.float64 else 2.0 ** -22
        np.testing.assert_allclose(se, exact, rtol=tol, atol=0)
        np.testing.assert_allclose(v, xd @ Phi.T, rtol=tol if dt == np.float64 else 1e-5, atol=1e-13 if dt == np.float64 else 1e-5)
    finally:
        eng.release_model(mid)


def raw_predict(model, x, l, u, t, cov, y=None, w=None, flags=0, value=True, se=True, bound_stride=0):
    batch, n = x.shape; k = t.shape[-1]
    vo = np.full((batch, k), -1.0) if value else None
    so = np.full((batch, k), -1.0) if se else None
    d = ModelDesc(int(model), flags, C.c_void_p(t.ctypes.data), None if y is None else C.c_void_p(y.ctypes.data), None, 0.0,
                  None if w is None else C.c_void_p(w.ctypes.data))
    p = lambda a: None if a is None else a.ctypes.data
    rc = eng.lib.mir_b200_predict_batched_d(None, C.byref(d), batch, k, n, p(x), p(l), p(u), bound_stride, p(cov), p(vo), p(so), -1)
    assert rc == 0, eng.lib.mir_b200_last_error()
    return vo, so


def test_what_is_never_read():
    rng = np.random.default_rng(81)
    wl = workloads.c2_gauss4(64, seed=82)
    x = np.ascontiguousarray(wl.truth)
    l = np.tile(wl.l, (64, 1)); u = np.tile(wl.u, (64, 1))
    l[:, 1] = x[:, 1]; u[::2, 3] = x[::2, 3]                     # parameter 1 fixed everywhere, parameter 3 in half the problems
    cov = spd(rng, 64, 4)
    ts = np.linspace(-4.0, 4.0, 23)
    v0, s0 = raw_predict(wl.model, x, l, u, ts, cov, bound_stride=4)
    assert np.all(s0 > 0)
    bad = cov.copy()
    bad[:, np.triu_indices(4, 1)[0], np.triu_indices(4, 1)[1]] = np.nan          # the strict upper triangle
    bad[:, 1, :] = np.nan; bad[:, :, 1] = np.nan                                  # the fixed parameter's row and column
    bad[::2, 3, :] = np.nan; bad[::2, :, 3] = np.nan
    ynan = np.full((64, 23), np.nan); wnan = np.full((64, 23), np.nan)
    v1, s1 = raw_predict(wl.model, x, l, u, ts, bad, y=ynan, w=wnan, flags=MODEL_WEIGHTED, bound_stride=4)
    assert v1.tobytes() == v0.tobytes() and s1.tobytes() == s0.tobytes()
    # n_F = 0: se = 0
    _, sz = raw_predict(wl.model, x, x.copy(), x.copy(), ts, bad, bound_stride=4)
    assert np.all(sz == 0) and not np.signbit(sz).any()
    # value only, cov = NULL
    vv, none = raw_predict(wl.model, x, l, u, ts, None, se=False, bound_stride=4)
    assert none is None and vv.tobytes() == v0.tobytes()
    # se only
    none, ss = raw_predict(wl.model, x, l, u, ts, cov, value=False, bound_stride=4)
    assert none is None and ss.tobytes() == s0.tobytes()


def test_determinism_slices_and_both_forms():
    import torch
    wl = workloads.c2_gauss4(4096)
    s, x, _ = fit(wl, np.float64)
    cov, _, _ = eng.covariance_batched(s, wl.model, x, wl.l, wl.u, t=wl.t, y=wl.y)
    ts = np.linspace(-4.0, 4.0, 64)
    v1, s1 = eng.predict_batched(s, wl.model, x, wl.l, wl.u, t=ts, cov=cov)
    v2, s2 = eng.predict_batched(s, wl.model, x, wl.l, wl.u, t=ts, cov=cov)
    assert v1.tobytes() == v2.tobytes() and s1.tobytes() == s2.tobytes()
    perm = np.random.default_rng(3).permutation(4096)
    vp, sp = eng.predict_batched(s, wl.model, x[perm], wl.l, wl.u, t=ts, cov=cov[perm])
    assert vp.tobytes() == v1[perm].tobytes() and sp.tobytes() == s1[perm].tobytes()
    vs, ss = eng.predict_batched(s, wl.model, x[1000:1700], wl.l, wl.u, t=ts, cov=cov[1000:1700])
    assert vs.tobytes() == v1[1000:1700].tobytes() and ss.tobytes() == s1[1000:1700].tobytes()
    dev = torch.device("cuda:0")
    T = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    vd, sd = eng.predict_batched_device(s, wl.model, T(x), T(wl.l), T(wl.u), t=T(ts), cov=T(cov))
    torch.cuda.synchronize()
    assert vd.cpu().numpy().tobytes() == v1.tobytes() and sd.cpu().numpy().tobytes() == s1.tobytes()
    # preallocated outputs, per-problem abscissae
    tp = np.random.default_rng(4).uniform(-4, 4, (4096, 16))
    vh, sh = eng.predict_batched(s, wl.model, x, wl.l, wl.u, t=tp, cov=cov)
    vo = torch.empty((4096, 16), dtype=torch.float64, device=dev); so = torch.empty_like(vo)
    eng.predict_batched_device(s, wl.model, T(x), T(wl.l), T(wl.u), t=T(tp), cov=T(cov), value=vo, se=so)
    torch.cuda.synchronize()
    assert vo.cpu().numpy().tobytes() == vh.tobytes() and so.cpu().numpy().tobytes() == sh.tobytes()


def test_resident_chain_equals_host_chain():
    import torch
    dev = torch.device("cuda:0")
    T = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    # Gauss4: fit -> covariance -> predict on the same device buffers
    wl = workloads.c2_gauss4(2048, seed=91)
    s = eng.settings()
    ts = np.linspace(-4.0, 4.0, 64)
    x = wl.x0.copy()
    eng.optimize_batched(s, wl.model, x, wl.l, wl.u, t=wl.t, y=wl.y)
    ch, _, _ = eng.covariance_batched(s, wl.model, x, wl.l, wl.u, t=wl.t, y=wl.y)
    vh, sh = eng.predict_batched(s, wl.model, x, wl.l, wl.u, t=ts, cov=ch)
    xd = T(wl.x0); ld, ud = T(wl.l), T(wl.u)
    eng.optimize_batched_device(s, wl.model, xd, ld, ud, t=T(wl.t), y=T(wl.y))
    cd, _, _ = eng.covariance_batched_device(s, wl.model, xd, ld, ud, t=T(wl.t), y=T(wl.y))
    vd, sd = eng.predict_batched_device(s, wl.model, xd, ld, ud, t=T(ts), cov=cd)
    torch.cuda.synchronize()
    assert xd.cpu().numpy().tobytes() == x.tobytes()
    assert vd.cpu().numpy().tobytes() == vh.tobytes() and sd.cpu().numpy().tobytes() == sh.tobytes()
    # the spline: the resident fit has m = P rows (the smoothing row replaces the last point's, fit_splie.d:67-80)
    rng = np.random.default_rng(12)
    batch, P, n, lam = 64, 50, 7, 1e-3
    px = np.sort(rng.uniform(0.0, 6.0, P)); knots = np.linspace(0.0, 6.0, n)
    py = np.cos(px)[None, :] + 0.05 * rng.standard_normal((batch, P))
    l = np.full(n, -5.0); u = np.full(n, 5.0)
    ts = np.linspace(0.0, 6.0, 40)
    vals, _ = eng.fit_spline_batched(s, px, py, knots, l, u, lam)
    ch, _, _ = eng.covariance_batched(s, ModelId.SPLINE, vals, l, u, t=px, y=py, fd_jacobian=True, aux=knots, param=lam)
    vh, sh = eng.predict_batched(s, ModelId.SPLINE, vals, l, u, t=ts, cov=ch, fd_jacobian=True, aux=knots, param=lam)
    xd = torch.zeros((batch, n), dtype=torch.float64, device=dev)
    eng.optimize_batched_device(s, ModelId.SPLINE, xd, T(l), T(u), t=T(px), y=T(py), fd_jacobian=True, aux=T(knots), param=lam)
    cd, _, _ = eng.covariance_batched_device(s, ModelId.SPLINE, xd, T(l), T(u), t=T(px), y=T(py), fd_jacobian=True, aux=T(knots), param=lam)
    vd, sd = eng.predict_batched_device(s, ModelId.SPLINE, xd, T(l), T(u), t=T(ts), cov=cd, fd_jacobian=True, aux=T(knots), param=lam)
    torch.cuda.synchronize()
    assert xd.cpu().numpy().tobytes() == vals.tobytes()
    assert vd.cpu().numpy().tobytes() == vh.tobytes() and sd.cpu().numpy().tobytes() == sh.tobytes()


NO_PREDICTION_DOUBLE = r"""
namespace mirb200 { template <> struct CtaTrailingRow<CtaUser<::UserModel<double>, double>>; }
"""


def test_user_model_prediction_program_is_built_at_the_first_predict_call():
    """Registration, the fit and the covariance build no prediction program; the first prediction call builds it (here
    it cannot compile for double, which makes the build visible), and float is unaffected.  After release_model a
    prediction returns EINVAL."""
    wl = workloads.c2_gauss4(64, seed=38)
    ts = np.linspace(-4.0, 4.0, 16)
    mid = eng.compile_model(GAUSS4_USER + NO_PREDICTION_DOUBLE)
    try:
        s = eng.settings(np.float64); s.maxIterations = 3
        x = wl.x0.copy(); eng.optimize_batched(s, mid, x, wl.l, wl.u, t=wl.t, y=wl.y)
        cov, _, _ = eng.covariance_batched(None, mid, x, wl.l, wl.u, t=wl.t, y=wl.y)
        with pytest.raises(B200Error) as e:
            eng.predict_batched(None, mid, x, wl.l, wl.u, t=ts, cov=cov)
        assert e.value.code == 2 and "does not compile" in str(e.value)
        vf, sf = eng.predict_batched(None, mid, x.astype(np.float32), wl.l, wl.u, t=ts, cov=cov)
        vb, sb = eng.predict_batched(None, ModelId.GAUSS4, x.astype(np.float32), wl.l, wl.u, t=ts, cov=cov)
        assert vf.tobytes() == vb.tobytes()
    finally:
        eng.release_model(mid)
    with pytest.raises(B200Error) as e:
        eng.predict_batched(None, mid, x, wl.l, wl.u, t=ts, cov=cov)
    assert e.value.code == 2
