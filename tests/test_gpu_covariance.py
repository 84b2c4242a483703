"""Batched parameter covariance on the B200 (mir_b200_covariance_batched_*) against the host reference of its definition
(tests/cov_util.py, residuals and Jacobians from the oracle's callbacks), plus info codes, argument checks, determinism,
the built-in functors against user-model restatements, and a statistical check of the standard errors."""
import ctypes as C

import numpy as np
import pytest

import mir_optim_b200 as mo
from mir_optim_b200 import ModelId, workloads
from mir_optim_b200._abi import ModelDesc
from mir_optim_b200.engine import B200Error
from cov_util import cov_bound, cov_error, cov_reference, oracle_callbacks
from user_models import EXPDECAY3_REPRO, LOGISTIC, RIDGE_POLY

pytestmark = pytest.mark.gpu

eng = mo.engine
DT = [np.float64, np.float32]

# a Gauss4 restatement as a user model, with the operation sequence of the built-in functor (models_large.cuh)
GAUSS4_USER = r'''
template <class REAL> struct UserModel {
    static constexpr bool kAnalytic = true;
    __device__ static REAL residual(const REAL* p, int n, int m, int row, REAL t, REAL y, const REAL* aux, REAL param) {
        using namespace mirb200;
        const REAL is = rcp_ni(p[2]);
        const REAL z = mul_rn(sub_rn(t, p[1]), is);
        return sub_rn(add_rn(mul_rn(p[0], exp_repro_tp(mul_rn((REAL)-0.5, mul_rn(z, z)))), p[3]), y);
    }
    __device__ static void jacobian(const REAL* p, int n, int m, int row, REAL t, REAL y, const REAL* aux, REAL param, REAL* J) {
        using namespace mirb200;
        const REAL is = rcp_ni(p[2]);
        const REAL z = mul_rn(sub_rn(t, p[1]), is);
        const REAL zz = mul_rn(z, z);
        const REAL e = exp_repro_tp(mul_rn((REAL)-0.5, zz));
        const REAL ae = mul_rn(p[0], e);
        J[0] = e; J[1] = mul_rn(mul_rn(ae, z), is); J[2] = mul_rn(mul_rn(ae, zz), is); J[3] = (REAL)1;
    }
};
'''


def fit(wl, dt, fd=False, **kw):
    s = eng.settings(dt)
    x = wl.x0.astype(dt).copy()
    res, _ = eng.optimize_batched(s, wl.model, x, wl.l.astype(dt), wl.u.astype(dt), t=wl.t.astype(dt), y=wl.y.astype(dt),
                                  fd_jacobian=fd, **kw)
    return s, x, res


def check_parity(cov, info, ref, rinfo, kap, dt, bound=None):
    assert np.array_equal(info, rinfo), np.nonzero(info != rinfo)
    ok = rinfo == 0
    e = cov_error(cov[ok], ref[ok])
    b = cov_bound(kap[ok], dt) if bound is None else bound
    assert np.all(e <= b), (float(e.max()), float(np.max(e / b)))
    # exact symmetry, zeros outside the free block
    assert np.array_equal(cov, np.swapaxes(cov, 1, 2), equal_nan=True)
    assert np.all(cov[ok][ref[ok] == 0] == 0)


@pytest.mark.parametrize("dt", DT)
def test_parity_analytic_gauss4(oracle_lib, dt):
    wl = workloads.c2_gauss4(4096, dtype=dt)
    s, x, _ = fit(wl, dt)
    cov, sd, info = eng.covariance_batched(s, wl.model, x, wl.l, wl.u, t=wl.t, y=wl.y)
    f, g = oracle_callbacks(oracle_lib, wl.model, dt, wl.t, wl.y)
    ref, rinfo, kap = cov_reference(f, g, x, wl.l.astype(dt), wl.u.astype(dt), s.jacobianEpsilon)
    check_parity(cov, info, ref, rinfo, kap, dt)
    assert (info == 0).mean() > 0.99
    d = np.einsum("bii->bi", cov.astype(np.float64))
    np.testing.assert_allclose(sd, np.sqrt(d).astype(dt), rtol=2e-7 if dt == np.float32 else 1e-15)


@pytest.mark.parametrize("dt", DT)
def test_parity_fd_sumexp8(oracle_lib, dt):
    wl = workloads.c3_sumexp8(512, dtype=dt)
    s, x, _ = fit(wl, dt, fd=True)
    cov, sd, info = eng.covariance_batched(s, wl.model, x, wl.l, wl.u, t=wl.t, y=wl.y, fd_jacobian=True)
    f, _ = oracle_callbacks(oracle_lib, wl.model, dt, wl.t, wl.y, fd=True)
    ref, rinfo, kap = cov_reference(f, None, x, wl.l.astype(dt), wl.u.astype(dt), s.jacobianEpsilon)
    check_parity(cov, info, ref, rinfo, kap, dt)


def test_parity_fd_expdecay3_m1000(oracle_lib):
    ws = [workloads.c1_expdecay3(seed=k) for k in range(1, 65)]
    wl = dict(ws[0]); wl["y"] = np.concatenate([w.y for w in ws]); wl["x0"] = np.repeat(ws[0].x0, 64, axis=0)
    wl = workloads.Workload(wl)
    s, x, _ = fit(wl, np.float64, fd=True)
    cov, sd, info = eng.covariance_batched(None, wl.model, x, wl.l, wl.u, t=wl.t, y=wl.y, fd_jacobian=True)
    f, _ = oracle_callbacks(oracle_lib, wl.model, np.float64, wl.t, wl.y, fd=True)
    ref, rinfo, kap = cov_reference(f, None, x, wl.l, wl.u, s.jacobianEpsilon)
    check_parity(cov, info, ref, rinfo, kap, np.float64)
    assert np.all(info == 0)


def gaussmix_workload(batch, m=200, seed=21):
    rng = np.random.default_rng(seed)
    t = np.linspace(0.0, 1.0, m)
    truth = np.tile(np.array([1.0, 0.25, 0.06, 0.7, 0.5, 0.05, 1.2, 0.75, 0.07, 0.2, -0.1]), (batch, 1))
    truth[:, 0:9:3] *= rng.uniform(0.8, 1.2, (batch, 3))
    y = np.empty((batch, m))
    for b in range(batch):
        p = truth[b]
        v = p[9] + p[10] * t
        for k in range(3):
            v = v + p[3 * k] * np.exp(-0.5 * ((t - p[3 * k + 1]) / p[3 * k + 2]) ** 2)
        y[b] = v + 0.01 * rng.standard_normal(m)
    l = np.full(11, -np.inf); u = np.full(11, np.inf)
    u[3] = 0.6                                          # the second amplitude's upper bound is active at the solution
    l[10] = -0.05                                       # and the slope's lower bound
    x0 = np.clip(truth * 1.03, l, u)
    return workloads.Workload(model=ModelId.GAUSSMIX, t=t, y=y, x0=x0, l=l, u=u)


def test_general_kernel_gaussmix_n11_with_active_bounds(oracle_lib):
    wl = gaussmix_workload(128)
    s, x, _ = fit(wl, np.float64)
    cov, sd, info = eng.covariance_batched(s, wl.model, x, wl.l, wl.u, t=wl.t, y=wl.y)
    f, g = oracle_callbacks(oracle_lib, wl.model, np.float64, wl.t, wl.y)
    ref, rinfo, kap = cov_reference(f, g, x, wl.l, wl.u, s.jacobianEpsilon)
    check_parity(cov, info, ref, rinfo, kap, np.float64)
    fixed = (x == wl.u) | (x == wl.l)
    assert fixed[:, 3].mean() > 0.5                     # the bound really is active for most problems
    assert np.all(cov[fixed] == 0) and np.all(sd[fixed] == 0)


def test_general_kernel_sumexp_n10(oracle_lib):
    rng = np.random.default_rng(5)
    t = np.linspace(0.0, 5.0, 100)
    x = np.empty((64, 10)); x[:, 0::2] = rng.uniform(1, 5, (64, 5)); x[:, 1::2] = np.array([0.2, 0.6, 1.5, 4.0, 10.0]) * rng.uniform(0.8, 1.2, (64, 5))
    y = np.einsum("bk,bkm->bm", x[:, 0::2], np.exp(-x[:, 1::2, None] * t)) + 0.01 * rng.standard_normal((64, 100))
    l = np.full(10, -np.inf); u = np.full(10, np.inf)
    for fd in (False, True):
        cov, sd, info = eng.covariance_batched(None, ModelId.SUMEXP, x, l, u, t=t, y=y, fd_jacobian=fd)
        f, g = oracle_callbacks(oracle_lib, ModelId.SUMEXP, np.float64, t, y, fd=fd)
        ref, rinfo, kap = cov_reference(f, g, x, l, u, 2.0 ** -26)
        check_parity(cov, info, ref, rinfo, kap, np.float64)


@pytest.mark.parametrize("lam", [0.0, 1e-3])
@pytest.mark.parametrize("per_problem_knots", [False, True])
def test_general_kernel_spline(oracle_lib, lam, per_problem_knots):
    rng = np.random.default_rng(8)
    batch, P, n = 32, 60, 8
    px = np.sort(rng.uniform(0.0, 10.0, P))
    py = np.sin(px)[None, :] + 0.05 * rng.standard_normal((batch, P))
    knots = np.linspace(0.0, 10.0, n)
    if per_problem_knots:
        knots = np.sort(knots[None, :] + np.concatenate([np.zeros((batch, 1)), rng.uniform(-0.2, 0.2, (batch, n - 2)), np.zeros((batch, 1))], axis=1), axis=1)
    l = np.full(n, -10.0); u = np.full(n, 10.0)
    s = eng.settings()
    vals, res = eng.fit_spline_batched(s, px, py, knots, l, u, lam)
    m = P + (1 if lam == 0 else 0)
    t = np.zeros(m); t[:P] = px
    y = np.zeros((batch, m)); y[:, :P] = py
    cov, sd, info = eng.covariance_batched(s, ModelId.SPLINE, vals, l, u, t=t, y=y, fd_jacobian=True, aux=knots, param=lam)
    f, _ = oracle_callbacks(oracle_lib, ModelId.SPLINE, np.float64, t, y, aux=knots, param=lam, fd=True)
    ref, rinfo, kap = cov_reference(f, None, vals, l, u, s.jacobianEpsilon)
    check_parity(cov, info, ref, rinfo, kap, np.float64)
    assert np.all(info == 0)


def test_user_models_logistic_fd_and_ridge_poly():
    # LOGISTIC uses CUDA's exp, so the host restatement differs in the last bits of each residual and the central
    # difference magnifies that by ~1/h: held to 1e-5 (double) and 1e-1 (float); RIDGE_POLY (polynomial rows) to 1e-10
    rng = np.random.default_rng(9)
    mid = eng.compile_model(LOGISTIC)
    try:
        t = np.linspace(0.0, 10.0, 80)
        x = np.column_stack([rng.uniform(4, 6, 32), rng.uniform(0.8, 1.2, 32), rng.uniform(4, 6, 32)])
        y = x[:, :1] / (1 + np.exp(-x[:, 1:2] * (t - x[:, 2:3]))) + 0.02 * rng.standard_normal((32, 80))
        inf = np.full(3, np.inf)
        for dt in DT:
            cov, sd, info = eng.covariance_batched(None, mid, x.astype(dt), -inf, inf, t=t, y=y)
            f = lambda b, p: (p[0] / (1 + np.exp(-p[1] * (t.astype(dt) - p[2]))) - y[b].astype(dt)).astype(dt)
            eps = eng.settings(dt).jacobianEpsilon
            ref, rinfo, kap = cov_reference(f, None, x.astype(dt), -inf.astype(dt), inf.astype(dt), eps)
            check_parity(cov, info, ref, rinfo, kap, dt, bound=1e-5 if dt == np.float64 else 1e-1)
    finally:
        eng.release_model(mid)
    mid = eng.compile_model(RIDGE_POLY)
    try:
        n, P = 4, 40
        t = np.linspace(-1.0, 1.0, P + n)
        aux = np.array([1.0, 2.0, 3.0, 4.0]); lam = 0.1
        x = rng.standard_normal((16, n))
        y = rng.standard_normal((16, P + n))

        def f(b, p):
            r = np.polyval(p[::-1], t) - y[b]
            r[P:] = np.sqrt(lam) * aux * p
            return r

        def g(b, p):
            J = np.vander(t, n, increasing=True)
            J[P:] = np.diag(np.sqrt(lam) * aux)
            return J

        cov, sd, info = eng.covariance_batched(None, mid, x, np.full(n, -np.inf), np.full(n, np.inf), t=t, y=y, aux=aux, param=lam)
        ref, rinfo, kap = cov_reference(f, g, x, np.full(n, -np.inf), np.full(n, np.inf), 2.0 ** -26)
        check_parity(cov, info, ref, rinfo, kap, np.float64, bound=1e-10)
    finally:
        eng.release_model(mid)


def test_bounds_tight_gauss4(oracle_lib):
    wl = workloads.c2_gauss4(2048, tight_bounds=True)
    s, x, _ = fit(wl, np.float64)
    cov, sd, info = eng.covariance_batched(s, wl.model, x, wl.l, wl.u, t=wl.t, y=wl.y)
    fixed = (x == wl.l) | (x == wl.u)
    assert fixed.any(axis=1).mean() > 0.3
    assert np.all(cov[fixed] == 0) and np.all(np.swapaxes(cov, 1, 2)[fixed] == 0) and np.all(sd[fixed] == 0)
    f, g = oracle_callbacks(oracle_lib, wl.model, np.float64, wl.t, wl.y)
    ref, rinfo, kap = cov_reference(f, g, x, wl.l, wl.u, s.jacobianEpsilon)       # reduced J, dof = m - n_F
    check_parity(cov, info, ref, rinfo, kap, np.float64)


def test_edge_cases():
    wl = workloads.c2_gauss4(4)
    x = wl.truth.copy(); x[0, 0] = 0.0                  # amplitude 0: the mu (and sigma) columns of J are zero
    inf4 = np.full(4, np.inf)
    cov, sd, info = eng.covariance_batched(None, wl.model, x, -inf4, inf4, t=wl.t, y=wl.y)
    assert info[0] == 2 and np.all(np.isnan(cov[0])) and np.all(np.isnan(sd[0]))
    assert np.all(info[1:] == 0)
    # unscaled = scaled / s^2
    cu, su, iu = eng.covariance_batched(None, wl.model, wl.truth, -inf4, inf4, t=wl.t, y=wl.y, scaled=False)
    cs, ss, is_ = eng.covariance_batched(None, wl.model, wl.truth, -inf4, inf4, t=wl.t, y=wl.y)
    r = wl.truth[:, 0:1] * np.exp(-0.5 * ((wl.t - wl.truth[:, 1:2]) / wl.truth[:, 2:3]) ** 2) + wl.truth[:, 3:4] - wl.y
    s2 = (r * r).sum(axis=1) / (64 - 4)
    np.testing.assert_allclose(cs, cu * s2[:, None, None], rtol=1e-12)
    # NaN in x
    xn = wl.truth.copy(); xn[1, 2] = np.nan
    cov, sd, info = eng.covariance_batched(None, wl.model, xn, -inf4, inf4, t=wl.t, y=wl.y)
    assert info[1] == -2 and np.all(np.isnan(cov[1][np.ix_([0, 1, 3], [0, 1, 3])])) and info[0] == 0
    # every parameter on a bound: zeros, info 0
    cov, sd, info = eng.covariance_batched(None, wl.model, wl.truth, wl.truth[0], wl.truth[0], t=wl.t, y=wl.y[:1].repeat(4, 0))
    assert np.all(info == 0) and np.all(cov[0] == 0) and np.all(sd[0] == 0)
    # m <= n_F: +inf, as scipy
    w3 = workloads.c1_expdecay3(m=3)
    inf3 = np.full(3, np.inf)
    cov, sd, info = eng.covariance_batched(None, w3.model, w3.truth, -inf3, inf3, t=w3.t, y=w3.y)
    assert info[0] == -1 and np.all(np.isposinf(cov[0])) and np.all(np.isposinf(sd[0]))


def test_batch_zero_and_argument_errors():
    wl = workloads.c2_gauss4(4)
    lib = eng.lib
    x = wl.x0.copy(); info = np.zeros(4, np.int32); sd = np.zeros((4, 4)); cv = np.zeros((4, 4, 4))

    def call(model=ModelId.GAUSS4, batch=4, m=64, n=4, t=wl.t, y=wl.y, xx=x, ii=info, c=cv, s=sd, desc=True, aux=None):
        d = ModelDesc(int(model), 0, None if t is None else C.c_void_p(t.ctypes.data), None if y is None else C.c_void_p(y.ctypes.data),
                      None if aux is None else C.c_void_p(aux.ctypes.data), 0.0)
        return lib.mir_b200_covariance_batched_d(None, C.byref(d) if desc else None, batch, m, n, None if xx is None else xx.ctypes.data,
                                                 wl.l.ctypes.data, wl.u.ctypes.data, 0, 0, None if c is None else c.ctypes.data,
                                                 None if s is None else s.ctypes.data, None if ii is None else ii.ctypes.data, -1)
    assert call() == 0 and np.all(info == 0)
    assert call(batch=0) == 0
    assert call(desc=False) == 2 and call(xx=None) == 2 and call(ii=None) == 2 and call(c=None, s=None) == 2
    assert call(n=0) == 2 and call(m=0) == 2 and call(t=None) == 2 and call(y=None) == 2
    assert call(n=5) == 2                                                       # Gauss4 has n = 4
    assert call(model=ModelId.SPLINE, n=4) == 2                                 # no knots
    big = np.zeros((4, 129))
    assert call(model=ModelId.GAUSSMIX, n=129, xx=big) == 3
    for mid in (ModelId.LINEAR2, ModelId.ROSENBROCK, ModelId.SQRTCIRCLE):
        assert call(model=mid, n=2) == 3
    assert call(model=0x1000 + 99999) == 2                                      # unknown user model
    assert call(c=None) == 0 and call(s=None) == 0


def test_determinism_and_both_forms():
    import torch
    wl = workloads.c2_gauss4(4096)
    s, x, _ = fit(wl, np.float64)
    c1, s1, i1 = eng.covariance_batched(s, wl.model, x, wl.l, wl.u, t=wl.t, y=wl.y)
    c2, s2, i2 = eng.covariance_batched(s, wl.model, x, wl.l, wl.u, t=wl.t, y=wl.y)
    assert c1.tobytes() == c2.tobytes() and s1.tobytes() == s2.tobytes() and np.array_equal(i1, i2)
    perm = np.random.default_rng(3).permutation(4096)
    cp, sp, ip = eng.covariance_batched(s, wl.model, x[perm], wl.l, wl.u, t=wl.t, y=wl.y[perm])
    assert cp.tobytes() == c1[perm].tobytes() and sp.tobytes() == s1[perm].tobytes()
    cs, ss, is_ = eng.covariance_batched(s, wl.model, x[:1000], wl.l, wl.u, t=wl.t, y=wl.y[:1000])
    assert cs.tobytes() == c1[:1000].tobytes() and ss.tobytes() == s1[:1000].tobytes()
    dev = torch.device("cuda:0")
    T = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    cd, sd, idv = eng.covariance_batched_device(s, wl.model, T(x), T(wl.l), T(wl.u), t=T(wl.t), y=T(wl.y))
    torch.cuda.synchronize()
    assert cd.cpu().numpy().tobytes() == c1.tobytes() and sd.cpu().numpy().tobytes() == s1.tobytes()
    assert np.array_equal(idv.cpu().numpy(), i1)
    _, sd_only, _ = eng.covariance_batched_device(None, wl.model, T(x), T(wl.l), T(wl.u), t=T(wl.t), y=T(wl.y), want_cov=False)
    torch.cuda.synchronize()
    assert sd_only.cpu().numpy().tobytes() == s1.tobytes()


@pytest.mark.parametrize("dt", DT)
def test_builtin_against_user_restatements(oracle_lib, dt):
    # EXPDECAY3_REPRO has the built-in functor's bits: only the code path differs, so they agree to 1e-13
    ws = [workloads.c1_expdecay3(seed=k, m=200) for k in range(1, 33)]
    y = np.concatenate([w.y for w in ws]); t = ws[0].t; x0 = np.repeat(ws[0].x0, 32, axis=0)
    wl = workloads.Workload(model=ModelId.EXPDECAY3, t=t, y=y, x0=x0, l=ws[0].l, u=ws[0].u)
    s, x, _ = fit(wl, dt)
    inf3 = np.full(3, np.inf)
    cb, sb, ib = eng.covariance_batched(s, ModelId.EXPDECAY3, x, -inf3, inf3, t=t, y=y)
    mid = eng.compile_model(EXPDECAY3_REPRO)
    try:
        cu, su, iu = eng.covariance_batched(s, mid, x, -inf3, inf3, t=t, y=y)
    finally:
        eng.release_model(mid)
    assert np.array_equal(ib, iu) and np.all(ib == 0)
    assert cov_error(cu, cb).max() <= 1e-13 + (2.0 ** -23 if dt == np.float32 else 0)
    # GAUSS4: the restatement follows the op sequence of models_large.cuh; held to the parity bound
    wl = workloads.c2_gauss4(1024, dtype=dt)
    s, x, _ = fit(wl, dt)
    cb, sb, ib = eng.covariance_batched(s, wl.model, x, wl.l, wl.u, t=wl.t, y=wl.y)
    mid = eng.compile_model(GAUSS4_USER)
    try:
        cu, su, iu = eng.covariance_batched(s, mid, x, wl.l, wl.u, t=wl.t, y=wl.y)
    finally:
        eng.release_model(mid)
    f, g = oracle_callbacks(oracle_lib, wl.model, dt, wl.t, wl.y)
    ref, rinfo, kap = cov_reference(f, g, x, wl.l.astype(dt), wl.u.astype(dt), s.jacobianEpsilon)
    check_parity(cu, iu, ref, rinfo, kap, dt)
    check_parity(cb, ib, ref, rinfo, kap, dt)


def test_standard_errors_match_the_spread_of_fits():
    N, m, sigma = 8192, 64, 0.05
    rng = np.random.default_rng(17)
    t = np.linspace(-4.0, 4.0, m)
    truth = np.array([5.0, 0.2, 0.8, 0.5])
    clean = truth[0] * np.exp(-0.5 * ((t - truth[1]) / truth[2]) ** 2) + truth[3]
    y = clean[None, :] + sigma * rng.standard_normal((N, m))
    l = np.array([0.0, -2.0, 0.1, -5.0]); u = np.array([50.0, 2.0, 5.0, 5.0])
    x = np.tile(truth * 1.05, (N, 1))
    s = eng.settings()
    res, _ = eng.optimize_batched(s, ModelId.GAUSS4, x, l, u, t=t, y=y)
    assert np.all(res["status"] >= 0)
    cov, sd, info = eng.covariance_batched(s, ModelId.GAUSS4, x, l, u, t=t, y=y)
    assert np.all(info == 0)
    emp = x.std(axis=0, ddof=1); pred = sd.mean(axis=0)
    assert np.all(np.abs(emp / pred - 1) < 0.05), (emp, pred)
    z = (x - truth) / sd
    zs = z.std(axis=0, ddof=1)
    assert np.all((zs > 0.95) & (zs < 1.05)), zs


def test_resident_spline_fit_then_covariance(oracle_lib):
    import torch
    dev = torch.device("cuda:0")
    rng = np.random.default_rng(12)
    batch, P, n, lam = 64, 50, 7, 1e-3
    px = np.sort(rng.uniform(0.0, 6.0, P)); knots = np.linspace(0.0, 6.0, n)
    py = np.cos(px)[None, :] + 0.05 * rng.standard_normal((batch, P))
    l = np.full(n, -5.0); u = np.full(n, 5.0)
    s = eng.settings()
    # host reference fit through fitSpline
    vals, res = eng.fit_spline_batched(s, px, py, knots, l, u, lam)
    # the same fit, resident: m = P rows (the smoothing row replaces the last point's residual, fit_splie.d:67-80)
    T = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    xd = torch.zeros((batch, n), dtype=torch.float64, device=dev)
    resd = eng.optimize_batched_device(s, ModelId.SPLINE, xd, T(l), T(u), t=T(px), y=T(py), fd_jacobian=True, aux=T(knots), param=lam)
    cd, sdd, idd = eng.covariance_batched_device(s, ModelId.SPLINE, xd, T(l), T(u), t=T(px), y=T(py), fd_jacobian=True,
                                                 aux=T(knots), param=lam)
    torch.cuda.synchronize()
    np.testing.assert_array_equal(xd.cpu().numpy(), vals)
    ch, sh, ih = eng.covariance_batched(s, ModelId.SPLINE, vals, l, u, t=px, y=py, fd_jacobian=True, aux=knots, param=lam)
    assert cd.cpu().numpy().tobytes() == ch.tobytes() and np.all(ih == 0) and np.array_equal(idd.cpu().numpy(), ih)
    # warm start: continue the resident fit from its own result; lambda and x are taken over
    r0 = eng.results_from_bytes(resd, np.float64)
    resw = eng.optimize_batched_device(s, ModelId.SPLINE, xd, T(l), T(u), t=T(px), y=T(py), fd_jacobian=True, aux=T(knots),
                                       param=lam, results=resd, warm_start=True)
    torch.cuda.synchronize()
    rw = eng.results_from_bytes(resw, np.float64)
    assert np.all(rw["status"] >= 0) and np.all(rw["residual"] <= r0["residual"])
