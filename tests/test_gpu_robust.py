"""Robust losses (MIR_MODEL_LOSS_SOFT_L1 / MIR_MODEL_LOSS_HUBER) on the B200: robust fits of the general kernel against the
robust host reference (tests/robust_util.py: the oracle LM with f~ = sign(u) sqrt(rho(u^2))), huber inside its quadratic
region against the squared loss bit for bit, the transform at extreme residuals against the host restatement bit for
bit, outlier recovery at batch scale, user models, and determinism across forms, calls and batch layouts."""
import numpy as np
import pytest

import mir_optim_b200 as mo
from mir_optim_b200 import ModelId, workloads
from oracle_util import oracle_batched, rel_err
from robust_util import oracle_batched_robust, robust_transform, with_outliers
from test_gpu_covariance import GAUSS4_USER
from test_gpu_cta_general import same_counters, sumexp
from test_gpu_weights import expdecay3, gauss4, gaussmix, spline_case
from test_robust_cpu import transform_arguments
from weights_util import sigma_weights

pytestmark = pytest.mark.gpu
eng = mo.engine
LOSSES = ("soft_l1", "huber")

# (model, data, fd, dtype, noise sigma of the data, weighted): the weighted cases use w = 0.3 / sigma times 1/sigma_i over a
# decade (so inlier |u| spans both sides of 1) with some zero rows; the unweighted ones see u = r.  Every case carries 10 %
# gross outliers of 1.5 to 15 (robust_util.with_outliers), so huber runs both of its regimes.
CASES = {
    "gauss4": (ModelId.GAUSS4, lambda: gauss4(160, 61), False, np.float64, 0.05, True),
    "gauss4_fd": (ModelId.GAUSS4, lambda: gauss4(160, 62), True, np.float64, 0.05, False),
    "gauss4_grid_per_problem": (ModelId.GAUSS4, lambda: gauss4(160, 63, per_problem_grid=True), False, np.float64, 0.05, True),
    "expdecay3": (ModelId.EXPDECAY3, lambda: expdecay3(160, 90, 64), False, np.float64, 0.02, False),
    "sumexp10": (ModelId.SUMEXP, lambda: sumexp(128, 5, 120, seed=65), False, np.float64, 0.01, True),
    "gaussmix11_bounds": (ModelId.GAUSSMIX, lambda: gaussmix(96, 150, 66), False, np.float64, 0.01, True),
    "spline_fd": (ModelId.SPLINE, lambda: spline_case(96, 67), True, np.float64, 0.05, False),
    "gauss4_float": (ModelId.GAUSS4, lambda: gauss4(256, 68), False, np.float32, 0.05, True),
}


def case_data(case):
    model, make, fd, dt, sigma, weighted = CASES[case]
    d = make()
    d["y"] = with_outliers(d["y"], 0.1, 0.3, seed=70 + list(CASES).index(case))
    B, m = d["y"].shape
    w = (0.3 / sigma) * sigma_weights(B, m, seed=list(CASES).index(case), zero_rows=max(1, m // 16)) if weighted else None
    return model, d, fd, dt, w


@pytest.mark.parametrize("loss", LOSSES)
@pytest.mark.parametrize("case", list(CASES))
def test_k_step_trajectories_against_the_robust_oracle(oracle_lib, case, loss):
    """k = 1, 2, 3 accepted steps: the same statuses and counters as the robust reference for >= 99 % of problems, x and
    lambda to rounding (the tolerances of the weighted test)."""
    model, d, fd, dt, w = case_data(case)
    B = d["y"].shape[0]
    args = {k: (v.astype(dt) if isinstance(v, np.ndarray) else v) for k, v in d.items() if k in ("t", "y", "aux", "param")}
    x0, l, u = d["x0"].astype(dt), d["l"].astype(dt), d["u"].astype(dt)
    wt = None if w is None else w.astype(dt)
    for k in (1, 2, 3):
        s = eng.settings(dt); s.maxIterations = k
        xg = x0.copy()
        rg, stats = eng.optimize_batched(s, model, xg, l, u, fd_jacobian=fd, want_stats=True, w=wt, loss=loss, **args)
        xo, ro = oracle_batched_robust(oracle_lib, s, model, x0, l, u, loss, w=wt, fd_jacobian=fd, **args)
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


def test_huber_inside_its_quadratic_region_is_the_squared_loss_bit_for_bit():
    """Where every |u| stays <= 1, huber's f~ = u and g = 1: weighted huber is the weighted fit (SUMEXP n = 10 and Gauss4,
    w small enough that |u| <= 1 on every evaluated point), and unweighted huber on SUMEXP n = 10 (general kernel either
    way) is the plain fit, on data and starting points whose residuals stay inside the region."""
    s = eng.settings(np.float64); s.maxIterations = 8
    d = sumexp(300, 5, 100, seed=71)
    wl = workloads.c2_gauss4(2048, noise=0.05, seed=72)
    for model, t, y, x0, l, u in ((ModelId.SUMEXP, d["t"], d["y"], d["x0"], d["l"], d["u"]), (wl.model, wl.t, wl.y, wl.x0, wl.l, wl.u)):
        w = 1e-4 * sigma_weights(x0.shape[0], y.shape[1], seed=73)
        xa = x0.copy(); ra, _ = eng.optimize_batched(s, model, xa, l, u, t=t, y=y, w=w)
        xb = x0.copy(); rb, _ = eng.optimize_batched(s, model, xb, l, u, t=t, y=y, w=w, loss="huber")
        assert xa.tobytes() == xb.tobytes() and ra.tobytes() == rb.tobytes(), model
    rng = np.random.default_rng(74)
    x0 = d["truth"] * rng.uniform(0.995, 1.005, d["truth"].shape)
    xa = x0.copy(); ra, _ = eng.optimize_batched(s, ModelId.SUMEXP, xa, d["l"], d["u"], t=d["t"], y=d["y"])
    xb = x0.copy(); rb, _ = eng.optimize_batched(s, ModelId.SUMEXP, xb, d["l"], d["u"], t=d["t"], y=d["y"], loss="huber")
    assert xa.tobytes() == xb.tobytes() and ra.tobytes() == rb.tobytes()


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("loss", LOSSES)
def test_extreme_residuals_equal_the_host_restatement(loss, dtype):
    """m = 1 EXPDECAY2 problems at p = 0 with every parameter fixed (l = u = x), t = 0: r = -y exactly, and Result.residual
    is f~^2 at x0, for u swept over the accuracy test's range (subnormals to the largest finite value, both signs).  It
    equals the host restatement's bits, and it is finite wherever f~^2 is representable in T (near the top of the range
    f~^2 ~ 2|u| overflows on both sides)."""
    u = transform_arguments(dtype)
    B = u.size
    y = (-u).reshape(B, 1)
    x = np.zeros((B, 2), dtype)
    s = eng.settings(dtype)
    res, _ = eng.optimize_batched(s, ModelId.EXPDECAY2, x, x.copy(), x.copy(), t=np.zeros(1, dtype), y=y, loss=loss)
    f, _ = robust_transform(loss, -y[:, 0])
    with np.errstate(over="ignore"):
        want = f * f
    assert res["residual"].dtype == dtype
    assert res["residual"].tobytes() == want.tobytes()
    representable = np.abs(f.astype(np.float64)) ** 2 <= float(np.finfo(dtype).max) * (1 - 2 * float(np.finfo(dtype).eps))
    assert np.all(np.isfinite(res["residual"][representable]))
    assert np.all(x == 0)


def test_outliers_are_resisted_at_batch_scale():
    """2^14 Gauss4 curves (sigma = 0.05) with 10 % of each curve's rows moved by 5 to 50 (100 to 1000 sigma): soft_l1 and
    huber with w = 1/sigma land near the fit of the clean data, the squared loss does not.

    Calibration (host reference, tests/robust_util.py, on 128 such curves, seeds 50 / 51): relative amplitude error to
    the clean fit, median / 90th percentile: squared 0.45 / 4.4, soft_l1 0.0021 / 0.0071, huber 0.0021 / 0.0065;
    absolute centre error: squared 0.46 / 1.4, soft_l1 0.0021 / 0.0069, huber 0.0019 / 0.0057.  Thresholds: robust
    median < 0.01 and 90th percentile < 0.03, squared median > 0.1."""
    B, sig = 1 << 14, 0.05
    wl = workloads.c2_gauss4(B, noise=sig, seed=50)
    y = with_outliers(wl.y, 0.1, 1.0, seed=51)
    s = eng.settings(np.float64)
    xc = wl.x0.copy(); eng.optimize_batched(s, wl.model, xc, wl.l, wl.u, t=wl.t, y=wl.y)

    def errors(x):
        ea = np.abs(x[:, 0] - xc[:, 0]) / xc[:, 0]; em = np.abs(x[:, 1] - xc[:, 1])
        return [(float(np.median(e)), float(np.percentile(e, 90))) for e in (ea, em)]
    xs = wl.x0.copy(); eng.optimize_batched(s, wl.model, xs, wl.l, wl.u, t=wl.t, y=y)
    for med, _ in errors(xs):
        assert med > 0.1, errors(xs)
    for loss in LOSSES:
        xr = wl.x0.copy(); eng.optimize_batched(s, wl.model, xr, wl.l, wl.u, t=wl.t, y=y, w=np.full(y.shape, 1 / sig), loss=loss)
        for med, p90 in errors(xr):
            assert med < 0.01 and p90 < 0.03, (loss, errors(xr))


# Declares CtaRobust<CtaUser<UserModel<double>>> without defining it: the robust double program fails to compile, every
# other program of the model is unaffected.
NO_ROBUST_DOUBLE = r"""
namespace mirb200 { template <> struct CtaRobust<CtaUser<::UserModel<double>, double>, double>; }
"""


def test_robust_user_model_gives_the_robust_builtin_bits():
    """A user model restating Gauss4 with the built-in operation sequence, under each loss, weighted and not: the bits
    of the robust built-in."""
    mid = eng.compile_model(GAUSS4_USER)
    try:
        wl = workloads.c2_gauss4(512, noise=0.05, seed=75)
        y = with_outliers(wl.y, 0.1, 0.3, seed=76)
        w = 6.0 * sigma_weights(512, wl.m, seed=77, zero_rows=4)
        s = eng.settings(np.float64); s.maxIterations = 5
        for loss in LOSSES:
            for kw in ({}, {"w": w}):
                xb = wl.x0.copy(); rb, _ = eng.optimize_batched(s, wl.model, xb, wl.l, wl.u, t=wl.t, y=y, loss=loss, **kw)
                xu = wl.x0.copy(); ru, _ = eng.optimize_batched(s, mid, xu, wl.l, wl.u, t=wl.t, y=y, loss=loss, **kw)
                assert xb.tobytes() == xu.tobytes() and rb.tobytes() == ru.tobytes(), (loss, float(np.max(rel_err(xb, xu))))
    finally:
        eng.release_model(mid)


def test_robust_user_program_compiles_at_the_first_robust_fit():
    """Registration, plain and weighted fits build no robust program; the first robust fit builds it (here it cannot
    compile, which makes the build visible), for either loss, and the float robust program is unaffected."""
    from mir_optim_b200.engine import B200Error
    mid = eng.compile_model(GAUSS4_USER + NO_ROBUST_DOUBLE)              # (the double fit program is built at registration)
    try:
        wl = workloads.c2_gauss4(64, noise=0.05, seed=78)
        w = sigma_weights(64, wl.m, seed=79)
        s = eng.settings(np.float64); s.maxIterations = 3
        eng.optimize_batched(s, mid, wl.x0.copy(), wl.l, wl.u, t=wl.t, y=wl.y)
        eng.optimize_batched(s, mid, wl.x0.copy(), wl.l, wl.u, t=wl.t, y=wl.y, w=w)
        for loss in LOSSES:
            with pytest.raises(B200Error) as e:
                eng.optimize_batched(s, mid, wl.x0.copy(), wl.l, wl.u, t=wl.t, y=wl.y, loss=loss)
            assert e.value.code == 2 and "does not compile" in str(e.value)
        xf = wl.x0.astype(np.float32)
        eng.optimize_batched(eng.settings(np.float32), mid, xf, wl.l, wl.u, t=wl.t, y=wl.y, loss="soft_l1")
    finally:
        eng.release_model(mid)


def test_host_form_equals_device_form_over_several_staging_chunks():
    """2^17 + 123 robust weighted problems: the host form (staged in chunks of 65536 problems) and the device form give
    the same bits, for each loss."""
    import torch
    B = (1 << 17) + 123
    wl = workloads.c2_gauss4(B, noise=0.05, seed=80)
    y = with_outliers(wl.y, 0.1, 0.3, seed=81)
    w = 6.0 * sigma_weights(B, wl.m, seed=82, zero_rows=2)
    s = eng.settings(np.float64); s.maxIterations = 6
    dev = torch.device("cuda")
    T = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)                            # noqa: E731
    for loss in LOSSES:
        xh = wl.x0.copy(); rh, _ = eng.optimize_batched(s, wl.model, xh, wl.l, wl.u, t=wl.t, y=y, w=w, loss=loss)
        xd = T(wl.x0)
        rd = eng.optimize_batched_device(s, wl.model, xd, T(wl.l), T(wl.u), t=T(wl.t), y=T(y), w=T(w), loss=loss)
        torch.cuda.synchronize()
        assert xd.cpu().numpy().tobytes() == xh.tobytes()
        assert eng.results_from_bytes(rd, np.float64).tobytes() == rh.tobytes()


@pytest.mark.parametrize("loss", LOSSES)
def test_repeatable_independent_of_batch_layout_and_warm_startable(loss):
    """Repeated calls give the same bits; a slice of the batch gives the bits of the same problems inside a permuted
    batch; warm start combines with the loss flag (a zero lambda is a cold start, a previous call's lambda continues
    the fit without raising any residual)."""
    B = 3000
    wl = workloads.c2_gauss4(B, noise=0.05, seed=83)
    y = with_outliers(wl.y, 0.1, 0.3, seed=84)
    w = 6.0 * sigma_weights(B, wl.m, seed=85, zero_rows=3)
    s = eng.settings(np.float64); s.maxIterations = 5

    def run(idx, x0=None, **kw):
        x = (wl.x0[idx] if x0 is None else x0).copy()
        r, _ = eng.optimize_batched(s, wl.model, x, wl.l, wl.u, t=wl.t, y=y[idx], w=w[idx], loss=loss, **kw)
        return x, r
    every = np.arange(B)
    xa, ra = run(every)
    xb, rb = run(every)
    assert xa.tobytes() == xb.tobytes() and ra.tobytes() == rb.tobytes()
    perm = np.random.default_rng(86).permutation(B)
    xp, rp = run(perm)
    sl = np.arange(100, 400)
    xs, rs = run(sl)
    inv = np.argsort(perm)
    assert xp[inv][sl].tobytes() == xs.tobytes() and rp[inv][sl].tobytes() == rs.tobytes()
    assert xp[inv].tobytes() == xa.tobytes()
    cold = ra.copy(); cold["lambda"] = 0
    xw, rw = run(every, results=cold, warm_start=True)
    assert xw.tobytes() == xa.tobytes() and rw.tobytes() == ra.tobytes()
    cont = ra.copy()
    xc, rc = run(every, x0=xa, results=cont, warm_start=True)
    ok = np.isfinite(ra["residual"]) & (ra["status"] >= 0)
    assert np.all(rc["residual"][ok] <= ra["residual"][ok])
    xr, rr = run(every, x0=xa)                                                # a cold restart from the same x
    assert not (xr.tobytes() == xc.tobytes() and rr.tobytes() == rc.tobytes())
