"""Host reference of the robust losses (MIR_MODEL_LOSS_SOFT_L1 / MIR_MODEL_LOSS_HUBER, include/mir_optim_b200.h): the
oracle LM (the reference restated, oracle/lm_oracle.cpp) run with f~ = sign(u) sqrt(rho(u^2)) and J~ = g(u) (w J), u = w r,
where r and J are the oracle's own host callbacks (the device functors' bits) and w scales as in weights_util.  Every step
is one IEEE operation on numpy arrays of the problem's dtype, in the header's order (numpy does not contract), so the bits
are the device's.  TEST INFRASTRUCTURE ONLY."""
import numpy as np

from cov_util import oracle_callbacks
from mir_optim_b200.api import ReferenceAPI
from mir_optim_b200.engine import RESULT_DTYPES


def robust_transform(loss, u):
    """(f~, g) of u (an array of float64 or float32) for loss "soft_l1" or "huber", with the header's operation sequence."""
    u = np.asarray(u)
    T = u.dtype.type
    a = np.abs(u)
    inner = a <= T(1)                      # False for NaN: a NaN takes the a > 1 branch, as on the device
    with np.errstate(all="ignore"):
        if loss == "huber":
            F = T(2) * np.sqrt(T(0.5) * (a - T(0.5)))
            g = T(1) / F
            f = np.where(u < 0, -F, F)
            return np.where(inner, u, f), np.where(inner, T(1), g)
        if loss != "soft_l1":
            raise ValueError(loss)
        s = np.sqrt(T(1) + a * a)
        r = np.sqrt(T(0.5) * (s + T(1)))
        f_in, g_in = u / r, r / s
        q = T(1) / a
        c = np.sqrt(T(1) + q * q)
        rq = np.sqrt(T(0.5) * (c + q))
        b = np.sqrt(a)
        F = b / rq
        g_out = rq / (b * c)
        f_out = np.where(u < 0, -F, F)
    return np.where(inner, f_in, f_out), np.where(inner, g_in, g_out)


def robust_callbacks(olib, model, dtype, t, y, loss, w=None, aux=None, param=0.0, fd=False):
    """f~(b, x) and g~(b, x) (None when fd) of problem b under `loss`, weighted by w (batch, m) when given."""
    f, g = oracle_callbacks(olib, model, dtype, t, y, aux=aux, param=param, fd=fd)
    w = None if w is None else np.ascontiguousarray(w, dtype=dtype)

    def u_of(b, x):
        r = f(b, x)
        return r if w is None else w[b] * r

    def fr(b, x):
        return robust_transform(loss, u_of(b, x))[0]

    def gr(b, x):
        _, gam = robust_transform(loss, u_of(b, x))
        J = g(b, x)
        wJ = J if w is None else w[b][:, None] * J
        return gam[:, None] * wJ

    return fr, (None if fd else gr)


def oracle_batched_robust(olib, settings, model, x0, l, u, loss, t=None, y=None, w=None, fd_jacobian=False, aux=None, param=0.0):
    """The oracle LM on every problem of a robust batch.  Same contract as oracle_util.oracle_batched: (x, results)."""
    x = np.array(x0, copy=True, order="C")
    dt = x.dtype
    batch, n = x.shape
    m = np.asarray(y).shape[1]
    fr, gr = robust_callbacks(olib, model, dt, t, y, loss, w=w, aux=aux, param=param, fd=fd_jacobian)
    l = np.ascontiguousarray(np.broadcast_to(np.asarray(l, dtype=dt), (batch, n)))
    u = np.ascontiguousarray(np.broadcast_to(np.asarray(u, dtype=dt), (batch, n)))
    api = ReferenceAPI(olib)
    results = np.empty(batch, dtype=RESULT_DTYPES[dt])
    for b in range(batch):
        def f(xv, yv, b=b):
            yv[:] = fr(b, xv)

        def g(xv, J, b=b):
            J[:] = gr(b, xv)
        xb = x[b].copy()
        r = api.optimize_least_squares(settings, m, xb, l[b].copy(), u[b].copy(), f, None if fd_jacobian else g)
        x[b] = xb
        results[b] = (r.status, r.iterations, r.fCalls, r.gCalls, r.residual, r.lambda_)
    return x, results


def with_outliers(y, frac, scale, seed):
    """y with a fraction `frac` of each problem's rows replaced by gross outliers: y + scale * (5 .. 50) * (+-1)."""
    rng = np.random.default_rng(seed)
    y = np.array(y, dtype=np.float64, copy=True)
    B, m = y.shape
    k = max(1, int(round(frac * m)))
    for b in range(B):
        idx = rng.choice(m, k, replace=False)
        y[b, idx] += scale * rng.uniform(5.0, 50.0, k) * rng.choice([-1.0, 1.0], k)
    return y
