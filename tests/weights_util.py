"""Host reference of weighted least squares (MIR_MODEL_WEIGHTED, include/mir_optim_b200.h): the oracle LM (the reference
restated, oracle/lm_oracle.cpp) run with f~ = w (.) f and J~ = w[:, None] (.) J, where f and J are the oracle's own host
callbacks oracle_model_{f,g}_{d,s} (the device functors' bits).  Each product is one IEEE multiplication in the
problem's precision, as the device's mul_rn; the finite-difference Jacobian is the reference's, taken of f~.
TEST INFRASTRUCTURE ONLY."""
import numpy as np

from cov_util import oracle_callbacks
from mir_optim_b200.api import ReferenceAPI
from mir_optim_b200.engine import RESULT_DTYPES


def weighted_callbacks(olib, model, dtype, t, y, w, aux=None, param=0.0, fd=False):
    """f~(b, x) -> w_b (.) r and g~(b, x) -> w_b[:, None] (.) J (None when fd) of problem b."""
    f, g = oracle_callbacks(olib, model, dtype, t, y, aux=aux, param=param, fd=fd)
    w = np.ascontiguousarray(w, dtype=dtype)

    def fw(b, x):
        return w[b] * f(b, x)

    def gw(b, x):
        return w[b][:, None] * g(b, x)

    return fw, (None if fd else gw)


def oracle_batched_weighted(olib, settings, model, x0, l, u, t=None, y=None, w=None, fd_jacobian=False, aux=None, param=0.0):
    """The oracle LM on every problem of a weighted batch.  Same contract as oracle_util.oracle_batched: (x, results)."""
    x = np.array(x0, copy=True, order="C")
    dt = x.dtype
    batch, n = x.shape
    m = np.asarray(y).shape[1]
    fw, gw = weighted_callbacks(olib, model, dt, t, y, w, aux=aux, param=param, fd=fd_jacobian)
    l = np.ascontiguousarray(np.broadcast_to(np.asarray(l, dtype=dt), (batch, n)))
    u = np.ascontiguousarray(np.broadcast_to(np.asarray(u, dtype=dt), (batch, n)))
    api = ReferenceAPI(olib)
    results = np.empty(batch, dtype=RESULT_DTYPES[dt])
    for b in range(batch):
        def f(xv, yv, b=b):
            yv[:] = fw(b, xv)

        def g(xv, J, b=b):
            J[:] = gw(b, xv)
        xb = x[b].copy()
        r = api.optimize_least_squares(settings, m, xb, l[b].copy(), u[b].copy(), f, None if fd_jacobian else g)
        x[b] = xb
        results[b] = (r.status, r.iterations, r.fCalls, r.gCalls, r.residual, r.lambda_)
    return x, results


def sigma_weights(batch, m, seed, zero_rows=0, dtype=np.float64):
    """w = 1/sigma with sigma varying over a decade within each problem, and `zero_rows` random rows of each problem at 0."""
    rng = np.random.default_rng(seed)
    sigma = 10.0 ** rng.uniform(-1.0, 0.0, (batch, m))
    w = 1.0 / sigma
    for b in range(batch):
        if zero_rows:
            w[b, rng.choice(m, zero_rows, replace=False)] = 0.0
    return w.astype(dtype)
