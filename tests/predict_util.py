"""Host reference of the batched prediction (definition in include/mir_optim_b200.h, mir_b200_predict_batched_d).

Values come from the oracle's host callbacks oracle_model_f_{d,s} with y = 0 (the device functors' bits, DESIGN.md
section 2), through cov_util.oracle_callbacks; the spline is evaluated with m = k + 1 rows and param = 0 and its last row
is dropped.  Gradients are the oracle's analytic Jacobian rows, or cov_util.fd_jacobian (the reference's central
difference with the bound clamp) on that f.  Models without an oracle callback pass `f` / `g` as Python callables.

numpy cannot restate the device's fma chain bit for bit, so se^2 is held to a bound rather than to bits:
    |se^2 - q| <= c n_F^2 2^-52 sum_a sum_c |g_a| |C_ac| |g_c|,   c = 2,
plus 2^-22 q for a float result.  The device's two nested fma chains of length n_F are within n_F 2^-52 of that sum
(2 n_F unit roundoffs of 2^-53), and numpy's einsum, in its own order and without fma, within about n_F^2 2^-53 of it;
c = 2 covers both with room.  Rounding se once to float moves se^2 by at most 2^-23 relative; 2^-22 covers it.
TEST INFRASTRUCTURE ONLY."""
import numpy as np

from cov_util import fd_jacobian, oracle_callbacks

C_BOUND = 2.0


def trailing_rows(model):
    from mir_optim_b200 import ModelId
    return 1 if int(model) == int(ModelId.SPLINE) else 0


def predict_callbacks(olib, model, dtype, t, batch, aux=None, fd=False):
    """(f, g, k) of the prediction at the abscissae t ((k,) or (batch, k)): f(b, x) and g(b, x) return all m = k (+ 1 for
    the spline) rows, with y = 0 and param = 0; g is None for finite differences (always for the spline)."""
    k = np.shape(t)[-1]
    extra = trailing_rows(model)
    f, g = oracle_callbacks(olib, model, dtype, t, np.zeros((batch, k + extra)), aux=aux, param=0.0, fd=fd or extra > 0)
    return f, g, k


def full_lower(cov):
    """The symmetric matrix the device reads: the lower triangle of cov mirrored (the upper triangle is never read)."""
    L = np.tril(np.asarray(cov, dtype=np.float64))
    return L + np.swapaxes(np.tril(L, -1), -1, -2)


def predict_reference(f, g, x, l, u, eps, cov, k):
    """Every problem's (value (batch, k) in T, q (batch, k) double, bound (batch, k) on |se^2 - q| before the rounding of se)."""
    x = np.asarray(x); batch, n = x.shape
    l = np.broadcast_to(np.asarray(l, dtype=x.dtype), (batch, n)); u = np.broadcast_to(np.asarray(u, dtype=x.dtype), (batch, n))
    value = np.empty((batch, k), dtype=x.dtype)
    q = np.zeros((batch, k)); bound = np.zeros((batch, k))
    for b in range(batch):
        xb = x[b].copy()
        free = (l[b] < xb) & (xb < u[b])
        value[b] = f(b, xb)[:k]
        if cov is None:
            continue
        fi = np.nonzero(free)[0]; nf = len(fi)
        if nf == 0:
            continue
        J = g(b, xb) if g is not None else fd_jacobian(f, b, xb, l[b], u[b], eps, free)
        G = J[:k][:, fi].astype(np.float64)
        Cf = full_lower(cov[b])[np.ix_(fi, fi)]
        q[b] = np.einsum("ia,ac,ic->i", G, Cf, G)
        bound[b] = C_BOUND * nf * nf * 2.0 ** -52 * np.einsum("ia,ac,ic->i", np.abs(G), np.abs(Cf), np.abs(G))
    return value, q, bound


def se_within_bound(se, q, bound, dtype):
    """Whether every se satisfies |se^2 - q| <= bound (+ 2^-22 q for float); returns (ok, worst ratio)."""
    s2 = np.asarray(se, dtype=np.float64) ** 2
    b = bound + (2.0 ** -22 * q if np.dtype(dtype) == np.float32 else 0.0)
    err = np.abs(s2 - q)
    ratio = np.where(b > 0, err / np.where(b > 0, b, 1.0), np.where(err > 0, np.inf, 0.0))
    return bool(np.all(ratio <= 1.0)), float(ratio.max())
