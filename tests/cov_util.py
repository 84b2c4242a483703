"""Host reference of the batched covariance (definition in include/mir_optim_b200.h, mir_b200_covariance_batched_d).

Residuals and analytic Jacobians come from the oracle's host callbacks oracle_model_{f,g}_{d,s}, which return the
device functors' bits (DESIGN.md section 2); the central difference is restated with the fit's bound clamp
(least_squares.d:1030-1047).  Models without an oracle callback (user models) pass `f` / `g` as Python callables.
TEST INFRASTRUCTURE ONLY."""
import ctypes as C

import numpy as np


class _Ctx(C.Structure):
    _fields_ = [("model", C.c_int), ("t", C.c_void_p), ("y", C.c_void_p), ("aux", C.c_void_p), ("param", C.c_double)]


def oracle_callbacks(olib, model, dtype, t, y, aux=None, param=0.0, fd=False):
    """f(b, x) -> r and g(b, x) -> J (None when fd) of problem b, through the oracle's host callbacks."""
    sfx = "d" if np.dtype(dtype) == np.float64 else "s"
    F = getattr(olib, f"oracle_model_f_{sfx}"); G = getattr(olib, f"oracle_model_g_{sfx}")
    for fn in (F, G):
        fn.argtypes = [C.c_void_p, C.c_size_t, C.c_size_t, C.c_void_p, C.c_void_p]; fn.restype = None
    t = None if t is None else np.ascontiguousarray(t, dtype=dtype)
    y = np.ascontiguousarray(y, dtype=dtype)
    aux = None if aux is None else np.ascontiguousarray(aux, dtype=dtype)
    m = y.shape[1]

    def ctx(b):
        tb = None if t is None else (t[b] if t.ndim == 2 else t)
        ab = None if aux is None else (aux[b] if aux.ndim == 2 else aux)
        c = _Ctx(int(model), None if tb is None else tb.ctypes.data, y[b].ctypes.data, None if ab is None else ab.ctypes.data, float(param))
        return c, (tb, ab)                      # (keep the arrays alive with the context)

    def f(b, x):
        c, keep = ctx(b); x = np.ascontiguousarray(x, dtype=dtype); r = np.empty(m, dtype=dtype)
        F(C.addressof(c), m, x.shape[0], x.ctypes.data, r.ctypes.data)
        return r

    def g(b, x):
        c, keep = ctx(b); x = np.ascontiguousarray(x, dtype=dtype); J = np.empty((m, x.shape[0]), dtype=dtype)
        G(C.addressof(c), m, x.shape[0], x.ctypes.data, J.ctypes.data)
        return J

    return f, (None if fd else g)


def fd_jacobian(f, b, x, l, u, eps, free):
    """The reference's central difference (least_squares.d:1018-1049) on the free columns, in the problem's precision."""
    dt = x.dtype.type
    r0 = f(b, x)
    J = np.zeros((r0.shape[0], x.shape[0]), dtype=x.dtype)
    for j in np.nonzero(free)[0]:
        xmh = np.maximum(dt(x[j] - dt(eps)), l[j]); xph = np.minimum(dt(x[j] + dt(eps)), u[j])
        twh = dt(xph - xmh)
        if twh != 0:
            xp = x.copy(); xp[j] = xph; fp = f(b, xp)
            xm = x.copy(); xm[j] = xmh; fm = f(b, xm)
            J[:, j] = (fp - fm) * (dt(1) / twh)
    return J


def potf2_lower(S):
    """LAPACK ?potf2 (lower) in double; returns (L, index of the failing pivot or -1)."""
    A = np.array(S, dtype=np.float64, copy=True)
    n = A.shape[0]
    for j in range(n):
        d = A[j, j]
        if not d > 0:
            return A, j
        ljj = np.sqrt(d); A[j, j] = ljj
        A[j + 1:, j] /= ljj
        A[j + 1:, j + 1:] -= np.outer(A[j + 1:, j], A[j + 1:, j])
    return np.tril(A), -1


def cov_one(r, J, free, m, scaled=True):
    """(cov n x n double, info, kappa of the scaled free block) from residuals r and Jacobian J of one problem."""
    n = J.shape[1]
    cov = np.zeros((n, n))
    fi = np.nonzero(free)[0]; nf = len(fi)
    if not (np.all(np.isfinite(r)) and np.all(np.isfinite(J[:, fi]))):
        cov[np.ix_(fi, fi)] = np.nan
        return cov, -2, np.nan
    if scaled and m <= nf:
        cov[np.ix_(fi, fi)] = np.inf
        return cov, -1, np.nan
    if nf == 0:
        return cov, 0, 1.0
    JF = J[:, fi].astype(np.float64)
    A = JF.T @ JF
    rr = float(np.dot(r.astype(np.float64), r.astype(np.float64)))
    d = np.diag(A)
    sc = np.where(d > 0, 1.0 / np.sqrt(np.where(d > 0, d, 1.0)), 0.0)
    S = A * sc[:, None] * sc[None, :]
    L, fail = potf2_lower(S)
    if fail >= 0:
        cov[np.ix_(fi, fi)] = np.nan
        return cov, int(fi[fail]) + 1, np.inf
    import scipy.linalg
    W = scipy.linalg.solve_triangular(L, np.eye(nf), lower=True)
    Sinv = W.T @ W
    s2 = rr / (m - nf) if scaled else 1.0
    cov[np.ix_(fi, fi)] = s2 * Sinv * sc[:, None] * sc[None, :]
    return cov, 0, float(np.linalg.cond(S))


def cov_reference(f, g, x, l, u, eps, scaled=True):
    """Reference of every problem: returns (cov (batch, n, n) double, info int32[batch], kappa[batch])."""
    x = np.asarray(x); batch, n = x.shape
    l = np.broadcast_to(np.asarray(l, dtype=x.dtype), (batch, n)); u = np.broadcast_to(np.asarray(u, dtype=x.dtype), (batch, n))
    cov = np.zeros((batch, n, n)); info = np.zeros(batch, dtype=np.int32); kap = np.ones(batch)
    for b in range(batch):
        xb = x[b].copy()
        free = (l[b] < xb) & (xb < u[b])
        if not np.all(np.isfinite(xb)):
            cov[b][np.ix_(free, free)] = np.nan; info[b] = -2; kap[b] = np.nan
            continue
        r = f(b, xb)
        J = g(b, xb) if g is not None else fd_jacobian(f, b, xb, l[b], u[b], eps, free)
        cov[b], info[b], kap[b] = cov_one(r, J, free, r.shape[0], scaled)
    return cov, info, kap


def cov_error(C_, R):
    """max over problems of max_ij |C_ij - R_ij| / sqrt(R_ii R_jj) on the entries where R is nonzero on the diagonal."""
    C_ = np.asarray(C_, dtype=np.float64); R = np.asarray(R, dtype=np.float64)
    d = np.sqrt(np.abs(np.einsum("bii->bi", R)))
    den = d[:, :, None] * d[:, None, :]
    e = np.where(den > 0, np.abs(C_ - R) / np.where(den > 0, den, 1.0), np.abs(C_ - R))
    return e.reshape(len(e), -1).max(axis=1)


def cov_bound(kappa, dtype):
    """The parity bound: max(1e-13, 32 kappa 2^-52), plus 2^-23 for the final rounding of a float result."""
    b = np.maximum(1e-13, 32.0 * np.asarray(kappa) * 2.0 ** -52)
    return b + (2.0 ** -23 if np.dtype(dtype) == np.float32 else 0.0)
