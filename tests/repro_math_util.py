"""References for the reproducible exp and the pivot square root (csrc/repro_math.cuh, oracle/repro_math.h).

Errors are measured in units in the last place of the exact value v: |y - v| / ulp(v), ulp(v) = 2^(max(floor(log2 v), emin)
- p).  v (e^x, sqrt(a), 1/sqrt(a), 1/l) is computed by `decimal` at 60 significant digits; everything after that is exact: a
float converts to Decimal without rounding, floor(log2 v) is found by exact comparisons with powers of two, and the
difference and the quotient are taken at a precision wide enough to hold every digit of their operands.  So a reported
error is the true one to within about 1e-40 ulp.

Also the argument sets shared by the CPU and GPU tests: ulp windows around the thresholds of the exp, the rint ties
x*log2(e) = k + 1/2, and NaNs with payloads.
"""
import ctypes as C
import decimal
import math
from decimal import Decimal as D

import numpy as np

REF = decimal.Context(prec=60)            # e^x, sqrt, 1/sqrt
EXACT = decimal.Context(prec=2200)        # |y - v| and the ratio: every digit of a subnormal double fits

# p (stored mantissa bits), emin, and the integer views
FMT = {np.float64: (52, -1022, np.uint64, np.int64), np.float32: (23, -126, np.uint32, np.int32)}
LN2 = REF.ln(D(2))


def ln2_times(k):
    return REF.multiply(D(k), LN2)


def fmt(dt):
    return FMT[np.dtype(dt).type]


def max_finite(dt):
    return D(float(np.finfo(dt).max))


def two(e):
    """2^e as an exact Decimal (e >= -1074, e <= 1023)."""
    return D(math.ldexp(1.0, e))


def ulp(v, dt):
    """ulp of the positive finite Decimal v in format dt, with the exponent clamped at emin (subnormal spacing)."""
    p, emin = fmt(dt)[:2]
    if v < two(emin):
        return two(emin - p)
    e = math.frexp(float(v))[1] - 1                  # estimate, then make floor(log2 v) exact
    while two(e) > v:
        e -= 1
    while e + 1 <= 1023 and two(e + 1) <= v:
        e += 1
    return two(e - p)


def ulp_err(y, v, dt):
    """|y - v| / ulp(v) for finite y and finite positive v, exactly (see the module doc)."""
    return float(EXACT.divide(abs(EXACT.subtract(D(float(y)), v)), ulp(v, dt)))


def overflow_limit(dt):
    """2^(emax+1): the value that inf stands for when an error is measured against an overflowing result."""
    return EXACT.power(D(2), 1024 if np.dtype(dt) == np.float64 else 128)


def exp_exact(x):
    return REF.exp(D(float(x)))


def exp_check(x, y, dt):
    """Checks one result of the exp against e^x: < 1 ulp, faithful into the subnormals and zero below them; inf
    exactly where the correctly rounded e^x overflows, except in the one-ulp boundary case (e^x between the largest
    finite value and 2^(emax+1), where both the largest finite value and inf are within one ulp).
    Returns None if the result is acceptable, else a description."""
    x = dt(x); y = dt(y)
    if np.isnan(x):
        return None if np.isnan(y) and x.tobytes() == y.tobytes() else f"NaN payload not kept: {y!r}"
    if abs(x) > 2000:                                # e^x is far past overflow, or far below half the smallest subnormal
        want = dt(np.inf) if x > 0 else dt(0.0)
        return None if y.tobytes() == want.tobytes() else f"exp({x}) = {y!r}"
    v = exp_exact(x)
    big = max_finite(dt)
    cr_overflows = v >= EXACT.add(big, EXACT.divide(ulp(big, dt), 2))          # round to nearest: these round to inf
    if np.isinf(y):
        if y < 0 or not v > big:
            return f"inf where e^x = {v:.6e} is below the largest finite value"
        return None
    if cr_overflows and not v < overflow_limit(dt):
        return f"finite {y!r} where e^x = {v:.6e} overflows by more than an ulp"
    if y < 0 or (y == 0 and np.signbit(y)):
        return f"negative result {y!r}"
    err = ulp_err(y, v, dt)
    return None if err < 1.0 else f"error {err:.4f} ulp (y = {float(y).hex()}, e^x = {v:.20e})"


def sqrt_rcp_errs(a, l, r, dt):
    """Errors in ulp of l against sqrt(a), of r against 1/l (the reciprocal of the pivot actually used, which is what
    LAPACK's potf2 scales the column by: 1 / the rounded sqrt), and of r against 1/sqrt(a), for a positive finite a
    (inf where l or r is not finite)."""
    if not (np.isfinite(l) and np.isfinite(r) and l > 0):
        return math.inf, math.inf, math.inf
    s = REF.sqrt(D(float(a)))
    return ulp_err(l, s, dt), ulp_err(r, REF.divide(D(1), D(float(l))), dt), ulp_err(r, REF.divide(D(1), s), dt)


# ---- argument sets ------------------------------------------------------------------------------------------------

def around(x0, n, dt):
    """The 2n + 1 values of dt nearest to x0 (n ulps either side, x0 first rounded to dt), same sign as x0."""
    it = fmt(dt)[3]
    a = np.array([abs(x0)], dtype=dt).view(it).astype(np.int64)[0]
    r = a + np.arange(-n, n + 1, dtype=np.int64)
    r = r[(r >= 0) & (r < np.array([np.inf], dtype=dt).view(it).astype(np.int64)[0])]
    v = r.astype(it).view(dt)
    return -v if x0 < 0 else v


def nearest(d, dt):
    """Decimal -> nearest value of dt."""
    return np.dtype(dt).type(float(d))


def thresholds(dt):
    """Named arguments where the exp switches behaviour, each as the nearest value of dt."""
    if np.dtype(dt) == np.float64:
        t = {"cutoff -745.2": D("-745.2"), "2^-1075 crossing": ln2_times(-1075), "subnormal onset": ln2_times(-1022),
             "tp ki = -1000": ln2_times(-1000), "tp ki = -1000 switch": ln2_times("-1000.5"),
             "tp ki = +1000": ln2_times(1000), "tp ki = +1000 switch": ln2_times("1000.5"),
             "conv -700": D(-700), "conv +700": D(700), "inf cutoff": D("709.782712893384"),
             "ln(DBL_MAX)": REF.ln(max_finite(np.float64))}
    else:
        t = {"cutoff -104": D(-104), "2^-150 crossing": ln2_times(-150), "subnormal onset": ln2_times(-126),
             "tp ki = -120": ln2_times(-120), "tp ki = -120 switch": ln2_times("-120.5"),
             "tp ki = +120": ln2_times(120), "tp ki = +120 switch": ln2_times("120.5"),
             "conv -80": D(-80), "conv +80": D(80), "inf cutoff": D(float(np.float32(88.72284))),
             "ln(FLT_MAX)": REF.ln(max_finite(np.float32))}
    return {k: nearest(v, dt) for k, v in t.items()}


def tie_windows(dt, n):
    """n ulps either side of every x with x*log2(e) = k + 1/2, k over the range where the exp is evaluated."""
    ks = range(-1075, 1025) if np.dtype(dt) == np.float64 else range(-150, 129)
    return np.concatenate([around(nearest(ln2_times(k + D("0.5")), dt), n, dt) for k in ks])


def specials(dt):
    """NaNs with payloads of both signs (quiet and signalling), +-inf, +-0, +-max, +-min subnormal."""
    if np.dtype(dt) == np.float64:
        nans = np.array([0x7FF8000000000000, 0x7FF8000000000001, 0x7FFDEADBEEF01234, 0x7FF0000000000001, 0x7FF4000000000000,
                         0xFFF8000000000000, 0xFFF8000000000001, 0xFFFCAFEBABE56789, 0xFFF0000000000001], dtype=np.uint64)
    else:
        nans = np.array([0x7FC00000, 0x7FC00001, 0x7FDEAD12, 0x7F800001, 0x7FA00000,
                         0xFFC00000, 0xFFC00001, 0xFFCAFE34, 0xFF800001], dtype=np.uint32)
    fi = np.finfo(dt)
    tiny = np.array([1], dtype=fmt(dt)[2]).view(dt)[0]
    rest = np.array([np.inf, -np.inf, 0.0, -0.0, fi.max, -fi.max, tiny, -tiny], dtype=dt)
    return np.concatenate([nans.view(dt), rest])


def log_uniform(rng, n, lo_exp, hi_exp, dt):
    """|x| = 2^u with u uniform in [lo_exp, hi_exp), random signs; reaches the subnormals when lo_exp is below emin."""
    u = rng.uniform(lo_exp, hi_exp, n)
    mag = np.exp2(u)                                # float64: exact enough, and subnormal down to 2^-1074
    x = (mag * rng.choice([-1.0, 1.0], n)).astype(dt)
    return x


def oracle_exp(lib, x):
    """oracle_exp_repro_{d,s}: the host restatement, elementwise."""
    x = np.ascontiguousarray(x)
    y = np.empty_like(x)
    fn = lib.oracle_exp_repro_d if x.dtype == np.float64 else lib.oracle_exp_repro_s
    fn.argtypes = [C.c_size_t, C.c_void_p, C.c_void_p]; fn.restype = None
    fn(x.size, x.ctypes.data, y.ctypes.data)
    return y
