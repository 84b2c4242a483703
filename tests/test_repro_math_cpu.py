"""The host restatement of the reproducible exp (oracle/repro_math.h) against `decimal`, no GPU.

Every device form of the exp is held bit for bit against this restatement (tests/test_gpu_repro_math.py), so its accuracy
is the accuracy of every residual functor: error below one ulp of e^x (measured exactly, tests/repro_math_util.py) on
ordinary, subnormal-result and threshold arguments; inf exactly where the correctly rounded e^x overflows (up to the
one-ulp boundary case); +0 below the subnormal range; exp(+-0) = 1, exp(-inf) = +0, exp(+inf) = inf; NaNs come back with
their payload.  Plus the argument checks of the device hook, which fail before any device is needed."""
import ctypes as C

import numpy as np
import pytest

from repro_math_util import (around, exp_check, exp_exact, log_uniform, max_finite, oracle_exp, specials, thresholds,
                             tie_windows, EXACT, ulp)

DTYPES = [np.float64, np.float32]
RANGE = {np.float64: (-745.2, 709.782712893384, -708.4), np.float32: (-104.0, 88.72284, -87.34)}   # lo, inf cutoff, subnormal onset


def _check_all(x, y, dt):
    bad = []
    for a, b in zip(x, y):
        msg = exp_check(a, b, dt)
        if msg is not None:
            bad.append(f"x = {float(a).hex()}: {msg}")
            if len(bad) >= 5:
                break
    assert not bad, "\n".join(bad)


@pytest.mark.parametrize("dt", DTYPES, ids=["double", "float"])
def test_exp_restatement_is_within_one_ulp(oracle_lib, dt):
    rng = np.random.default_rng(20261021)
    lo, hi, sub = RANGE[dt]
    tiny_exp = -1074 if dt == np.float64 else -149
    x = np.concatenate([
        rng.uniform(lo, hi, 3000).astype(dt),                       # the whole evaluated range
        rng.uniform(-1.0, 1.0, 1000).astype(dt),                    # k = 0, +-1
        rng.uniform(lo, sub, 2000).astype(dt),                      # subnormal results
        log_uniform(rng, 1000, tiny_exp, 0, dt),                    # |x| down to the smallest subnormal: e^x near 1
        np.concatenate([around(t, 32, dt) for t in thresholds(dt).values()]),
        tie_windows(dt, 2),                                         # x log2(e) near k + 1/2: the rint ties
    ])
    x = x[(x > lo) & (x <= hi)]
    _check_all(x, oracle_exp(oracle_lib, x), dt)


@pytest.mark.parametrize("dt", DTYPES, ids=["double", "float"])
def test_exp_restatement_overflows_where_the_rounded_value_does(oracle_lib, dt):
    t = thresholds(dt)
    x = np.unique(np.concatenate([around(t["inf cutoff"], 4096, dt), around(t[next(k for k in t if k.startswith("ln("))], 4096, dt)]))
    y = oracle_exp(oracle_lib, x)
    _check_all(x, y, dt)
    big = max_finite(dt)
    cr_inf = np.array([exp_exact(a) >= EXACT.add(big, EXACT.divide(ulp(big, dt), 2)) for a in x])
    assert cr_inf.any() and not cr_inf.all()
    differ = x[np.isinf(y) != cr_inf]
    assert differ.size <= 1, [float(a).hex() for a in differ]      # at most the one argument at the boundary
    assert np.all(np.diff(np.isinf(y).astype(int)) >= 0)           # finite below, inf above: one switch


@pytest.mark.parametrize("dt", DTYPES, ids=["double", "float"])
def test_exp_restatement_special_values(oracle_lib, dt):
    lo = RANGE[dt][0]
    rng = np.random.default_rng(7)
    below = np.concatenate([rng.uniform(-1e4, lo, 1000).astype(dt), around(lo, 64, dt), [np.finfo(dt).min]]).astype(dt)
    below = below[below <= lo]
    y = oracle_exp(oracle_lib, below)
    assert np.all(y.view(f"u{np.dtype(dt).itemsize}") == 0), "exp below the subnormal range must be +0"
    s = specials(dt)
    _check_all(s, oracle_exp(oracle_lib, s), dt)                   # NaN payloads, +-inf, +-0, +-max, +-min subnormal
    z = oracle_exp(oracle_lib, np.array([0.0, -0.0, -np.inf, np.inf], dtype=dt))
    assert z.tobytes() == np.array([1.0, 1.0, 0.0, np.inf], dtype=dt).tobytes()


def test_math_hook_argument_errors():
    import mir_optim_b200
    eng = mir_optim_b200.engine
    x = np.zeros(4); y = np.zeros(4)
    for sfx in ("d", "s"):
        fn = getattr(eng.lib, f"mir_b200_math_hook_{sfx}")
        for v in (-1, 8):
            assert fn(v, 4, x.ctypes.data, y.ctypes.data, y.ctypes.data, -1) == 3                  # MIR_B200_EUNSUPPORTED
            assert eng.lib.mir_b200_last_error().decode()
        assert fn(0, 4, None, y.ctypes.data, None, -1) == 2                                       # MIR_B200_EINVAL
        assert fn(0, 4, x.ctypes.data, None, None, -1) == 2
        assert fn(7, 4, x.ctypes.data, y.ctypes.data, None, -1) == 2                              # sqrt_rcp needs y2
        assert "null" in eng.lib.mir_b200_last_error().decode()
        if eng.device_count() == 0:
            assert fn(0, 4, x.ctypes.data, y.ctypes.data, None, -1) == 1                          # MIR_B200_ENODEVICE
