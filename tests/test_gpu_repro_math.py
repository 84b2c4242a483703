"""Every device form of the reproducible exp, and the mux kernel's pivot square root, on their own (csrc/math_hooks.cu).

repro_math.cuh promises that its exp returns the bits of the host restatement oracle/repro_math.h for every input: that
is what lets the finite-difference kernels match the oracle to 1e-10 while residual differences are amplified ~3e7.  The
header has five forms of it (scalar with early returns, out of line, inlined, K interleaved chains, and the warp-vote fast
path), and each is checked here bit for bit against the restatement, which tests/test_repro_math_cpu.py checks against
`decimal`:
  * float: every argument with -104 < x <= 88.8f (about 2.2e9 bit patterns), plus NaN payloads, +-inf, +-max;
  * double: ~1.45e7 arguments: uniform over the evaluated range and [-1, 1], log-uniform |x| down to 2^-1074, 4096 ulps
    around each threshold (the -745.2 cut-off, the 2^-1075 rounding crossing, the subnormal onset, the ki = +-1000 switch
    of exp_repro_tp, the +-700 fast-path switch, the inf cut-off, ln(DBL_MAX)), 64 ulps around every rint tie
    x log2(e) = k + 1/2, and NaNs with payloads of both signs; float gets the same windows;
  * the fast path of exp_repro_many_conv against its general path on the same arguments, with the warps laid out once
    all in range and once with one out-of-range lane each, and whole warps just past the switch;
  * mux_sqrt_rcp: l within one ulp of sqrt(a) and r within one ulp of 1/l (measured exactly against `decimal`), over
    all positive finite a, subnormals and the tiny-pivot rescaling switch included.
"""
import numpy as np
import pytest

from repro_math_util import (around, fmt, log_uniform, oracle_exp, specials, sqrt_rcp_errs, thresholds, tie_windows,
                             two)

pytestmark = pytest.mark.gpu

EXP_VARIANTS = {0: "exp_repro_tp", 1: "exp_repro", 2: "exp_repro_inl", 3: "exp_repro_many<4>", 4: "exp_repro_many<16>",
                5: "exp_repro_many_conv<4>", 6: "exp_repro_many_conv<16>"}
CONV_K = {5: 4, 6: 16}
FAST_LIMIT = {np.float64: 700.0, np.float32: 80.0}     # |x| below this for every lane of a warp: the conv fast path
SQRT_RCP = 7


@pytest.fixture(scope="module")
def eng():
    import mir_optim_b200
    assert mir_optim_b200.engine.device_count() > 0, "no CUDA device"
    return mir_optim_b200.engine


def bits(a):
    return a.view(np.uint64 if a.dtype == np.float64 else np.uint32)


def mismatch(x, y, yo):
    """None when y and yo agree bit for bit, else the count and the first mismatching argument (hex)."""
    bad = np.flatnonzero(bits(y) != bits(yo))
    if bad.size == 0:
        return None
    i = bad[0]
    return (f"{bad.size} of {x.size} differ; first at x = {float(x[i]).hex()} (bits {int(bits(x[i:i + 1])[0]):#x}): "
            f"device {float(y[i]).hex()}, host {float(yo[i]).hex()}")


def assert_variants_match_oracle(eng, oracle_lib, x, what, variants=EXP_VARIANTS):
    yo = oracle_exp(oracle_lib, x)
    errs = []
    for v in variants:
        msg = mismatch(x, eng.math_hook(x, v), yo)
        if msg:
            errs.append(f"{EXP_VARIANTS[v]} (variant {v}), {what}: {msg}")
    assert not errs, "\n".join(errs)


# ---- float: every argument -------------------------------------------------------------------------------------------

def test_float_exp_every_argument(eng, oracle_lib):
    """All float bit patterns with -104 < x <= 88.8f (beyond them the results are 0 and inf by a compare), in chunks."""
    hi_pos = int(bits(np.array([88.8], dtype=np.float32))[0])
    neg_104 = int(bits(np.array([-104.0], dtype=np.float32))[0])
    chunk = 1 << 26
    for lo, hi in ((0, hi_pos + 1), (0x80000000, neg_104)):     # +0 .. 88.8f, and -0 .. the float above -104
        for a in range(lo, hi, chunk):
            x = np.arange(a, min(a + chunk, hi), dtype=np.uint32).view(np.float32)
            assert_variants_match_oracle(eng, oracle_lib, x, f"bit patterns [{a:#x}, {min(a + chunk, hi):#x})")
    assert_variants_match_oracle(eng, oracle_lib, specials(np.float32), "NaN payloads, +-inf, +-0, +-max, +-min subnormal")


def test_float_exp_threshold_windows(eng, oracle_lib):
    """The windows the sweep covers, plus what it does not: arguments at and below -104, above 88.8f, and the specials."""
    rng = np.random.default_rng(11)
    x = np.concatenate([np.concatenate([around(t, 4096, np.float32) for t in thresholds(np.float32).values()]),
                        tie_windows(np.float32, 64), around(np.float32(-104.0), 4096, np.float32),
                        rng.uniform(-1e4, -104, 100000).astype(np.float32), rng.uniform(88.8, 1e4, 100000).astype(np.float32),
                        specials(np.float32)])
    assert_variants_match_oracle(eng, oracle_lib, x, "float windows")


# ---- double: targeted ------------------------------------------------------------------------------------------------

def double_arguments():
    rng = np.random.default_rng(20261021)
    return np.concatenate([
        rng.uniform(-746.0, 710.0, 6_000_000),
        rng.uniform(-1.0, 1.0, 2_000_000),
        log_uniform(rng, 6_000_000, -1074, 9.55, np.float64),                    # |x| from 2^-1074 to ~750
        np.concatenate([around(t, 4096, np.float64) for t in thresholds(np.float64).values()]),
        tie_windows(np.float64, 64),                                            # k in [-1075, 1024]: ~2.7e5 arguments
        rng.uniform(-1e6, 1e6, 100_000),
        specials(np.float64),
    ])


def test_double_exp_targeted_arguments(eng, oracle_lib):
    x = double_arguments()
    assert x.size > 14_000_000
    assert_variants_match_oracle(eng, oracle_lib, x, "double arguments")


@pytest.mark.parametrize("dt", [np.float64, np.float32], ids=["double", "float"])
def test_exp_short_inputs_and_tails(eng, oracle_lib, dt):
    """n not a multiple of K or of a warp's 32 K inputs: the padded lanes must not disturb the real ones."""
    rng = np.random.default_rng(5)
    for n in (1, 3, 17, 127, 129, 511, 513, 1000):
        lim = 700.0 if dt == np.float64 else 80.0
        assert_variants_match_oracle(eng, oracle_lib, rng.uniform(-1.5 * lim, 1.05 * lim, n).astype(dt), f"n = {n}")


# ---- the conv fast path against the general path -------------------------------------------------------------------

@pytest.mark.parametrize("variant", [5, 6], ids=["K4", "K16"])
@pytest.mark.parametrize("dt", [np.float64, np.float32], ids=["double", "float"])
def test_conv_fast_path_equals_general_path(eng, oracle_lib, dt, variant):
    K = CONV_K[variant]
    W = 32 * K                                              # inputs per warp
    lim = FAST_LIMIT[dt]
    rng = np.random.default_rng(variant)
    inner = np.concatenate([rng.uniform(-lim, lim, 400_000).astype(dt), rng.uniform(-1, 1, 50_000).astype(dt),
                            around(dt(lim), 8192, dt), around(dt(-lim), 8192, dt),
                            log_uniform(rng, 50_000, -1074 if dt == np.float64 else -149, 6, dt),
                            tie_windows(dt, 4)])
    inner = inner[np.abs(inner) < lim]
    nw = -(-inner.size // (W - 1))
    inner = np.concatenate([inner, np.zeros(nw * (W - 1) - inner.size, dtype=dt)])

    # layout A: every warp in range -> fast path
    ya = eng.math_hook(inner, variant)
    # layout B: the same arguments, W - 1 per warp, and one lane per warp out of range (750 or NaN) -> general path
    poison = np.zeros(nw * W, dtype=bool)
    poison[np.arange(nw) * W + rng.integers(0, W, nw)] = True
    xb = np.empty(nw * W, dtype=dt)
    xb[~poison] = inner
    xb[poison] = np.where(np.arange(nw) % 2 == 0, dt(750.0), dt(np.nan))
    yb = eng.math_hook(xb, variant)

    yo = oracle_exp(oracle_lib, inner)
    msg_a = mismatch(inner, ya, yo)
    msg_b = mismatch(inner, yb[~poison], ya)
    assert msg_a is None, f"{EXP_VARIANTS[variant]} fast path against the host: {msg_a}"
    assert msg_b is None, f"{EXP_VARIANTS[variant]} general path against the fast path: {msg_b}"
    assert mismatch(xb[poison], yb[poison], oracle_exp(oracle_lib, xb[poison])) is None

    # whole warps just past the switch (subnormal and overflowing results among them) must not take the fast path
    top = 709.9 if dt == np.float64 else 88.8
    bot = -745.3 if dt == np.float64 else -104.1
    xc = np.concatenate([rng.uniform(lim, top, 32 * W), rng.uniform(bot, -lim, 32 * W)]).astype(dt)
    xc = xc[np.abs(xc) >= lim]
    assert_variants_match_oracle(eng, oracle_lib, xc, "whole warps with |x| past the fast-path switch", variants=[variant])


# ---- mux_sqrt_rcp --------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("dt", [np.float64, np.float32], ids=["double", "float"])
def test_mux_sqrt_rcp_within_one_ulp(eng, dt):
    p, emin = fmt(dt)[:2]
    lo_exp, hi_exp = emin - p, (1024 if dt == np.float64 else 128)
    switch = two(-900 if dt == np.float64 else -100)
    rng = np.random.default_rng(3)
    a = np.concatenate([
        np.abs(log_uniform(rng, 20_000, lo_exp, hi_exp, dt)),                   # all positive finite magnitudes
        around(dt(switch), 256, dt),                                            # the tiny-pivot rescaling switch
        np.concatenate([around(dt(np.ldexp(1.0, e)), 1, dt) for e in range(lo_exp, hi_exp)]),   # 2^e and neighbours
    ])
    a = np.concatenate([a[np.isfinite(a) & (a > 0)], [np.finfo(dt).max, np.array([1], dtype=fmt(dt)[2]).view(dt)[0]]]).astype(dt)
    l, r = eng.math_hook(a, SQRT_RCP)
    # l against sqrt(a) and r against 1/l, the reciprocal of the returned pivot: the IEEE sequence this replaces (and
    # LAPACK's potf2) scales by 1 / the rounded sqrt, not by a rounded 1/sqrt(a).  Both within one ulp; against
    # 1/sqrt(a) itself that composes to below two (l's relative error is at most 2^-p-1, one ulp of r or less).
    names = ("sqrt(a)", "1/l", "1/sqrt(a)")
    worst = [(0.0, None)] * 3
    for ai, li, ri in zip(a, l, r):
        for k, e in enumerate(sqrt_rcp_errs(ai, li, ri, dt)):
            if e > worst[k][0]:
                worst[k] = (e, ai)
    desc = {names[k]: (e, float(x).hex() if x is not None else None) for k, (e, x) in enumerate(worst)}
    assert worst[0][0] < 1.0 and worst[1][0] < 1.0 and worst[2][0] < 2.0, f"worst ulp error and its argument: {desc}"


@pytest.mark.parametrize("dt", [np.float64, np.float32], ids=["double", "float"])
def test_mux_sqrt_rcp_invalid_pivots_run_without_fault(eng, dt):
    """a <= 0, NaN and inf give values nobody reads (the caller has recorded the breakdown); they must only not fault."""
    a = np.array([0.0, -0.0, -1.0, -np.finfo(dt).tiny, -np.finfo(dt).max, np.nan, np.inf, -np.inf], dtype=dt)
    l, r = eng.math_hook(a, SQRT_RCP)
    assert l.shape == r.shape == a.shape
    ok = np.array([4.0], dtype=dt)
    l, r = eng.math_hook(ok, SQRT_RCP)                      # the device is still usable
    assert l[0] == 2 and r[0] == dt(0.5)
