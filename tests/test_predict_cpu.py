"""CPU checks of the batched prediction: the host reference (tests/predict_util.py) agrees with the textbook form on a
linear model and with scipy's curve_fit pcov propagated through a numerical gradient, the entry points reject bad
arguments before touching a device, the built library carries the prediction kernels for sm_100a, and without a CUDA
device the entry points fail loudly (no CPU fallback)."""
import ctypes as C
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

from predict_util import predict_callbacks, predict_reference, se_within_bound

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SO = os.path.join(ROOT, "mir_optim_b200", "libmir_optim_b200.so")
CUOBJDUMP = shutil.which("cuobjdump") or ("/usr/local/cuda/bin/cuobjdump" if os.path.exists("/usr/local/cuda/bin/cuobjdump") else None)


def test_reference_equals_textbook_form_on_a_linear_model():
    rng = np.random.default_rng(4)
    n, k = 5, 40
    ts = np.linspace(-1.0, 2.0, k)
    Phi = np.vander(ts, n, increasing=True)
    A = rng.standard_normal((n, n)); Cm = A @ A.T + 0.1 * np.eye(n)
    f = lambda b, p: Phi @ p
    g = lambda b, p: Phi
    x = rng.standard_normal((1, n)); inf = np.full(n, np.inf)
    value, q, bound = predict_reference(f, g, x, -inf, inf, 2.0 ** -26, Cm[None], k)
    np.testing.assert_allclose(value[0], Phi @ x[0], rtol=1e-15, atol=0)
    np.testing.assert_allclose(np.sqrt(q[0]), np.sqrt(np.diag(Phi @ Cm @ Phi.T)), rtol=1e-13)
    # the upper triangle is not read
    Cu = Cm.copy(); Cu[np.triu_indices(n, 1)] = np.nan
    _, q2, _ = predict_reference(f, g, x, -inf, inf, 2.0 ** -26, Cu[None], k)
    assert np.array_equal(q2, q)
    # a fixed parameter drops out: its row and column are never read
    xl = x.copy(); l = -inf.copy(); l[2] = xl[0, 2]
    Cn = Cm.copy(); Cn[2, :] = np.nan; Cn[:, 2] = np.nan
    _, q3, _ = predict_reference(f, g, xl, l, inf, 2.0 ** -26, Cn[None], k)
    keep = [0, 1, 3, 4]
    np.testing.assert_allclose(q3[0], np.diag(Phi[:, keep] @ Cm[np.ix_(keep, keep)] @ Phi[:, keep].T), rtol=1e-13)
    ok, worst = se_within_bound(np.sqrt(np.diag(Phi @ Cm @ Phi.T))[None], q, bound, np.float64)
    assert ok, worst


def test_reference_matches_curve_fit_pcov_through_a_numerical_gradient(oracle_lib):
    from scipy.optimize import curve_fit
    from mir_optim_b200 import ModelId, workloads
    wl = workloads.c2_gauss4(4, noise=0.05, seed=11)

    def fm(t, A, mu, s, c):
        return A * np.exp(-0.5 * ((t - mu) / s) ** 2) + c

    ts = np.linspace(wl.t[0], wl.t[-1], 33)
    popt = np.empty((4, 4)); pcov = np.empty((4, 4, 4))
    for b in range(4):
        p0, _ = curve_fit(fm, wl.t, wl.y[b], p0=wl.truth[b])
        popt[b], pcov[b] = curve_fit(fm, wl.t, wl.y[b], p0=p0)
    f, g, k = predict_callbacks(oracle_lib, ModelId.GAUSS4, np.float64, ts, 4)
    inf = np.full(4, np.inf)
    value, q, _ = predict_reference(f, g, popt, -inf, inf, 2.0 ** -26, pcov, k)
    for b in range(4):
        np.testing.assert_allclose(value[b], fm(ts, *popt[b]), rtol=1e-13, atol=1e-13)
        h = 1e-6 * np.maximum(np.abs(popt[b]), 1.0)
        G = np.stack([(fm(ts, *(popt[b] + h[j] * np.eye(4)[j])) - fm(ts, *(popt[b] - h[j] * np.eye(4)[j]))) / (2 * h[j])
                      for j in range(4)], axis=1)
        np.testing.assert_allclose(np.sqrt(q[b]), np.sqrt(np.einsum("ia,ac,ic->i", G, pcov[b], G)), rtol=1e-6)


def _call(eng, sfx, model=6, batch=4, k=8, n=4, t=True, x=True, l=True, u=True, cov=True, value=True, se=True, aux=None,
          bound_stride=0, dev=False):
    dt = np.float64 if sfx == "d" else np.float32
    kk = min(max(k, 1), 64)                              # (the arrays are never read past what a rejected call could touch)
    ts = np.linspace(-1, 1, kk).astype(dt); xs = np.ones((batch, max(n, 1)), dt)
    lo = np.full(max(n, 1), -np.inf, dt); up = np.full(max(n, 1), np.inf, dt)
    cv = np.zeros((batch, max(n, 1), max(n, 1)), dt); out = np.zeros((batch, kk), dt); out2 = out.copy()
    from mir_optim_b200._abi import ModelDesc
    d = ModelDesc(int(model or 0), 0, C.c_void_p(ts.ctypes.data) if t else None, None,
                  None if aux is None else C.c_void_p(aux.ctypes.data), 0.0)
    p = lambda a, on: a.ctypes.data if on else None
    fn = getattr(eng.lib, f"mir_b200_predict_batched{'_dev' if dev else ''}_{sfx}")
    return fn(None, C.byref(d) if model is not None else None, batch, k, n, p(xs, x), p(lo, l), p(up, u), bound_stride,
              p(cv, cov), p(out, value), p(out2, se), None if dev else -1)


@pytest.mark.parametrize("sfx", ["d", "s"])
@pytest.mark.parametrize("dev", [False, True])
def test_argument_errors_before_any_device(sfx, dev):
    import mir_optim_b200
    from mir_optim_b200 import ModelId
    eng = mir_optim_b200.engine
    E, U = 2, 3                                                                      # MIR_B200_EINVAL, MIR_B200_EUNSUPPORTED
    c = lambda **kw: _call(eng, sfx, dev=dev, **kw)
    assert c(model=None) == E
    assert c(x=False) == E and c(l=False) == E and c(u=False) == E
    assert c(value=False, se=False) == E                                             # nothing to compute
    assert c(cov=False) == E                                                         # se without cov
    assert c(n=0) == E and c(k=0) == E
    assert c(t=False) == E                                                           # a data model without abscissae
    assert c(model=ModelId.SPLINE) == E                                              # no knots
    assert c(bound_stride=2) == E
    assert c(n=5) == E                                                               # Gauss4 has n = 4
    assert c(model=ModelId.GAUSSMIX, n=129) == U
    assert c(k=(1 << 31) - 1, batch=0) == U
    for mid in (ModelId.LINEAR2, ModelId.ROSENBROCK, ModelId.SQRTCIRCLE):
        assert c(model=mid, n=2) == U
    assert c(batch=0) == 0 or not dev                                                 # batch == 0 does nothing (device form)
    # the checks run before the device is looked for: these fail the same way with or without one
    assert c(model=ModelId.GAUSSMIX, n=129, x=False) == U                            # (the covariance's order: n before x)


def test_no_device_means_prediction_fails_loudly():
    import mir_optim_b200
    from mir_optim_b200 import workloads
    from mir_optim_b200.engine import B200Error
    eng = mir_optim_b200.engine
    if eng.device_count() > 0:
        pytest.skip("a CUDA device is present")
    wl = workloads.c2_gauss4(4)
    for dt in (np.float64, np.float32):
        with pytest.raises(B200Error) as ei:
            eng.predict_batched(None, wl.model, wl.x0.astype(dt), wl.l, wl.u, t=wl.t, cov=np.zeros((4, 4, 4)))
        assert ei.value.code == 1                                                     # MIR_B200_ENODEVICE
        assert "no usable CUDA device" in str(ei.value)
        assert _call(eng, "d" if dt == np.float64 else "s", dev=True) == 1
        assert _call(eng, "d" if dt == np.float64 else "s", batch=0) == 1             # the host form looks for the device


@pytest.mark.skipif(CUOBJDUMP is None or not os.path.exists(SO), reason="needs cuobjdump and the built library")
def test_library_contains_prediction_kernels_for_sm_100a():
    out = subprocess.run([CUOBJDUMP, "-res-usage", SO], capture_output=True, text=True, check=True).stdout
    blocks = re.findall(r"Function (\S*lm_pred_cta_kernel\S*):\s*\n\s*REG:(\d+) STACK:(\d+) SHARED:(\d+) LOCAL:(\d+)", out)
    dem = subprocess.run(["c++filt"] + [b[0] for b in blocks], capture_output=True, text=True, check=True).stdout
    # every model of visit_cta_model, both precisions, analytic and FD
    for model in ("LModelExpDecay2", "LModelExpTau3", "LModelExpDecay3", "LModelGauss4", "LModelSumExp", "LModelGaussMix", "CtaSpline"):
        assert dem.count(model) == 4, model
    assert len(blocks) == 28
    for name, reg, stack, shared, local in blocks:
        # no local arrays; the only stack is the call frame of the exactly rounded helpers (noinline, repro_math.cuh)
        assert int(local) == 0 and int(stack) <= 64, (name, stack, local)
    elf = subprocess.run([CUOBJDUMP, "-lelf", SO], capture_output=True, text=True, check=True).stdout
    assert set(re.findall(r"sm_(\d+a?)", elf)) == {"100a"}
