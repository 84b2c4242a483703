"""CPU checks of per-observation weights (MIR_MODEL_WEIGHTED): the weighted host reference (tests/weights_util.py) against
scipy, the ABI of the grown mir_model_desc, the argument errors (raised before any device is touched), the
no-device error, and the weighted kernels of the built library (sm_100a only)."""
import ctypes as C
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

from weights_util import oracle_batched_weighted, sigma_weights

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SO = os.path.join(ROOT, "mir_optim_b200", "libmir_optim_b200.so")
CUOBJDUMP = shutil.which("cuobjdump") or ("/usr/local/cuda/bin/cuobjdump" if os.path.exists("/usr/local/cuda/bin/cuobjdump") else None)


def gauss4(t, p):
    z = (t - p[1]) / p[2]
    e = np.exp(-0.5 * z * z)
    return p[0] * e + p[3], np.stack([e, p[0] * e * z / p[2], p[0] * e * z * z / p[2], np.ones_like(t)], axis=1)


@pytest.mark.parametrize("fd", [False, True])
def test_weighted_oracle_fit_matches_scipy_least_squares(oracle_lib, fd):
    """The weighted reference, run to convergence, lands where scipy's least_squares on w (.) r does."""
    from scipy.optimize import least_squares
    from mir_optim_b200 import ModelId, api, workloads
    B = 6
    wl = workloads.c2_gauss4(B, noise=0.05, seed=8)
    w = sigma_weights(B, wl.m, seed=2, zero_rows=4)
    s = api.ReferenceAPI(oracle_lib).settings(np.float64)
    x, res = oracle_batched_weighted(oracle_lib, s, ModelId.GAUSS4, wl.x0, wl.l, wl.u, t=wl.t, y=wl.y, w=w, fd_jacobian=fd)
    assert np.all(res["status"] >= 0), res["status"]
    for b in range(B):
        ref = least_squares(lambda p: w[b] * (gauss4(wl.t, p)[0] - wl.y[b]), wl.x0[b], jac=lambda p: w[b][:, None] * gauss4(wl.t, p)[1],
                            bounds=(wl.l, wl.u), xtol=1e-15, ftol=1e-15, gtol=1e-15)
        assert np.max(np.abs(x[b] - ref.x) / np.maximum(np.abs(ref.x), 1e-3)) < (1e-7 if not fd else 1e-6), (b, x[b], ref.x)
        assert abs(res["residual"][b] - 2 * ref.cost) <= 1e-9 * 2 * ref.cost


def test_model_desc_abi():
    from mir_optim_b200 import _abi
    assert C.sizeof(_abi.ModelDesc) == 48 and _abi.ModelDesc.w.offset == 40 and _abi.ModelDesc.param.offset == 32
    assert _abi.MODEL_WEIGHTED == 32
    hdr = open(os.path.join(ROOT, "include", "mir_optim_b200.h")).read()
    assert re.search(r"MIR_MODEL_WEIGHTED\s*=\s*32u", hdr)
    assert re.search(r"double\s+param;[^\n]*\n\s*const void\* w;", hdr)
    d = open(os.path.join(ROOT, "d", "mir", "optim", "b200.d")).read()
    assert "enum uint mirModelWeighted = 32;" in d and re.search(r"double param = 0;[^\n]*\n\s*const\(void\)\* w;", d)


def _desc(model, flags, t, y, w):
    from mir_optim_b200 import _abi
    vp = lambda a: None if a is None else C.c_void_p(a.ctypes.data)      # noqa: E731
    return _abi.ModelDesc(int(model), flags, vp(t), vp(y), None, 0.0, vp(w))


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_argument_errors(dtype):
    """Checked before the device is touched: NULL w with the flag (EINVAL), the flag on a data-free model (EUNSUPPORTED), the
    sharded entry (EUNSUPPORTED) and the legacy entry in device-model mode (numericError and a message)."""
    import mir_optim_b200
    from mir_optim_b200 import ModelId, _abi
    eng = mir_optim_b200.engine
    sfx = "d" if dtype == np.float64 else "s"
    S = _abi.LeastSquaresSettingsD if dtype == np.float64 else _abi.LeastSquaresSettingsS
    st = eng.settings(dtype)
    B, m, n = 3, 16, 4
    t = np.linspace(-1, 1, m).astype(dtype); y = np.zeros((B, m), dtype); w = np.ones((B, m), dtype)
    x = np.ones((B, n), dtype); l = np.full(n, -np.inf, dtype); u = np.full(n, np.inf, dtype)
    res = np.zeros(B * 32, np.uint8); info = np.zeros(B, np.int32); sd = np.zeros((B, n), dtype)
    W = _abi.MODEL_WEIGHTED
    assert isinstance(st, S)

    def fit(desc, dev=False, nn=n):
        fn = getattr(eng.lib, f"mir_optimize_least_squares_batched_{'dev_' if dev else ''}{sfx}")
        return fn(C.byref(st), C.byref(desc), B, m, nn, x.ctypes.data, l.ctypes.data, u.ctypes.data, 0, res.ctypes.data, None,
                  None if dev else -1)

    def cov(desc, dev=False, nn=n):
        fn = getattr(eng.lib, f"mir_b200_covariance_batched_{'dev_' if dev else ''}{sfx}")
        return fn(None, C.byref(desc), B, m, nn, x.ctypes.data, l.ctypes.data, u.ctypes.data, 0, 0, None, sd.ctypes.data,
                  info.ctypes.data, None if dev else -1)

    for dev in (False, True):
        assert fit(_desc(ModelId.GAUSS4, W, t, y, None), dev) == 2
        assert b"model->w must not be NULL" in eng.lib.mir_b200_last_error()
        assert cov(_desc(ModelId.GAUSS4, W, t, y, None), dev) == 2
        for model in (ModelId.LINEAR2, ModelId.ROSENBROCK, ModelId.SQRTCIRCLE):
            assert fit(_desc(model, W, None, None, np.ones((B, 2), dtype)), dev, 2) == 3
            assert b"MIR_MODEL_WEIGHTED" in eng.lib.mir_b200_last_error()
            assert cov(_desc(model, W, None, None, np.ones((B, 2), dtype)), dev, 2) == 3
    if dtype == np.float64:
        xs = np.ones(n)
        rc = eng.lib.mir_optimize_least_squares_sharded_d(C.byref(st), C.byref(_desc(ModelId.GAUSS4, W, t, y, w)), m, n, xs.ctypes.data,
                                                          l.ctypes.data, u.ctypes.data, None, None, C.byref(_abi.LeastSquaresResultD()), None)
        assert rc == 3 and b"MIR_MODEL_WEIGHTED" in eng.lib.mir_b200_last_error()
    # the reference's own entry point with the device-model sentinel: a weighted desc is refused, not run unweighted
    from mir_optim_b200.api import _types
    _, real, _, _, Sl, _, _ = _types(dtype)
    desc = _desc(ModelId.GAUSS4, W, t, y[0], w[0])
    for fd in (False, True):
        g_ptr = None if fd else C.cast(getattr(eng.lib, f"mir_b200_device_model_jac_{sfx}"), C.c_void_p)
        xs = x[0].copy()
        r = getattr(eng.lib, f"mir_optimize_least_squares_{sfx}")(
            C.byref(st), m, n, xs.ctypes.data_as(C.POINTER(real)), l.ctypes.data_as(C.POINTER(real)), u.ctypes.data_as(C.POINTER(real)),
            Sl(0, None), _abi.SliceI(0, None), C.cast(C.pointer(desc), C.c_void_p),
            C.cast(getattr(eng.lib, f"mir_b200_device_model_{sfx}"), C.c_void_p), None, g_ptr, None, None)
        assert r.status == _abi.LeastSquaresStatus.numericError and r.fCalls == 0 and np.all(xs == 1)
        assert b"supported by the batched and covariance entry points" in eng.lib.mir_b200_last_error()


def test_no_device_means_weighted_entries_fail_loudly():
    import mir_optim_b200
    from mir_optim_b200 import workloads
    from mir_optim_b200.engine import B200Error
    eng = mir_optim_b200.engine
    if eng.device_count() > 0:
        pytest.skip("a CUDA device is present")
    wl = workloads.c2_gauss4(4)
    w = sigma_weights(4, wl.m, seed=3)
    for dt in (np.float64, np.float32):
        with pytest.raises(B200Error) as ei:
            eng.optimize_batched(eng.settings(dt), wl.model, wl.x0.astype(dt), wl.l, wl.u, t=wl.t, y=wl.y, w=w)
        assert ei.value.code == 1                                                     # MIR_B200_ENODEVICE
        with pytest.raises(B200Error) as ei:
            eng.covariance_batched(None, wl.model, wl.x0.astype(dt), wl.l, wl.u, t=wl.t, y=wl.y, w=w)
        assert ei.value.code == 1


@pytest.mark.skipif(CUOBJDUMP is None or not os.path.exists(SO), reason="needs cuobjdump and the built library")
def test_library_contains_weighted_kernels_for_sm_100a():
    out = subprocess.run([CUOBJDUMP, "-res-usage", SO], capture_output=True, text=True, check=True).stdout
    mangled = re.findall(r"Function (\S+):", out)
    dem = subprocess.run(["c++filt"] + mangled, capture_output=True, text=True, check=True).stdout.splitlines()
    fit = [d for d in dem if "lm_cta_kernel<mirb200::CtaWeighted<" in d]
    cov = [d for d in dem if "lm_cov_cta_weighted_kernel<mirb200::CtaWeighted<" in d]
    # every built-in model of the general kernel, both precisions, analytic and FD
    for model in ("LModelExpDecay2", "LModelExpTau3", "LModelExpDecay3", "LModelGauss4", "LModelSumExp", "LModelGaussMix", "CtaSpline"):
        assert sum(model in d for d in fit) == 4, model
        assert sum(model in d for d in cov) == 4, model
    assert len(fit) == 28 and len(cov) == 28
    elf = subprocess.run([CUOBJDUMP, "-lelf", SO], capture_output=True, text=True, check=True).stdout
    assert set(re.findall(r"sm_(\d+a?)", elf)) == {"100a"}
