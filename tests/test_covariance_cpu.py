"""CPU checks of the batched covariance: the host reference (tests/cov_util.py) agrees with scipy's curve_fit pcov and with
LAPACK's ?potrf / ?potri, the built library carries the covariance kernels for sm_100a, and without a CUDA device the
covariance entry points fail loudly (no CPU fallback)."""
import ctypes as C
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

from cov_util import cov_one, cov_reference, oracle_callbacks

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SO = os.path.join(ROOT, "mir_optim_b200", "libmir_optim_b200.so")
CUOBJDUMP = shutil.which("cuobjdump") or ("/usr/local/cuda/bin/cuobjdump" if os.path.exists("/usr/local/cuda/bin/cuobjdump") else None)


def test_reference_matches_curve_fit_pcov(oracle_lib):
    from scipy.optimize import curve_fit
    from mir_optim_b200 import ModelId, workloads
    wl = workloads.c2_gauss4(4, noise=0.05, seed=11)

    def f(t, A, mu, s, c):
        return A * np.exp(-0.5 * ((t - mu) / s) ** 2) + c

    def jac(t, A, mu, s, c):
        z = (t - mu) / s; e = np.exp(-0.5 * z * z)
        return np.stack([e, A * e * z / s, A * e * z * z / s, np.ones_like(t)], axis=1)

    for b in range(4):
        p0, _ = curve_fit(f, wl.t, wl.y[b], p0=wl.truth[b], jac=jac)
        popt, pcov = curve_fit(f, wl.t, wl.y[b], p0=p0, jac=jac)                    # started at the optimum, unbounded
        fo, go = oracle_callbacks(oracle_lib, ModelId.GAUSS4, np.float64, wl.t, wl.y[b:b + 1])
        cov, info, _ = cov_reference(fo, go, popt[None, :], np.full(4, -np.inf), np.full(4, np.inf), 2.0 ** -26)
        assert info[0] == 0
        np.testing.assert_allclose(cov[0], pcov, rtol=1e-6, atol=1e-6 * np.sqrt(np.outer(np.diag(pcov), np.diag(pcov))).max())


def test_reference_matches_lapack_potrf_potri():
    from scipy.linalg import lapack
    rng = np.random.default_rng(7)
    for n, m in ((2, 5), (4, 64), (8, 128), (11, 40), (30, 200)):
        J = rng.standard_normal((m, n)) * np.logspace(0, 3, n)[None, :]
        r = rng.standard_normal(m)
        cov, info, kappa = cov_one(r, J, np.ones(n, dtype=bool), m)
        assert info == 0
        A = J.T @ J
        c, i1 = lapack.dpotrf(A, lower=1)
        inv, i2 = lapack.dpotri(c, lower=1)
        assert i1 == 0 and i2 == 0
        inv = np.tril(inv) + np.tril(inv, -1).T
        ref = inv * (r @ r) / (m - n)
        d = np.sqrt(np.outer(np.diag(ref), np.diag(ref)))
        assert np.max(np.abs(cov - ref) / d) < 1e-12, (n, m)


def test_reference_info_codes():
    J = np.array([[1.0, 0.0, 1.0], [2.0, 0.0, 1.0], [3.0, 0.0, 1.0], [4.0, 0.0, 1.0]])
    r = np.ones(4)
    cov, info, _ = cov_one(r, J, np.ones(3, dtype=bool), 4)
    assert info == 2 and np.all(np.isnan(cov))                                       # zero column of parameter 1
    cov, info, _ = cov_one(r, J[:3], np.array([True, False, True]), 3)
    assert info == 0 and np.all(cov[1] == 0) and np.all(cov[:, 1] == 0)
    cov, info, _ = cov_one(r[:2], J[:2], np.ones(3, dtype=bool), 2)
    assert info == -1 and np.all(np.isinf(cov))


@pytest.mark.skipif(CUOBJDUMP is None or not os.path.exists(SO), reason="needs cuobjdump and the built library")
def test_library_contains_covariance_kernels_for_sm_100a():
    out = subprocess.run([CUOBJDUMP, "-res-usage", SO], capture_output=True, text=True, check=True).stdout
    blocks = re.findall(r"Function (\S*lm_cov_cta_kernel\S*):\s*\n\s*REG:(\d+) STACK:(\d+) SHARED:(\d+) LOCAL:(\d+)", out)
    dem = subprocess.run(["c++filt"] + [b[0] for b in blocks], capture_output=True, text=True, check=True).stdout
    # the general kernel for every built-in model with a run-time-n functor, both precisions, analytic and FD
    for model in ("LModelExpDecay2", "LModelExpTau3", "LModelExpDecay3", "LModelGauss4", "LModelSumExp", "LModelGaussMix", "CtaSpline"):
        assert dem.count(model) == 4, model
    for name, reg, stack, shared, local in blocks:
        # no local arrays; the only stack is the call frame of the exactly rounded helpers (noinline, repro_math.cuh)
        assert int(local) == 0 and int(stack) <= 32, (name, stack, local)
    elf = subprocess.run([CUOBJDUMP, "-lelf", SO], capture_output=True, text=True, check=True).stdout
    assert set(re.findall(r"sm_(\d+a?)", elf)) == {"100a"}


def test_no_device_means_covariance_fails_loudly():
    import mir_optim_b200
    from mir_optim_b200 import workloads
    from mir_optim_b200.engine import B200Error
    eng = mir_optim_b200.engine
    if eng.device_count() > 0:
        pytest.skip("a CUDA device is present")
    wl = workloads.c2_gauss4(4)
    for dt in (np.float64, np.float32):
        with pytest.raises(B200Error) as ei:
            eng.covariance_batched(None, wl.model, wl.x0.astype(dt), wl.l, wl.u, t=wl.t, y=wl.y)
        assert ei.value.code == 1                                                     # MIR_B200_ENODEVICE
        assert "no usable CUDA device" in str(ei.value)
        desc = mir_optim_b200._abi.ModelDesc(int(wl.model), 0, C.c_void_p(wl.t.ctypes.data), C.c_void_p(wl.y.ctypes.data))
        sfx = "d" if dt == np.float64 else "s"
        x = wl.x0.astype(dt); info = np.zeros(4, np.int32); sd = np.zeros((4, 4), dt)
        rc = getattr(eng.lib, f"mir_b200_covariance_batched_dev_{sfx}")(None, C.byref(desc), 4, 64, 4, x.ctypes.data, wl.l.astype(dt).ctypes.data,
                                                                       wl.u.astype(dt).ctypes.data, 0, 0, None, sd.ctypes.data,
                                                                       info.ctypes.data, None)
        assert rc == 1
