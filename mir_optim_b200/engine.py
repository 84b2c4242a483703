"""Batched / device-resident entry points (header part 2) with numpy and torch front ends.

numpy arrays are HOST buffers: the library stages them to the GPU and back (the end-to-end
path).  torch CUDA tensors are passed as device pointers to the ``*_dev`` entry points and are
enqueued on torch's current stream (the resident path).  torch is plumbing only.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _abi
from ._abi import BatchStats, ModelDesc, ModelId, MODEL_FD_JACOBIAN, MODEL_GRID_PER_PROBLEM, MODEL_NO_TAIL_SHORTCUT
from .api import ReferenceAPI, _types

RESULT_DTYPES = {
    np.dtype(np.float64): np.dtype([("status", "<i4"), ("iterations", "<u4"), ("fCalls", "<u4"), ("gCalls", "<u4"),
                                    ("residual", "<f8"), ("lambda", "<f8")]),
    np.dtype(np.float32): np.dtype([("status", "<i4"), ("iterations", "<u4"), ("fCalls", "<u4"), ("gCalls", "<u4"),
                                    ("residual", "<f4"), ("lambda", "<f4")]),
}
assert RESULT_DTYPES[np.dtype(np.float64)].itemsize == 32 and RESULT_DTYPES[np.dtype(np.float32)].itemsize == 24


class B200Error(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"mir_optim_b200 error {code}: {message}")
        self.code = code


def _vp(a):
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        return C.c_void_p(a.ctypes.data)
    return C.c_void_p(a.data_ptr())      # torch tensor


def _model_desc(model, x, t, y, m, aux, param, fd_jacobian, w=None):
    """(m, ModelDesc) of a batched call on x (batch, n): the model id and constants (aux, param), its samples t and y (or m
    for a model without samples), the observation weights w (batch, m) if given, and the flags they imply.  numpy inputs
    are converted to x's dtype, and the desc holds the converted arrays; torch tensors are passed as they are."""
    if isinstance(x, np.ndarray):
        t, y, aux, w = (None if a is None else np.ascontiguousarray(a, dtype=x.dtype) for a in (t, y, aux, w))
        assert y is None or y.shape[0] == x.shape[0]
    if y is not None and m is None:
        m = y.shape[1]
    assert m is not None, "m is required for models without samples"
    if w is not None:
        assert tuple(w.shape) == ((x.shape[0], m) if y is None else tuple(y.shape)), "w must have the shape (batch, m) of y"
    flags = ((MODEL_FD_JACOBIAN if fd_jacobian else 0) | (MODEL_GRID_PER_PROBLEM if t is not None and t.ndim == 2 else 0)
             | (_abi.MODEL_AUX_PER_PROBLEM if aux is not None and aux.ndim == 2 else 0) | (_abi.MODEL_WEIGHTED if w is not None else 0))
    desc = ModelDesc(int(model), flags, _vp(t), _vp(y), _vp(aux), float(param), _vp(w))
    desc.arrays = (t, y, aux, w)
    return m, desc


class Engine(ReferenceAPI):
    def __init__(self, lib):
        super().__init__(lib)
        _abi.bind_b200_abi(lib)

    # -- helpers ----------------------------------------------------------------------
    def _check(self, rc: int):
        if rc != 0:
            raise B200Error(rc, self.lib.mir_b200_last_error().decode())

    def device_count(self) -> int:
        return self.lib.mir_b200_device_count()

    def kernel_launches(self) -> int:
        return int(self.lib.mir_b200_kernel_launches())

    # -- batched LM, host buffers -------------------------------------------------------
    def optimize_batched(self, settings, model: ModelId, x: np.ndarray, l: np.ndarray, u: np.ndarray,
                         t: np.ndarray | None = None, y: np.ndarray | None = None, m: int | None = None,
                         fd_jacobian: bool = False, want_stats: bool = False, device: int = -1, tail_shortcut: bool = True,
                         results: np.ndarray | None = None, aux: np.ndarray | None = None, param: float = 0.0,
                         warm_start: bool = False, w: np.ndarray | None = None):
        """Solve ``batch`` independent problems; x (batch, n) is updated in place.
        l/u: shape (n,) shared, or (batch, n).  Returns (results structured array, stats dict | None).
        results: optional preallocated structured array (e.g. a view of pinned memory) to receive the Result PODs.
        w: optional observation weights (batch, m): row i's residual and Jacobian row are scaled by w_i (1/sigma_i for
        a chi^2 fit; 0 removes the row)."""
        sfx, real, S, R, *_ = _types(x.dtype)
        assert isinstance(settings, S)
        assert x.ndim == 2 and x.flags.c_contiguous
        batch, n = x.shape
        l = np.ascontiguousarray(l, dtype=x.dtype); u = np.ascontiguousarray(u, dtype=x.dtype)
        bound_stride = 0 if l.ndim == 1 else n
        m, desc = _model_desc(model, x, t, y, m, aux, param, fd_jacobian, w)
        desc.flags |= 0 if tail_shortcut else MODEL_NO_TAIL_SHORTCUT
        if warm_start:
            assert results is not None, "warm_start reads results['lambda'] of a previous call"
            desc.flags |= _abi.MODEL_WARM_START
        if results is None:
            results = np.empty(batch, dtype=RESULT_DTYPES[x.dtype])
        assert results.dtype == RESULT_DTYPES[x.dtype] and results.shape == (batch,) and results.flags.c_contiguous
        stats = BatchStats() if want_stats else None
        fn = getattr(self.lib, f"mir_optimize_least_squares_batched_{sfx}")
        rc = fn(C.byref(settings), C.byref(desc), batch, m, n, _vp(x), _vp(l), _vp(u), bound_stride,
                _vp(results), C.cast(C.pointer(stats), C.c_void_p) if stats is not None else None, device)
        self._check(rc)
        return results, (stats.as_dict() if stats is not None else None)

    # -- batched LM, device-resident torch tensors ----------------------------------------
    def optimize_batched_device(self, settings, model: ModelId, x, l, u, t=None, y=None, m: int | None = None,
                                fd_jacobian: bool = False, results=None, stats=None, stream=None, tail_shortcut: bool = True,
                                aux=None, param: float = 0.0, warm_start: bool = False, w=None):
        """All tensors are CUDA tensors on the current device; asynchronous on `stream` (default:
        torch's current stream).  `results` : uint8 tensor (batch * sizeof(Result)); `stats`: int64[8] tensor.
        aux: (n,) shared or (batch, n) model constants (the knots of ModelId.SPLINE); param: the model constant;
        warm_start: results holds a previous call's Result PODs and their lambda is the initial damping;
        w: observation weights (batch, m), as in :meth:`optimize_batched`."""
        import torch
        dt = np.dtype({torch.float64: np.float64, torch.float32: np.float32}[x.dtype])
        sfx, real, S, R, *_ = _types(dt)
        assert isinstance(settings, S) and x.is_cuda and x.is_contiguous()
        batch, n = x.shape
        bound_stride = 0 if l.dim() == 1 else n
        m, desc = _model_desc(model, x, t, y, m, aux, param, fd_jacobian, w)
        desc.flags |= 0 if tail_shortcut else MODEL_NO_TAIL_SHORTCUT
        if warm_start:
            assert results is not None, "warm_start reads the lambda of a previous call's results"
            desc.flags |= _abi.MODEL_WARM_START
        if results is None:
            results = torch.empty(batch * RESULT_DTYPES[dt].itemsize, dtype=torch.uint8, device=x.device)
        if stream is None:
            stream = torch.cuda.current_stream(x.device).cuda_stream
        fn = getattr(self.lib, f"mir_optimize_least_squares_batched_dev_{sfx}")
        rc = fn(C.byref(settings), C.byref(desc), batch, m, n, _vp(x), _vp(l), _vp(u), bound_stride,
                _vp(results), _vp(stats), C.c_void_p(stream))
        self._check(rc)
        return results

    # -- parameter covariance at a given point -------------------------------------------------
    def covariance_batched(self, settings, model: ModelId, x: np.ndarray, l: np.ndarray, u: np.ndarray,
                           t: np.ndarray | None = None, y: np.ndarray | None = None, m: int | None = None,
                           fd_jacobian: bool = False, aux: np.ndarray | None = None, param: float = 0.0,
                           scaled: bool = True, want_cov: bool = True, device: int = -1, w: np.ndarray | None = None):
        """Covariance and standard errors of the parameters x (batch, n) -- normally a fit's output -- with the model data
        of :meth:`optimize_batched`, weights w included.  settings may be None (only jacobianEpsilon is read).
        scaled=False: s^2 = 1; with w = 1/sigma that is scipy's absolute_sigma=True, and scaled=True (s^2 from the weighted
        residuals over the rows with w != 0) is absolute_sigma=False.  Returns (cov (batch, n, n) or None,
        stddev (batch, n), info int32[batch]); info: 0 OK, k > 0 breakdown at parameter k-1, -1 m <= number of free
        parameters, -2 non-finite values (see mir_b200_covariance_batched_d in the header)."""
        x = np.ascontiguousarray(x)
        sfx, real, S, R, *_ = _types(x.dtype)
        assert settings is None or isinstance(settings, S)
        assert x.ndim == 2
        batch, n = x.shape
        l = np.ascontiguousarray(l, dtype=x.dtype); u = np.ascontiguousarray(u, dtype=x.dtype)
        bound_stride = 0 if l.ndim == 1 else n
        m, desc = _model_desc(model, x, t, y, m, aux, param, fd_jacobian, w)
        cov = np.empty((batch, n, n), dtype=x.dtype) if want_cov else None
        stddev = np.empty((batch, n), dtype=x.dtype)
        info = np.empty(batch, dtype=np.int32)
        fn = getattr(self.lib, f"mir_b200_covariance_batched_{sfx}")
        rc = fn(C.byref(settings) if settings is not None else None, C.byref(desc), batch, m, n, _vp(x), _vp(l), _vp(u),
                bound_stride, 0 if scaled else _abi.COV_UNSCALED, _vp(cov), _vp(stddev), _vp(info), device)
        self._check(rc)
        return cov, stddev, info

    def covariance_batched_device(self, settings, model: ModelId, x, l, u, t=None, y=None, m: int | None = None,
                                  fd_jacobian: bool = False, aux=None, param: float = 0.0, scaled: bool = True,
                                  want_cov: bool = True, cov=None, stddev=None, info=None, stream=None, w=None):
        """:meth:`covariance_batched` on CUDA tensors of the current device, asynchronous on `stream` (default: torch's
        current stream).  cov / stddev / info may be preallocated.  Returns (cov or None, stddev, info) tensors."""
        import torch
        dt = np.dtype({torch.float64: np.float64, torch.float32: np.float32}[x.dtype])
        sfx, real, S, R, *_ = _types(dt)
        assert (settings is None or isinstance(settings, S)) and x.is_cuda and x.is_contiguous()
        batch, n = x.shape
        bound_stride = 0 if l.dim() == 1 else n
        m, desc = _model_desc(model, x, t, y, m, aux, param, fd_jacobian, w)
        if cov is None and want_cov:
            cov = torch.empty((batch, n, n), dtype=x.dtype, device=x.device)
        if stddev is None:
            stddev = torch.empty((batch, n), dtype=x.dtype, device=x.device)
        if info is None:
            info = torch.empty(batch, dtype=torch.int32, device=x.device)
        if stream is None:
            stream = torch.cuda.current_stream(x.device).cuda_stream
        fn = getattr(self.lib, f"mir_b200_covariance_batched_dev_{sfx}")
        rc = fn(C.byref(settings) if settings is not None else None, C.byref(desc), batch, m, n, _vp(x), _vp(l), _vp(u),
                bound_stride, 0 if scaled else _abi.COV_UNSCALED, _vp(cov), _vp(stddev), _vp(info), C.c_void_p(stream))
        self._check(rc)
        return cov, stddev, info

    # -- user-defined device models (NVRTC) ---------------------------------------------------
    def compile_model(self, cuda_source: str) -> int:
        """Registers a residual model written in CUDA C++ (``template <class REAL> struct UserModel {...}``, see
        include/mir_optim_b200.h) and returns its model id, usable wherever a ModelId is.  Raises B200Error with the NVRTC
        log if the source does not compile."""
        mid = C.c_uint32()
        self._check(self.lib.mir_b200_model_compile(cuda_source.encode(), C.byref(mid)))
        return int(mid.value)

    def release_model(self, model_id: int):
        self._check(self.lib.mir_b200_model_release(int(model_id)))

    # -- fitSpline (fit_splie.d:26-85) ------------------------------------------------------
    def fit_spline(self, settings, points: np.ndarray, x: np.ndarray, l: np.ndarray, u: np.ndarray, lam: float = 0.0):
        """The reference's ``fitSpline(settings, points, x, l, u, lambda)``: points (P, 2) = [x_i, y_i], x = knots.
        Returns (values at the knots, LeastSquaresResult); raises ValueError with the reference's message where it throws
        (points.length < x.length with lambda == 0, fit_splie.d:45-49)."""
        points = np.ascontiguousarray(points)
        v, r = self.fit_spline_batched(settings, points[:, 0], points[None, :, 1], x, l, u, lam)
        return v[0], r[0]

    def fit_spline_batched(self, settings, points_x: np.ndarray, points_y: np.ndarray, x: np.ndarray, l: np.ndarray, u: np.ndarray,
                           lam: float = 0.0, device: int = -1, tail_shortcut: bool = True):
        """Many curves at once: points_y (batch, P); points_x (P,) shared or (batch, P); knots x (n,) shared or (batch, n);
        bounds l / u (n,).  Returns (values (batch, n), results structured array)."""
        dt = np.dtype(points_y.dtype)
        sfx, real, S, R, *_ = _types(dt)
        assert isinstance(settings, S)
        points_y = np.ascontiguousarray(points_y); batch, P = points_y.shape
        points_x = np.ascontiguousarray(points_x, dtype=dt); x = np.ascontiguousarray(x, dtype=dt)
        l = np.ascontiguousarray(l, dtype=dt); u = np.ascontiguousarray(u, dtype=dt)
        n = x.shape[-1]
        flags = (MODEL_GRID_PER_PROBLEM if points_x.ndim == 2 else 0) | (_abi.MODEL_AUX_PER_PROBLEM if x.ndim == 2 else 0)
        flags |= 0 if tail_shortcut else MODEL_NO_TAIL_SHORTCUT
        values = np.empty((batch, n), dtype=dt)
        results = np.empty(batch, dtype=RESULT_DTYPES[dt])
        rc = getattr(self.lib, f"mir_fit_spline_batched_{sfx}")(C.byref(settings), batch, P, _vp(points_x), _vp(points_y), n, _vp(x), _vp(l), _vp(u),
                                                                 real(lam), flags, _vp(values), _vp(results), device)
        if rc == 2 and b"fitSpline:" in self.lib.mir_b200_last_error():
            raise ValueError(self.lib.mir_b200_last_error().decode())
        self._check(rc)
        return values, results

    # -- solveBoxQP (boxcqp.d:85-102) -----------------------------------------------------
    def solve_box_qp(self, P: np.ndarray, q: np.ndarray, l: np.ndarray, u: np.ndarray, x: np.ndarray, settings=None):
        """argmin 1/2 x'Px + q'x, l <= x <= u.  Only the lower triangle of P (row-major) is read.  Returns BoxQPStatus."""
        sfx = _types(P.dtype)[0]
        n = q.shape[0]
        assert P.shape == (n, n) and P.flags.c_contiguous
        st = getattr(self.lib, f"mir_solve_box_qp_{sfx}")(C.byref(settings) if settings is not None else None, n,
                                                          _vp(P), _vp(q), _vp(l), _vp(u), _vp(x))
        if st < 0:
            self._check(-st)
        return _abi.BoxQPStatus(st)

    def solve_box_qp_batched(self, P: np.ndarray, q: np.ndarray, l: np.ndarray, u: np.ndarray, settings=None, device: int = -1):
        """P (batch, n, n), q/l/u (batch, n) host arrays.  Returns (x, status int32[batch], iterations uint32[batch])."""
        sfx = _types(P.dtype)[0]
        batch, n = q.shape
        assert P.shape == (batch, n, n) and P.flags.c_contiguous and q.flags.c_contiguous
        l = np.ascontiguousarray(l, dtype=P.dtype); u = np.ascontiguousarray(u, dtype=P.dtype)
        x = np.zeros((batch, n), dtype=P.dtype)
        status = np.full(batch, -1, dtype=np.int32); iters = np.zeros(batch, dtype=np.uint32)
        rc = getattr(self.lib, f"mir_solve_box_qp_batched_{sfx}")(C.byref(settings) if settings is not None else None, batch, n,
                                                                  _vp(P), _vp(q), _vp(l), _vp(u), _vp(x), _vp(status), _vp(iters), device)
        self._check(rc)
        return x, status, iters

    def solve_box_qp_batched_device(self, P, q, l, u, x, status, iterations=None, settings=None, stream=None):
        """torch CUDA tensors; asynchronous on torch's current stream."""
        import torch
        dt = np.dtype({torch.float64: np.float64, torch.float32: np.float32}[P.dtype])
        sfx = _types(dt)[0]
        batch, n = q.shape
        if stream is None:
            stream = torch.cuda.current_stream(P.device).cuda_stream
        rc = getattr(self.lib, f"mir_solve_box_qp_batched_dev_{sfx}")(C.byref(settings) if settings is not None else None, batch, n,
                                                                      _vp(P), _vp(q), _vp(l), _vp(u), _vp(x), _vp(status),
                                                                      _vp(iterations), C.c_void_p(stream))
        self._check(rc)

    def posvx_batched(self, A: np.ndarray, b: np.ndarray, variant: int, device: int = -1):
        """Diagnostics: the device restatement of LAPACK ?posvx('E','L') alone.  A (batch, n, n) row-major (lower triangle
        read), b (batch, n).  Returns (x, info int32[batch], equed int32[batch]).  variant: see the header."""
        sfx = _types(A.dtype)[0]
        batch, n = b.shape
        assert A.shape == (batch, n, n) and A.flags.c_contiguous and b.flags.c_contiguous and b.dtype == A.dtype
        x = np.zeros((batch, n), dtype=A.dtype)
        info = np.full(batch, -1, dtype=np.int32); equed = np.full(batch, -1, dtype=np.int32)
        self._check(getattr(self.lib, f"mir_b200_posvx_batched_{sfx}")(variant, batch, n, _vp(A), _vp(b), _vp(x), _vp(info), _vp(equed), device))
        return x, info, equed

    def math_hook(self, x: np.ndarray, variant: int, device: int = -1):
        """Diagnostics: one device form of the reproducible exp (variants 0-6) or the mux Cholesky pivot step (variant 7)
        applied elementwise to x (1-d, float64 or float32).  Returns y, or (sqrt(x), 1/sqrt(x)) for variant 7.  The
        variants are listed in the header."""
        sfx = _types(x.dtype)[0]
        x = np.ascontiguousarray(x)
        assert x.ndim == 1
        y = np.empty_like(x)
        y2 = np.empty_like(x) if variant == 7 else None
        self._check(getattr(self.lib, f"mir_b200_math_hook_{sfx}")(variant, x.size, _vp(x), _vp(y), _vp(y2), device))
        return (y, y2) if variant == 7 else y

    # -- one problem through the reference's own entry point, residual model on the device ------
    def optimize_device_model(self, settings, model: ModelId, x: np.ndarray, l: np.ndarray, u: np.ndarray,
                              t: np.ndarray | None = None, y: np.ndarray | None = None, m: int | None = None,
                              fd_jacobian: bool = False, tail_shortcut: bool = True, aux: np.ndarray | None = None, param: float = 0.0):
        """mir_optimize_least_squares_{d,s} (least_squares.d:705-748) with f = mir_b200_device_model_*:
        the whole solve, residuals included, runs on the GPU.  x (n,) in/out.  Returns the Result POD."""
        sfx, real, S, R, Sl, FT, _ = _types(x.dtype)
        assert isinstance(settings, S) and x.ndim == 1 and x.flags.c_contiguous
        n = x.shape[0]
        if y is not None:
            y = np.ascontiguousarray(y, dtype=x.dtype).reshape(-1); m = y.shape[0] if m is None else m
        if t is not None:
            t = np.ascontiguousarray(t, dtype=x.dtype).reshape(-1)
        l = np.ascontiguousarray(l, dtype=x.dtype); u = np.ascontiguousarray(u, dtype=x.dtype)
        if aux is not None:
            aux = np.ascontiguousarray(aux, dtype=x.dtype).reshape(-1)
        desc = ModelDesc(int(model), 0 if tail_shortcut else MODEL_NO_TAIL_SHORTCUT, _vp(t), _vp(y), _vp(aux), float(param))
        f_ptr = C.cast(getattr(self.lib, f"mir_b200_device_model_{sfx}"), C.c_void_p)
        g_ptr = None if fd_jacobian else C.cast(getattr(self.lib, f"mir_b200_device_model_jac_{sfx}"), C.c_void_p)
        fn = getattr(self.lib, f"mir_optimize_least_squares_{sfx}")
        res = fn(C.byref(settings), m, n, x.ctypes.data_as(C.POINTER(real)), l.ctypes.data_as(C.POINTER(real)),
                 u.ctypes.data_as(C.POINTER(real)), Sl(0, None), _abi.SliceI(0, None),
                 C.cast(C.pointer(desc), C.c_void_p), f_ptr, None, g_ptr, None, None)
        if res.status == _abi.LeastSquaresStatus.numericError and self.lib.mir_b200_last_error():
            raise B200Error(-1, self.lib.mir_b200_last_error().decode())
        return res

    # -- one large problem, rows sharded over ranks -------------------------------------------
    def optimize_sharded(self, settings, model: ModelId, x: np.ndarray, l: np.ndarray, u: np.ndarray, t, y,
                         comm=None, fd_jacobian: bool = False, want_stats: bool = False, stream=None, tail_shortcut: bool = True):
        """t, y: torch CUDA tensors with THIS rank's rows.  x (n,) host, identical on every rank, in/out.
        comm: handle from :meth:`nccl_comm_init` (None = single GPU, no collective).  Blocking."""
        import torch
        assert isinstance(settings, _abi.LeastSquaresSettingsD) and x.dtype == np.float64 and x.ndim == 1
        assert t.dtype == torch.float64 and y.dtype == torch.float64 and t.is_cuda and y.is_cuda
        n = x.shape[0]
        l = np.ascontiguousarray(l, dtype=np.float64); u = np.ascontiguousarray(u, dtype=np.float64)
        desc = ModelDesc(int(model), (MODEL_FD_JACOBIAN if fd_jacobian else 0) | (0 if tail_shortcut else MODEL_NO_TAIL_SHORTCUT), _vp(t), _vp(y))
        res = _abi.LeastSquaresResultD()
        stats = BatchStats() if want_stats else None
        if stream is None:
            stream = torch.cuda.current_stream(t.device).cuda_stream
        rc = self.lib.mir_optimize_least_squares_sharded_d(C.byref(settings), C.byref(desc), t.shape[0], n, _vp(x), _vp(l), _vp(u),
                                                           comm, C.c_void_p(stream), C.byref(res),
                                                           C.byref(stats) if stats is not None else None)
        self._check(rc)
        return res, (stats.as_dict() if stats is not None else None)

    def syrk_lower_device(self, J, n: int, packed, stream=None):
        """packed[tri(i,j)] = (J^T J)[i][j], i >= j; J: (rows, ldj) float64 CUDA tensor, rows % 32 == 0.  Asynchronous."""
        import torch
        if stream is None:
            stream = torch.cuda.current_stream(J.device).cuda_stream
        self._check(self.lib.mir_b200_syrk_lower_dev_d(_vp(J), J.shape[0], n, J.shape[1], _vp(packed), C.c_void_p(stream)))

    # -- NCCL bootstrap (the library binds NCCL at run time) -----------------------------------
    def nccl_unique_id(self) -> bytes:
        buf = C.create_string_buffer(128)
        self._check(self.lib.mir_b200_nccl_unique_id(buf))
        return buf.raw

    def nccl_comm_init(self, nranks: int, unique_id: bytes, rank: int):
        comm = C.c_void_p()
        self._check(self.lib.mir_b200_nccl_comm_init(C.byref(comm), nranks, C.c_char_p(unique_id), rank))
        return comm

    def nccl_comm_destroy(self, comm):
        self._check(self.lib.mir_b200_nccl_comm_destroy(comm))

    @staticmethod
    def results_from_bytes(buf, dtype) -> np.ndarray:
        """uint8 torch tensor (device or host) -> structured numpy array of Result PODs."""
        return np.frombuffer(buf.cpu().numpy().tobytes(), dtype=RESULT_DTYPES[np.dtype(dtype)])
