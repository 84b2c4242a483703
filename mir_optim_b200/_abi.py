"""ctypes mirror of include/mir_optim_b200.h.

Part 1 of the header (the reference's extern(C) surface, least_squares.d:637-799 and
boxcqp.d:31-51) is bound by :func:`bind_reference_abi`; any shared object exporting those
symbols can be bound -- the CUDA library (product) or, in tests only, the CPU oracle.
Part 2 (batched / sharded additions) is bound by :func:`bind_b200_abi`.
"""
from __future__ import annotations

import ctypes as C
import enum

lapackint = C.c_int32


class LeastSquaresStatus(enum.IntEnum):
    """least_squares.d:20-46"""
    maxIterations = -1
    furtherImprovement = 0
    xConverged = 1
    gConverged = 2
    fConverged = 3
    badBounds = -32
    badGuess = -31
    badMinStepQuality = -30
    badGoodStepQuality = -29
    badStepQuality = -28
    badLambdaParams = -27
    numericError = -26


class BoxQPStatus(enum.IntEnum):
    """boxcqp.d:18-26"""
    solved = 0
    numericError = 1
    maxIterations = 2


class ModelId(enum.IntEnum):
    LINEAR2 = 0
    ROSENBROCK = 1
    EXPDECAY2 = 2
    EXPTAU3 = 3
    SQRTCIRCLE = 4
    EXPDECAY3 = 5
    GAUSS4 = 6
    SUMEXP = 7
    GAUSSMIX = 8
    SPLINE = 9


MODEL_FD_JACOBIAN = 1
MODEL_GRID_PER_PROBLEM = 2
MODEL_NO_TAIL_SHORTCUT = 4
MODEL_AUX_PER_PROBLEM = 8
MODEL_WARM_START = 16
MODEL_WEIGHTED = 32
COV_UNSCALED = 1


def _settings_types(real):
    class BoxQPSettings(C.Structure):
        """boxcqp.d:56-71"""
        _fields_ = [("relTolerance", real), ("absTolerance", real), ("maxIterations", C.c_uint32)]

    class LeastSquaresSettings(C.Structure):
        """least_squares.d:85-123"""
        _fields_ = [
            ("maxIterations", C.c_uint32), ("maxAge", C.c_uint32),
            ("jacobianEpsilon", real), ("absTolerance", real), ("relTolerance", real),
            ("gradTolerance", real), ("maxGoodResidual", real), ("maxStep", real),
            ("maxLambda", real), ("minLambda", real), ("minStepQuality", real),
            ("goodStepQuality", real), ("lambdaIncrease", real), ("lambdaDecrease", real),
            ("qpSettings", BoxQPSettings),
        ]

    class LeastSquaresResult(C.Structure):
        """least_squares.d:128-143"""
        _fields_ = [("status", C.c_int32), ("iterations", C.c_uint32), ("fCalls", C.c_uint32),
                    ("gCalls", C.c_uint32), ("residual", real), ("lambda_", real)]

        def __repr__(self):
            return (f"LeastSquaresResult(status={LeastSquaresStatus(self.status).name}, iterations={self.iterations}, "
                    f"fCalls={self.fCalls}, gCalls={self.gCalls}, residual={self.residual!r}, lambda={self.lambda_!r})")

    class Slice(C.Structure):
        _fields_ = [("length", C.c_size_t), ("ptr", C.POINTER(real))]

    return BoxQPSettings, LeastSquaresSettings, LeastSquaresResult, Slice


BoxQPSettingsD, LeastSquaresSettingsD, LeastSquaresResultD, SliceD = _settings_types(C.c_double)
BoxQPSettingsS, LeastSquaresSettingsS, LeastSquaresResultS, SliceS = _settings_types(C.c_float)


class SliceI(C.Structure):
    _fields_ = [("length", C.c_size_t), ("ptr", C.POINTER(lapackint))]


class LSTask(C.Structure):
    """D delegate LeastSquaresTask (least_squares.d:560-564), opaque 16 bytes."""
    _fields_ = [("context", C.c_void_p), ("funcptr", C.c_void_p)]


class ModelDesc(C.Structure):
    _fields_ = [("model", C.c_uint32), ("flags", C.c_uint32), ("t", C.c_void_p), ("y", C.c_void_p),
                ("aux", C.c_void_p), ("param", C.c_double), ("w", C.c_void_p)]


class BatchStats(C.Structure):
    _fields_ = [(k, C.c_uint64) for k in ("problems", "passes", "accepted", "fresh_jacobians", "broyden_updates",
                                         "model_evals", "qp_solves", "qp_iterations")]

    def as_dict(self):
        return {k: int(getattr(self, k)) for k, _ in self._fields_}


# callback types, least_squares.d:78-80, 567-572, 672-678
FunctionD = C.CFUNCTYPE(None, C.c_void_p, C.c_size_t, C.c_size_t, C.POINTER(C.c_double), C.POINTER(C.c_double))
JacobianD = FunctionD
FunctionS = C.CFUNCTYPE(None, C.c_void_p, C.c_size_t, C.c_size_t, C.POINTER(C.c_float), C.POINTER(C.c_float))
JacobianS = FunctionS
TaskFn = C.CFUNCTYPE(None, LSTask, C.c_uint, C.c_uint, C.c_uint)
ThreadManager = C.CFUNCTYPE(None, C.c_void_p, C.c_uint, LSTask, TaskFn)

REFERENCE_SYMBOLS = [
    "mir_least_squares_work_length", "mir_least_squares_iwork_length",
    "mir_box_qp_work_length", "mir_box_qp_iwork_length",
    "mir_least_squares_status_string",
    "mir_least_squares_init_d", "mir_least_squares_init_s",
    "mir_least_squares_reset_d", "mir_least_squares_reset_s",
    "mir_optimize_least_squares_d", "mir_optimize_least_squares_s",
]

B200_SYMBOLS = [
    "mir_b200_last_error", "mir_b200_kernel_launches", "mir_b200_device_count", "mir_b200_version",
    "mir_b200_measure_peak_tflops",
    "mir_b200_device_model_d", "mir_b200_device_model_jac_d", "mir_b200_device_model_s", "mir_b200_device_model_jac_s",
    "mir_optimize_least_squares_batched_d", "mir_optimize_least_squares_batched_s",
    "mir_optimize_least_squares_batched_dev_d", "mir_optimize_least_squares_batched_dev_s",
    "mir_solve_box_qp_d", "mir_solve_box_qp_s",
    "mir_solve_box_qp_batched_d", "mir_solve_box_qp_batched_s",
    "mir_solve_box_qp_batched_dev_d", "mir_solve_box_qp_batched_dev_s",
    "mir_optimize_least_squares_sharded_d", "mir_b200_syrk_lower_dev_d",
    "mir_b200_posvx_batched_d", "mir_b200_posvx_batched_s",
    "mir_b200_math_hook_d", "mir_b200_math_hook_s",
    "mir_b200_nccl_unique_id", "mir_b200_nccl_comm_init", "mir_b200_nccl_comm_destroy",
    "mir_fit_spline_d", "mir_fit_spline_s", "mir_fit_spline_batched_d", "mir_fit_spline_batched_s",
    "mir_b200_model_compile", "mir_b200_model_release",
    "mir_b200_covariance_batched_d", "mir_b200_covariance_batched_s",
    "mir_b200_covariance_batched_dev_d", "mir_b200_covariance_batched_dev_s",
]


def bind_reference_abi(lib):
    """Attach argtypes/restypes for the reference's extern(C) symbols to `lib` (a ctypes.CDLL)."""
    for name in ("mir_least_squares_work_length", "mir_least_squares_iwork_length"):
        fn = getattr(lib, name); fn.argtypes = [C.c_size_t, C.c_size_t]; fn.restype = C.c_size_t
    for name in ("mir_box_qp_work_length", "mir_box_qp_iwork_length"):
        fn = getattr(lib, name); fn.argtypes = [C.c_size_t]; fn.restype = C.c_size_t
    lib.mir_least_squares_status_string.argtypes = [C.c_int]
    lib.mir_least_squares_status_string.restype = C.c_char_p
    for sfx, S in (("d", LeastSquaresSettingsD), ("s", LeastSquaresSettingsS)):
        for op in ("init", "reset"):
            fn = getattr(lib, f"mir_least_squares_{op}_{sfx}"); fn.argtypes = [C.POINTER(S)]; fn.restype = None
    for sfx, S, R, Sl, real in (("d", LeastSquaresSettingsD, LeastSquaresResultD, SliceD, C.c_double),
                                ("s", LeastSquaresSettingsS, LeastSquaresResultS, SliceS, C.c_float)):
        fn = getattr(lib, f"mir_optimize_least_squares_{sfx}")
        fn.argtypes = [C.POINTER(S), C.c_size_t, C.c_size_t, C.POINTER(real), C.POINTER(real), C.POINTER(real),
                       Sl, SliceI, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        fn.restype = R
    return lib


def bind_b200_abi(lib):
    """Attach prototypes for part 2 of the header (this engine's additions)."""
    lib.mir_b200_last_error.argtypes = []; lib.mir_b200_last_error.restype = C.c_char_p
    lib.mir_b200_kernel_launches.argtypes = []; lib.mir_b200_kernel_launches.restype = C.c_uint64
    lib.mir_b200_device_count.argtypes = []; lib.mir_b200_device_count.restype = C.c_int
    lib.mir_b200_version.argtypes = []; lib.mir_b200_version.restype = C.c_char_p
    lib.mir_b200_measure_peak_tflops.argtypes = [C.c_int, C.c_int]; lib.mir_b200_measure_peak_tflops.restype = C.c_double
    vp = C.c_void_p
    for sfx, S, R, Q in (("d", LeastSquaresSettingsD, LeastSquaresResultD, BoxQPSettingsD),
                         ("s", LeastSquaresSettingsS, LeastSquaresResultS, BoxQPSettingsS)):
        for dev in ("", "_dev"):
            fn = getattr(lib, f"mir_optimize_least_squares_batched{dev}_{sfx}")
            fn.argtypes = [C.POINTER(S), C.POINTER(ModelDesc), C.c_size_t, C.c_size_t, C.c_size_t,
                           vp, vp, vp, C.c_size_t, vp, vp, vp if dev else C.c_int]
            fn.restype = C.c_int
            fn = getattr(lib, f"mir_solve_box_qp_batched{dev}_{sfx}")
            fn.argtypes = [C.POINTER(Q), C.c_size_t, C.c_size_t, vp, vp, vp, vp, vp, vp, vp, vp if dev else C.c_int]
            fn.restype = C.c_int
        fn = getattr(lib, f"mir_solve_box_qp_{sfx}")
        fn.argtypes = [C.POINTER(Q), C.c_size_t, vp, vp, vp, vp, vp]
        fn.restype = C.c_int
        for dev in ("", "_dev"):
            fn = getattr(lib, f"mir_b200_covariance_batched{dev}_{sfx}")
            fn.argtypes = [C.POINTER(S), C.POINTER(ModelDesc), C.c_size_t, C.c_size_t, C.c_size_t,
                           vp, vp, vp, C.c_size_t, C.c_uint, vp, vp, vp, vp if dev else C.c_int]
            fn.restype = C.c_int
    fn = lib.mir_optimize_least_squares_sharded_d
    fn.argtypes = [C.POINTER(LeastSquaresSettingsD), C.POINTER(ModelDesc), C.c_size_t, C.c_size_t, vp, vp, vp,
                   vp, vp, C.POINTER(LeastSquaresResultD), C.POINTER(BatchStats)]
    fn.restype = C.c_int
    lib.mir_b200_syrk_lower_dev_d.argtypes = [vp, C.c_size_t, C.c_size_t, C.c_size_t, vp, vp]
    lib.mir_b200_syrk_lower_dev_d.restype = C.c_int
    for sfx in ("d", "s"):
        fn = getattr(lib, f"mir_b200_posvx_batched_{sfx}")
        fn.argtypes = [C.c_int, C.c_size_t, C.c_size_t, vp, vp, vp, vp, vp, C.c_int]; fn.restype = C.c_int
        fn = getattr(lib, f"mir_b200_math_hook_{sfx}")
        fn.argtypes = [C.c_int, C.c_size_t, vp, vp, vp, C.c_int]; fn.restype = C.c_int
    for sfx, S, R, real in (("d", LeastSquaresSettingsD, LeastSquaresResultD, C.c_double), ("s", LeastSquaresSettingsS, LeastSquaresResultS, C.c_float)):
        fn = getattr(lib, f"mir_fit_spline_{sfx}")
        fn.argtypes = [C.POINTER(S), C.c_size_t, vp, vp, C.c_size_t, vp, vp, vp, real, vp, C.POINTER(R)]; fn.restype = C.c_int
        fn = getattr(lib, f"mir_fit_spline_batched_{sfx}")
        fn.argtypes = [C.POINTER(S), C.c_size_t, C.c_size_t, vp, vp, C.c_size_t, vp, vp, vp, real, C.c_uint, vp, vp, C.c_int]; fn.restype = C.c_int
    lib.mir_b200_model_compile.argtypes = [C.c_char_p, C.POINTER(C.c_uint32)]; lib.mir_b200_model_compile.restype = C.c_int
    lib.mir_b200_model_release.argtypes = [C.c_uint32]; lib.mir_b200_model_release.restype = C.c_int
    lib.mir_b200_nccl_unique_id.argtypes = [vp]; lib.mir_b200_nccl_unique_id.restype = C.c_int
    lib.mir_b200_nccl_comm_init.argtypes = [C.POINTER(vp), C.c_int, vp, C.c_int]; lib.mir_b200_nccl_comm_init.restype = C.c_int
    lib.mir_b200_nccl_comm_destroy.argtypes = [vp]; lib.mir_b200_nccl_comm_destroy.restype = C.c_int
    return lib
