/*
 * mir_optim_b200.h -- C ABI of the B200-native Levenberg-Marquardt / BOXCQP engine.
 *
 * This header is the drop-in boundary.  Part 1 re-declares, symbol for symbol, the
 * extern(C) surface of libmir/mir-optim (the reference) so that the reference's own D
 * wrappers (`optimize`, `optimizeLeastSquares`, `solveBoxQP`) or any C caller can bind to
 * libmir_optim_b200.so instead of the D/LAPACK build.  Part 2 adds the batched, device
 * resident and row-sharded entry points that the reference does not have; they take the
 * same Settings / Result PODs unchanged.
 *
 * Citations are to the reference tree:
 *   LS = source/mir/optim/least_squares.d      BQ = source/mir/optim/boxcqp.d
 *
 * All functions are nothrow, re-entrant, and never abort; failures are reported through
 * the LeastSquaresStatus / BoxQPStatus enums (reference convention, LS:20-46, BQ:18-26) or,
 * for the new entry points, through a non-zero mir_b200_error return value.
 */
#ifndef MIR_OPTIM_B200_H
#define MIR_OPTIM_B200_H

#ifdef __CUDACC_RTC__   /* run-time compilation of user models (NVRTC has no C library headers) */
typedef unsigned long long uint64_t; typedef unsigned int uint32_t; typedef int int32_t; typedef unsigned long uintptr_t;
#else
#include <stddef.h>
#include <stdint.h>
#endif

#ifdef __cplusplus
extern "C" {
#endif

/* ------------------------------------------------------------------------------------
 * Part 1 -- the reference's own extern(C) surface (types + symbols)
 * ---------------------------------------------------------------------------------- */

/* `lapackint` (LS:16): 32-bit unless an ILP64 LAPACK configuration is chosen (dub.sdl:50-52). */
typedef int32_t mir_lapackint;

/* enum LeastSquaresStatus, LS:20-46 */
typedef enum mir_least_squares_status {
    mir_ls_maxIterations      = -1,
    mir_ls_furtherImprovement = 0,
    mir_ls_xConverged         = 1,
    mir_ls_gConverged         = 2,
    mir_ls_fConverged         = 3,
    mir_ls_badBounds          = -32,
    mir_ls_badGuess           = -31,
    mir_ls_badMinStepQuality  = -30,
    mir_ls_badGoodStepQuality = -29,
    mir_ls_badStepQuality     = -28,
    mir_ls_badLambdaParams    = -27,
    mir_ls_numericError       = -26
} mir_least_squares_status;

/* enum BoxQPStatus, BQ:18-26 */
typedef enum mir_box_qp_status {
    mir_qp_solved        = 0,
    mir_qp_numericError  = 1,
    mir_qp_maxIterations = 2
} mir_box_qp_status;

/* struct BoxQPSettings!T, BQ:56-71.  Defaults: relTolerance = absTolerance = 16*eps,
 * maxIterations = 0 (meaning 10*n + 100, BQ:224-226). */
typedef struct mir_box_qp_settings_d {
    double   relTolerance;
    double   absTolerance;
    uint32_t maxIterations;
} mir_box_qp_settings_d;                       /* 24 bytes */

typedef struct mir_box_qp_settings_s {
    float    relTolerance;
    float    absTolerance;
    uint32_t maxIterations;
} mir_box_qp_settings_s;                       /* 12 bytes */

/* struct LeastSquaresSettings!T, LS:85-123 (field order and defaults are the reference's). */
typedef struct mir_least_squares_settings_d {
    uint32_t maxIterations;     /* 1000 */
    uint32_t maxAge;            /* 0 => g ? 3 : 2n  (LS:945) */
    double   jacobianEpsilon;   /* 2^-26, absolute central-difference step (LS:98, 1028-1029) */
    double   absTolerance;      /* eps */
    double   relTolerance;      /* 0 */
    double   gradTolerance;     /* eps */
    double   maxGoodResidual;   /* eps^2 */
    double   maxStep;           /* sqrt(max)/16 */
    double   maxLambda;         /* max/16 */
    double   minLambda;         /* min_normal*16 */
    double   minStepQuality;    /* 0.1 */
    double   goodStepQuality;   /* 0.5 */
    double   lambdaIncrease;    /* 2 */
    double   lambdaDecrease;    /* 1/(2*phi) */
    mir_box_qp_settings_d qpSettings;
} mir_least_squares_settings_d;                /* 128 bytes */

typedef struct mir_least_squares_settings_s {
    uint32_t maxIterations;
    uint32_t maxAge;
    float    jacobianEpsilon;   /* 2^-11 */
    float    absTolerance;
    float    relTolerance;
    float    gradTolerance;
    float    maxGoodResidual;
    float    maxStep;
    float    maxLambda;
    float    minLambda;
    float    minStepQuality;
    float    goodStepQuality;
    float    lambdaIncrease;
    float    lambdaDecrease;
    mir_box_qp_settings_s qpSettings;
} mir_least_squares_settings_s;                /* 68 bytes */

/* struct LeastSquaresResult!T, LS:128-143.  Returned BY VALUE by the reference. */
typedef struct mir_least_squares_result_d {
    int32_t  status;            /* mir_least_squares_status; .init = numericError */
    uint32_t iterations;        /* accepted steps */
    uint32_t fCalls;
    uint32_t gCalls;
    double   residual;          /* ||f(x)||^2; .init = +inf */
    double   lambda;            /* last damping value */
} mir_least_squares_result_d;                  /* 32 bytes */

typedef struct mir_least_squares_result_s {
    int32_t  status;
    uint32_t iterations;
    uint32_t fCalls;
    uint32_t gCalls;
    float    residual;
    float    lambda;
} mir_least_squares_result_s;                  /* 24 bytes */

/* mir.ndslice `Slice!(T*)` (Contiguous, 1-D) as passed by value at LS:713-714: {length, ptr}. */
typedef struct mir_slice_d  { size_t length; double*        ptr; } mir_slice_d;
typedef struct mir_slice_s  { size_t length; float*         ptr; } mir_slice_s;
typedef struct mir_slice_i  { size_t length; mir_lapackint* ptr; } mir_slice_i;

/* LeastSquaresFunctionBetterC / LeastSquaresJacobianBetterC, LS:78-80.  J is row-major m x n. */
typedef void (*mir_ls_function_d)(void* context, size_t m, size_t n, const double* x, double* y);
typedef void (*mir_ls_jacobian_d)(void* context, size_t m, size_t n, const double* x, double* J);
typedef void (*mir_ls_function_s)(void* context, size_t m, size_t n, const float* x, float* y);
typedef void (*mir_ls_jacobian_s)(void* context, size_t m, size_t n, const float* x, float* J);

/* LeastSquaresTask is a D delegate (LS:560-564): {context pointer, function pointer}, 16 bytes,
 * passed by value; opaque to C.  LeastSquaresTaskBetterC LS:567-572, thread manager LS:672-678. */
typedef struct mir_ls_task { void* context; void* funcptr; } mir_ls_task;
typedef void (*mir_ls_task_fn)(mir_ls_task task, unsigned totalThreads, unsigned threadId, unsigned i);
typedef void (*mir_ls_thread_manager)(void* context, unsigned count, mir_ls_task task, mir_ls_task_fn fn);

/* LS:642-646: mir_box_qp_work_length(n) + 5n + n^2 + n*m + 2m  T-elements. */
size_t mir_least_squares_work_length(size_t m, size_t n);
/* LS:651-656: max(mir_box_qp_iwork_length(n), n) lapackints. */
size_t mir_least_squares_iwork_length(size_t m, size_t n);
/* BQ:36-42: 2n^2 + 8n.   BQ:47-50: n + ceil(n / sizeof(lapackint)). */
size_t mir_box_qp_work_length(size_t n);
size_t mir_box_qp_iwork_length(size_t n);

/* LS:666-669 (strings LS:528-557).  NUL-terminated, static storage. */
const char* mir_least_squares_status_string(int status);

/* LS:761-792: both assign LeastSquaresSettings!T.init. */
void mir_least_squares_init_d (mir_least_squares_settings_d* settings);
void mir_least_squares_init_s (mir_least_squares_settings_s* settings);
void mir_least_squares_reset_d(mir_least_squares_settings_d* settings);
void mir_least_squares_reset_s(mir_least_squares_settings_s* settings);

/*
 * LS:705-724 / LS:729-748.  Same signature, argument meaning and status codes as the
 * reference.  `x` is in/out; `work`/`iwork` are caller scratch of at least the advertised
 * lengths (kept for ABI compatibility; the engine's state lives in device memory).
 *
 * Execution: the LM state machine and all dense algebra (J^T r, J^T J, damped BoxQP /
 * Cholesky step, gain ratio, lambda control) run on the GPU.  `f`/`g` are host function
 * pointers and are therefore evaluated on the host once per pass and staged to the device
 * (host-callback mode), unless `f == mir_b200_device_model_{d,s}`: then `fContext` points to a
 * mir_model_desc whose arrays are HOST pointers and the whole solve, residuals included,
 * runs on-device (g == NULL selects the finite-difference Jacobian exactly as in the
 * reference, g == mir_b200_device_model_jac_{d,s} the analytic one).
 * The float entry runs with the real `m`; the reference passes the literal 2 (LS:629), which
 * is a defect we do not reproduce (DESIGN.md, "deviations").
 * There is no CPU fallback: without a usable CUDA device the result is status numericError
 * and mir_b200_last_error() explains why.
 */
mir_least_squares_result_d mir_optimize_least_squares_d(
    const mir_least_squares_settings_d* settings, size_t m, size_t n,
    double* x, const double* l, const double* u,
    mir_slice_d work, mir_slice_i iwork,
    void* fContext, mir_ls_function_d f,
    void* gContext, mir_ls_jacobian_d g,
    void* tmContext, mir_ls_thread_manager tm);

mir_least_squares_result_s mir_optimize_least_squares_s(
    const mir_least_squares_settings_s* settings, size_t m, size_t n,
    float* x, const float* l, const float* u,
    mir_slice_s work, mir_slice_i iwork,
    void* fContext, mir_ls_function_s f,
    void* gContext, mir_ls_jacobian_s g,
    void* tmContext, mir_ls_thread_manager tm);

/* ------------------------------------------------------------------------------------
 * Part 2 -- additions of this engine
 * ---------------------------------------------------------------------------------- */

typedef enum mir_b200_error {
    MIR_B200_OK            = 0,
    MIR_B200_ENODEVICE     = 1,   /* no CUDA device / driver: there is no CPU fallback        */
    MIR_B200_EINVAL        = 2,   /* bad argument (null pointer, unknown model, n mismatch)   */
    MIR_B200_EUNSUPPORTED  = 3,   /* shape outside what the kernels are instantiated for      */
    MIR_B200_ECUDA         = 4,   /* a CUDA runtime call failed                               */
    MIR_B200_ENCCL         = 5    /* NCCL could not be loaded or a collective failed          */
} mir_b200_error;

/* Human-readable description of the last error on the calling thread ("" if none). */
const char* mir_b200_last_error(void);
/* Number of kernels this library has launched so far in this process (all threads). */
uint64_t    mir_b200_kernel_launches(void);
/* Number of visible CUDA devices (0 when there is none; never fails). */
int         mir_b200_device_count(void);
const char* mir_b200_version(void);
/* Roofline denominators not in MEASURED_PEAKS.json, measured on the current device:
 * kind 0 = FP64 FMA pipe, 1 = FP64 tensor (mma.sync m8n8k4 f64 -> DMMA), 2 = FP32 FMA pipe.
 * Returns TFLOP/s (best of `reps` launches) or a negative mir_b200_error. */
double      mir_b200_measure_peak_tflops(int kind, int reps);

/*
 * Device residual models ("device functors").  r = residual vector (length m), p = parameters
 * (length n), t = abscissa, y = observations.  Every model has an analytic Jacobian on
 * the device; MIR_MODEL_FD_JACOBIAN ignores it and uses the reference's central difference
 * (LS:1016-1050), i.e. the behaviour of passing g == null.
 */
typedef enum mir_model_id {
    MIR_MODEL_LINEAR2       = 0,  /* r = (p0, 2 - p1)                       m=2 n=2  (LS:217-245)  */
    MIR_MODEL_ROSENBROCK    = 1,  /* r = (10 (p1 - p0^2), 1 - p0)           m=2 n=2  (LS:247-331)  */
    MIR_MODEL_EXPDECAY2     = 2,  /* r_i = p0 exp(-t_i p1) - y_i            n=2      (LS:333-363)  */
    MIR_MODEL_EXPTAU3       = 3,  /* r_i = p0 exp(-t_i / p1) + p2 - y_i     n=3      (LS:365-411)  */
    MIR_MODEL_SQRTCIRCLE    = 4,  /* r   = sqrt(1 - (p0^2 + p1^2))          m=1 n=2  (LS:413-434)  */
    MIR_MODEL_EXPDECAY3     = 5,  /* r_i = p0 exp(-p1 t_i) + p2 - y_i       n=3      BASELINE configs[0] */
    MIR_MODEL_GAUSS4        = 6,  /* r_i = p0 exp(-(t_i-p1)^2/(2 p2^2)) + p3 - y_i   n=4  configs[1] */
    MIR_MODEL_SUMEXP        = 7,  /* r_i = sum_k p[2k] exp(-p[2k+1] t_i) - y_i       n=8  configs[2] */
    MIR_MODEL_GAUSSMIX      = 8,  /* r_i = sum_k p[3k] exp(-(t_i-p[3k+1])^2/(2 p[3k+2]^2))
                                            + p[n-2] + p[n-1] t_i - y_i   n=3K+2   configs[3] */
    MIR_MODEL_SPLINE        = 9,  /* fitSpline's residual (fit_splie.d:58-80): p = values of a C2 cubic spline
                                     (not-a-knot ends) at the knots `aux`; r_i = spline(t_i) - y_i, last row =
                                     sqrt(param * integral term); n = number of knots >= 2; finite differences only */
    MIR_MODEL_COUNT_,
    MIR_MODEL_USER_BASE     = 0x1000  /* ids returned by mir_b200_model_compile (models compiled at run time) */
} mir_model_id;

enum {
    MIR_MODEL_FD_JACOBIAN      = 1u,  /* g == null semantics: central differences, maxAge default 2n */
    MIR_MODEL_GRID_PER_PROBLEM = 2u,  /* t has batch*m entries instead of m shared ones              */
    MIR_MODEL_NO_TAIL_SHORTCUT = 4u,  /* verification only: execute every pass of the lambda-overflow tail
                                         instead of fast-forwarding it (results are identical, DESIGN.md 4.3) */
    MIR_MODEL_AUX_PER_PROBLEM  = 8u,  /* aux has batch*n entries instead of n shared ones                   */
    MIR_MODEL_WARM_START       = 16u, /* batched entries: results[b].lambda on entry (> 0, finite) is the initial
                                         damping instead of 0 (LS:966); the reference documents Result.lambda as
                                         the initial trust-region value (LS:141-142) but never reads it back.
                                         Chain it with the x of a previous call to continue a fit.            */
    MIR_MODEL_WEIGHTED         = 32u, /* per-observation weights in model->w (an extension; the reference has none):
                                         every row's residual and Jacobian row are scaled by w_i, see mir_model_desc */
    MIR_MODEL_LOSS_SOFT_L1     = 64u, /* robust loss rho(z) = 2 (sqrt(1 + z) - 1) (scipy's least_squares(loss=
                                         'soft_l1')); an extension, see "Robust losses" below                     */
    MIR_MODEL_LOSS_HUBER       = 128u /* robust loss rho(z) = z (z <= 1), 2 sqrt(z) - 1 (z > 1) (loss='huber');
                                         at most one of the two loss flags                                       */
};

typedef struct mir_model_desc {
    uint32_t    model;   /* mir_model_id */
    uint32_t    flags;
    const void* t;       /* abscissa, T[m] (shared) or T[batch*m]; NULL for data-free models */
    const void* y;       /* observations, T[batch*m]; NULL for data-free models             */
    const void* aux;     /* model constants, T[n] (shared) or T[batch*n]: the knots of MIR_MODEL_SPLINE; else NULL */
    double      param;   /* model constant: the smoothing weight lambda of MIR_MODEL_SPLINE; else 0  */
    const void* w;       /* observation weights, T[batch*m], row-aligned with y; used only with MIR_MODEL_WEIGHTED */
} mir_model_desc;                              /* 48 bytes (40 before w was added: the library copies the whole
                                                  struct, so binaries built against the older header must be rebuilt) */

/*
 * Weighted least squares (MIR_MODEL_WEIGHTED).  For every row i < m of a problem the solver sees
 *     r~_i = w_i * r_i(p)        (rounded once in T)
 *     J~_ij = w_i * J_ij         (analytic Jacobian, each entry rounded once); the finite-difference Jacobian is the
 *                                reference's central difference (LS:1016-1050, with the bound clamp) taken of r~
 * and everything downstream -- the LM loop, Result.residual = sum r~_i^2 (chi^2 with w = 1/sigma), the g-test, J^T J, the
 * covariance -- is exactly the reference run with f = w (.) r.  w follows y: host pointer in the host forms, device
 * pointer in the _dev_ forms.  Values are the caller's contract, like y: w_i = 0 removes row i (pad short problems of a
 * ragged batch to a common m with zero weights; the padded rows' residuals must still be finite, since 0 * inf is NaN),
 * and a non-finite weight acts like a non-finite observation.
 * Honoured by mir_optimize_least_squares_batched_{d,s} / _dev_{d,s} and mir_b200_covariance_batched_{d,s} / _dev_{d,s}
 * (with any of the other flags); weighted fits always run the general batched kernel (lm_cta.cuh).  MIR_B200_EINVAL
 * for w == NULL (batch > 0, m > 0); MIR_B200_EUNSUPPORTED for the data-free models LINEAR2, ROSENBROCK and SQRTCIRCLE
 * and from mir_optimize_least_squares_sharded_d.  The legacy entry points in device-model mode return numericError.
 */

/*
 * Robust losses (MIR_MODEL_LOSS_SOFT_L1, MIR_MODEL_LOSS_HUBER; an extension, the reference has none).  Outlier-resistant
 * fitting as scipy's least_squares(loss=...), minimising sum_i rho(u_i^2) with u_i = w_i r_i (MIR_MODEL_WEIGHTED) or
 * u_i = r_i.  There is no separate scale: the weights are the scale, so least_squares(loss=L, f_scale=C) is w_i = 1/C and
 * curve_fit(sigma=s, loss=L) is w = 1/s; each problem (each row) can have its own.  With z = u^2:
 *     soft_l1   rho(z) = 2 (sqrt(1 + z) - 1)
 *     huber     rho(z) = z for z <= 1, 2 sqrt(z) - 1 otherwise
 * The solver sees the square-root form, row by row: the residual f~_i = sign(u_i) sqrt(rho(u_i^2)), so sum f~_i^2 =
 * sum rho(u_i^2), and the Jacobian row J~_i = g(u_i) (w_i J_i) with g = d f~ / du = rho'(u^2) |u| / sqrt(rho(u^2)).  A
 * finite-difference Jacobian is the reference's central difference (LS:1016-1050, with the bound clamp) taken of f~.
 * Everything downstream is the reference run with f = f~:
 *   Result.residual = sum rho(u_i^2): 2 * scipy's cost with f_scale = 1, and 2 cost / C^2 with w = 1/C in place of
 *                     f_scale = C; maxGoodResidual is compared with that sum.
 *   g-test            J~^T f~ = sum rho'(u^2) u grad(u), the gradient of sum rho / 2.
 *   solutions         the stationary points of scipy's robust objective.  The iterates differ from scipy's (which runs TRF
 *                     with a Triggs-corrected Jacobian), so compare at the solution.
 * Each operation below is rounded once in T (no contraction), with a = |u|, and f~ = -F for u < 0, else F:
 *   huber,   a <= 1:  f~ = u, g = 1 (the row is bit for bit the squared-loss row)
 *   huber,   a > 1:   v = a - 0.5;  F = 2 * sqrt(0.5 * v);  g = 1 / F
 *   soft_l1, a <= 1:  s = sqrt(1 + a * a);  r = sqrt(0.5 * (s + 1));  F = a / r (f~ = u / r);  g = r / s
 *   soft_l1, a > 1:   q = 1 / a;  c = sqrt(1 + q * q);  r = sqrt(0.5 * (c + q));  b = sqrt(a);  F = b / r;  g = r / (b * c)
 *   J~_ij = g * (w_i * J_ij) (w_i = 1 without MIR_MODEL_WEIGHTED)
 * The a > 1 forms never square u and never divide into the subnormals (q only meets 1 and c), so for every finite u, in
 * both precisions, f~ and g are finite and within 4 ulp of their exact values (the naive u sqrt(2 / (s + 1)) gives f~ = 0
 * for a float |u| > 1.8e19, and such a trial point would be accepted).  A NaN or infinite u gives a NaN or infinite f~,
 * which the reference's non-finite handling (LS:1117-1122) treats as for any residual.  f~^2 ~ 2|u| overflows in T only
 * for |u| near the largest finite value.
 * Honoured by mir_optimize_least_squares_batched_{d,s} / _dev_{d,s} with any of the other flags; robust fits always run
 * the general batched kernel (lm_cta.cuh).  MIR_B200_EINVAL for both loss flags at once; MIR_B200_EUNSUPPORTED for
 * LINEAR2, ROSENBROCK and SQRTCIRCLE, from mir_b200_covariance_batched_* (a covariance of a robust fit is not defined
 * here: the squared-loss covariance at a robust solution would mislead) and from mir_optimize_least_squares_sharded_d.
 * The legacy entry points in device-model mode return numericError.  mir_b200_predict_batched_* ignores the flags (a
 * prediction is of f).  User models compile their robust program at the first robust fit per precision.
 */

/*
 * User-defined residual models on the device (the reference takes arbitrary f / g, LS:78-80; SURVEY 8f-2).  `source`
 * is CUDA C++ defining, in the global namespace,
 *
 *     template <class REAL> struct UserModel {
 *         static constexpr bool kAnalytic = false;       // true: jacobian() below is provided
 *         // residual of row `row` (0 <= row < m) for the parameters p[n]; t, y: the row's entries of model->t / model->y
 *         // (0 when those are NULL); aux: model->aux of this problem (may be NULL); param: model->param
 *         __device__ static REAL residual(const REAL* p, int n, int m, int row, REAL t, REAL y, const REAL* aux, REAL param);
 *         // row `row` of the Jacobian, d residual / d p[k] into Jrow[k]
 *         __device__ static void jacobian(const REAL* p, int n, int m, int row, REAL t, REAL y, const REAL* aux, REAL param, REAL* Jrow);
 *     };
 *
 * It is compiled with NVRTC for sm_100a together with the general batched LM kernel (lm_cta.cuh, whose sources are
 * embedded in the library) at the first use per precision; the returned id (>= MIR_MODEL_USER_BASE) goes into
 * mir_model_desc.model of the batched entry points -- or of the legacy entry point in device-model mode, which gives the
 * reference's own signature a GPU path for user models.  libnvrtc.so.12 and libcuda.so.1 are bound at run time.
 * Compile errors: MIR_B200_EINVAL, the NVRTC log is in mir_b200_last_error().  Without this, arbitrary f / g passed as
 * host function pointers run on the host with one transfer of y (and J) per pass (host-callback mode).
 */
int  mir_b200_model_compile(const char* source, uint32_t* model_id);
int  mir_b200_model_release(uint32_t model_id);

/* Sentinels for the legacy entry points: pass as `f` / `g` with fContext = mir_model_desc*. */
void mir_b200_device_model_d    (void* context, size_t m, size_t n, const double* x, double* y);
void mir_b200_device_model_jac_d(void* context, size_t m, size_t n, const double* x, double* J);
void mir_b200_device_model_s    (void* context, size_t m, size_t n, const float* x, float* y);
void mir_b200_device_model_jac_s(void* context, size_t m, size_t n, const float* x, float* J);

/* Work counters summed over a batch (device side, for roofline accounting). */
typedef struct mir_batch_stats {
    uint64_t problems;       /* problems processed                                   */
    uint64_t passes;         /* loop passes (LS:972-1175), accepted or not           */
    uint64_t accepted;       /* accepted steps (= sum of Result.iterations)          */
    uint64_t fresh_jacobians;/* analytic or finite-difference Jacobian evaluations   */
    uint64_t broyden_updates;/* rank-1 updates (LS:1001-1006)                        */
    uint64_t model_evals;    /* residual-vector evaluations actually executed        */
    uint64_t qp_solves;      /* posvx-equivalent solves (1 + active-set iterations)  */
    uint64_t qp_iterations;  /* BOXCQP main-loop iterations (BQ:234)                 */
} mir_batch_stats;

/*
 * Batched LM: `batch` independent problems of identical shape (m, n), each with the
 * semantics of one mir_optimize_least_squares_{d,s} call (LS:877-1176) with
 * f = model, g = model's analytic Jacobian (or null with MIR_MODEL_FD_JACOBIAN).
 *   x        T[batch*n]  in: initial guesses, out: solutions
 *   l, u     T[n] shared by all problems when bound_stride == 0, else T[batch*bound_stride]
 *   results  one reference Result POD per problem
 *   stats    optional (may be NULL)
 * Host-pointer form: copies inputs to `device` (-1 = current), runs, copies x/results back.
 * Returns mir_b200_error.  A failing problem (e.g. numericError) never affects its neighbours.
 */
int mir_optimize_least_squares_batched_d(
    const mir_least_squares_settings_d* settings, const mir_model_desc* model,
    size_t batch, size_t m, size_t n,
    double* x, const double* l, const double* u, size_t bound_stride,
    mir_least_squares_result_d* results, mir_batch_stats* stats, int device);

int mir_optimize_least_squares_batched_s(
    const mir_least_squares_settings_s* settings, const mir_model_desc* model,
    size_t batch, size_t m, size_t n,
    float* x, const float* l, const float* u, size_t bound_stride,
    mir_least_squares_result_s* results, mir_batch_stats* stats, int device);

/* Device-resident form: every pointer (model->t, model->y, x, l, u, results, stats) is a
 * device pointer on the current device; `settings` and `model` themselves are host structs.
 * Enqueued on `cuda_stream` (a cudaStream_t, NULL = legacy default stream); asynchronous. */
int mir_optimize_least_squares_batched_dev_d(
    const mir_least_squares_settings_d* settings, const mir_model_desc* model,
    size_t batch, size_t m, size_t n,
    double* x, const double* l, const double* u, size_t bound_stride,
    mir_least_squares_result_d* results, mir_batch_stats* stats, void* cuda_stream);

int mir_optimize_least_squares_batched_dev_s(
    const mir_least_squares_settings_s* settings, const mir_model_desc* model,
    size_t batch, size_t m, size_t n,
    float* x, const float* l, const float* u, size_t bound_stride,
    mir_least_squares_result_s* results, mir_batch_stats* stats, void* cuda_stream);

/*
 * Batched parameter covariance and standard errors at a given point (normally the x of a fit).  The reference has no
 * covariance; this is an extension.  For one problem, with x the given parameters, r = f(x) (m rows) and J = dr/dx at x:
 *
 *   Free set   F = { i : l_i < x_i < u_i }.  A parameter exactly on a bound is fixed (the fit clamps its trial point with
 *              max(min(., u), l), LS:1108-1110, so an active bound holds exactly).  n_F = |F|.
 *   Jacobian   the model's analytic Jacobian, or the reference's central difference when MIR_MODEL_FD_JACOBIAN is set or
 *              the model has none: settings->jacobianEpsilon and the bound clamp of LS:1030-1047, so a free parameter
 *              within h of a bound gets the same one-sided difference the fit used.
 *   Normal     A = J_F^T J_F and ||r||^2, accumulated in double also for float problems (float times float is exact in
 *   matrix     double).
 *   Inverse    S = D^-1/2 A D^-1/2 with D = diag(A); the Cholesky factor of S is inverted (LAPACK ?potrf + ?potri
 *              semantics) and unscaled.  A zero diagonal entry of A, or a pivot <= 0 or NaN, stops the factorisation.
 *   Scale      s^2 = ||r||^2 / (m - n_F); with MIR_COV_UNSCALED s^2 = 1.  With MIR_MODEL_WEIGHTED, r and J are the
 *              weighted r~ and J~, and m counts only the rows with w_i != 0 (m_w), so a problem padded with zero
 *              weights has the covariance of the unpadded one.  With w = 1/sigma, MIR_COV_UNSCALED is scipy's
 *              curve_fit(sigma=..., absolute_sigma=True) and the scaled form is absolute_sigma=False.
 *   Outputs    cov = s^2 A^-1 on F x F; rows and columns of fixed parameters are exactly 0.  Both triangles are written
 *              and are exactly symmetric (the lower triangle is computed and mirrored).  stddev_i = sqrt(cov_ii).
 *              Everything is computed in double and rounded once to T.
 *   info[b]    0   OK, including n_F = 0 (cov all zeros)
 *              k>0 the factorisation broke down at the pivot of parameter k-1 (1-based, original numbering); free block NaN
 *              -1  m <= n_F (m_w <= n_F when weighted) and scaled; free block +inf, as in scipy
 *              -2  a residual, a Jacobian entry or an x_i is not finite; free block NaN
 *              (checked in the order -2, -1, k).
 *
 * Model data as in the batched LM entries: t shared or MIR_MODEL_GRID_PER_PROBLEM, y, aux shared or
 * MIR_MODEL_AUX_PER_PROBLEM, param, w with MIR_MODEL_WEIGHTED, l / u shared (bound_stride == 0) or T[batch*bound_stride],
 * MIR_MODEL_FD_JACOBIAN;
 * MIR_MODEL_WARM_START and MIR_MODEL_NO_TAIL_SHORTCUT are ignored.  settings may be NULL (defaults); only
 * jacobianEpsilon is read.  User models (mir_b200_model_compile) are compiled for the covariance at their first
 * covariance call per precision.
 *   x        T[batch*n]
 *   cov      T[batch*n*n] or NULL;  stddev  T[batch*n] or NULL (not both NULL);  info  int32[batch]
 * Returns MIR_B200_EINVAL for a NULL model, x, l, u or info, cov and stddev both NULL, n == 0 or m == 0, a data model
 * with NULL t / y, or an n the model rejects; MIR_B200_EUNSUPPORTED for n > 128 and for LINEAR2, ROSENBROCK and
 * SQRTCIRCLE.  batch == 0 does nothing.  A problem's output bits depend only on its own inputs (not on the batch size,
 * its position or the run).
 * Host-pointer form: stages the inputs to `device` (-1 = current), runs, copies cov / stddev / info back.  Device form:
 * every pointer (model->t, model->y, model->aux, x, l, u, cov, stddev, info) is a device pointer on the current device;
 * asynchronous on `cuda_stream`.
 */
enum { MIR_COV_UNSCALED = 1u };

int mir_b200_covariance_batched_d(const mir_least_squares_settings_d* settings, const mir_model_desc* model,
    size_t batch, size_t m, size_t n, const double* x, const double* l, const double* u, size_t bound_stride,
    unsigned cov_flags, double* cov, double* stddev, int32_t* info, int device);
int mir_b200_covariance_batched_s(const mir_least_squares_settings_s* settings, const mir_model_desc* model,
    size_t batch, size_t m, size_t n, const float* x, const float* l, const float* u, size_t bound_stride,
    unsigned cov_flags, float* cov, float* stddev, int32_t* info, int device);
int mir_b200_covariance_batched_dev_d(const mir_least_squares_settings_d* settings, const mir_model_desc* model,
    size_t batch, size_t m, size_t n, const double* x, const double* l, const double* u, size_t bound_stride,
    unsigned cov_flags, double* cov, double* stddev, int32_t* info, void* cuda_stream);
int mir_b200_covariance_batched_dev_s(const mir_least_squares_settings_s* settings, const mir_model_desc* model,
    size_t batch, size_t m, size_t n, const float* x, const float* l, const float* u, size_t bound_stride,
    unsigned cov_flags, float* cov, float* stddev, int32_t* info, void* cuda_stream);

/*
 * Batched model prediction at new abscissae and its delta-method standard error (lmfit's eval_uncertainty) from a
 * covariance, normally mir_b200_covariance_batched_*'s output at a fit's x.  The reference has none; this is an
 * extension.  For problem b, with t*_0 .. t*_{k-1} the evaluation abscissae:
 *
 *   Inputs     model->t holds t*: T[k] shared, or T[batch*k] with MIR_MODEL_GRID_PER_PROBLEM.  aux, param,
 *              MIR_MODEL_AUX_PER_PROBLEM and MIR_MODEL_FD_JACOBIAN mean what they mean in the fit.  model->y and model->w
 *              are not read, and MIR_MODEL_WEIGHTED, MIR_MODEL_WARM_START and MIR_MODEL_NO_TAIL_SHORTCUT are ignored: a
 *              prediction is of f, weights describe observations, and the cov passed in already carries the weighting.
 *   Value      value[b*k+i] = f(t*_i; x_b): the model's residual of row i with y_i = 0, so it has the bits the fit's
 *              functor computes.  MIR_MODEL_SPLINE is evaluated with m = k + 1 and param = 0: rows 0..k-1 are
 *              spline(t*_i), and the trailing smoothing row is computed and discarded.  User models see m = k (and
 *              y = 0), so a user model whose residual depends on `row` or `m` gets what it computes for those.
 *   Free set   F = { a : l_a < x_a < u_a }, exactly as in the covariance.  Rows and columns of cov outside F are never read.
 *   Gradient   g_a = d f(t*_i) / d p_a for a in F: the analytic Jacobian row, or the reference's central difference with
 *              settings->jacobianEpsilon and the bound clamp (LS:1030-1047), as in the covariance.
 *   Quadratic  q is computed in double, each step an fma, in this order:
 *   form           q = 0
 *                  for a in F (ascending):  acc = 0
 *                                           for c in F (ascending): acc = fma(C(a,c), g_c, acc)
 *                                           q = fma(g_a, acc, q)
 *              with C(a,c) = cov[b*n*n + max(a,c)*n + min(a,c)]: only the lower triangle is read, in the layout
 *              mir_b200_covariance_batched_* writes.  g and C are converted from T to double.
 *   Output     se[b*k+i] = sqrt(q), rounded once to T; 0 when n_F = 0.  Non-finite inputs propagate through IEEE
 *              arithmetic.  There is no info array: the caller already holds the covariance's info.
 *
 * Usage: a confidence band of the fitted curve is value -/+ t_q * se with t_q a quantile of Student's t with m - n_F
 * degrees of freedom (as lmfit's eval_uncertainty(sigma=...)); a prediction band for a new observation adds the
 * caller's observation variance to se^2 first: sqrt(se^2 + sigma_obs^2).
 *
 *   x        T[batch*n];  l, u  T[n] shared (bound_stride == 0) or T[batch*bound_stride]
 *   cov      T[batch*n*n]; must be non-NULL when se is requested, not read otherwise
 *   value    T[batch*k] or NULL;  se  T[batch*k] or NULL (not both NULL)
 * settings may be NULL (defaults); only jacobianEpsilon is read.  User models (mir_b200_model_compile) are compiled for
 * the prediction at their first prediction call per precision.
 * Returns MIR_B200_EINVAL for a NULL model, x, l or u, value and se both NULL, se without cov, n == 0 or k == 0, a data
 * model with NULL t, a spline with no knots (aux), bound_stride neither 0 nor >= n, an n the model rejects, or an
 * unknown user id; MIR_B200_EUNSUPPORTED for n > 128, k >= 2^31 - 1 and for LINEAR2, ROSENBROCK and SQRTCIRCLE.  The
 * checks run in the covariance's order.  batch == 0 does nothing.  A problem's output bits depend only on its own inputs
 * (not on the batch size, its position or the run).
 * Host-pointer form: stages the inputs to `device` (-1 = current), runs, copies value / se back.  Device form: every
 * pointer (model->t, model->aux, x, l, u, cov, value, se) is a device pointer on the current device; asynchronous on
 * `cuda_stream`.
 */
int mir_b200_predict_batched_d(const mir_least_squares_settings_d* settings, const mir_model_desc* model,
    size_t batch, size_t k, size_t n, const double* x, const double* l, const double* u, size_t bound_stride,
    const double* cov, double* value, double* se, int device);
int mir_b200_predict_batched_s(const mir_least_squares_settings_s* settings, const mir_model_desc* model,
    size_t batch, size_t k, size_t n, const float* x, const float* l, const float* u, size_t bound_stride,
    const float* cov, float* value, float* se, int device);
int mir_b200_predict_batched_dev_d(const mir_least_squares_settings_d* settings, const mir_model_desc* model,
    size_t batch, size_t k, size_t n, const double* x, const double* l, const double* u, size_t bound_stride,
    const double* cov, double* value, double* se, void* cuda_stream);
int mir_b200_predict_batched_dev_s(const mir_least_squares_settings_s* settings, const mir_model_desc* model,
    size_t batch, size_t k, size_t n, const float* x, const float* l, const float* u, size_t bound_stride,
    const float* cov, float* value, float* se, void* cuda_stream);

/*
 * fitSpline (fit_splie.d:26-85): least-squares fit of a C2 cubic spline (mir.interpolate.spline with the default
 * SplineConfiguration: not-a-knot ends) with FIXED knots x[n] to `points` data points; the unknowns are the spline
 * values at the knots, bounded by l[n] <= spline(x) <= u[n]; lambda >= 0 weighs the smoothing term
 * (fit_splie.d:67-80).  Exactly as the reference: start from zeros, finite-difference Jacobian, m = points +
 * (lambda == 0) residual rows, and with lambda != 0 the smoothing row takes the place of the last point's residual.
 *   points_x  T[points] (shared by all curves) or T[batch*points] with MIR_MODEL_GRID_PER_PROBLEM in flags
 *   points_y  T[batch*points]
 *   x         knots, T[n] or T[batch*n] with MIR_MODEL_AUX_PER_PROBLEM
 *   values    T[batch*n] out: the fitted spline values at the knots (the reference returns them inside Spline!T;
 *             its first derivatives follow from them, see mir_b200_spline_eval)
 * Returns MIR_B200_EINVAL (message = the reference's exception text) for points < n with lambda == 0,
 * fit_splie.d:45-49.  Host pointers; every curve is one CTA of the general batched kernel (lm_cta.cuh).
 */
int mir_fit_spline_d(const mir_least_squares_settings_d* settings, size_t points, const double* points_x, const double* points_y,
                     size_t n, const double* x, const double* l, const double* u, double lambda, double* values,
                     mir_least_squares_result_d* result);
int mir_fit_spline_s(const mir_least_squares_settings_s* settings, size_t points, const float* points_x, const float* points_y,
                     size_t n, const float* x, const float* l, const float* u, float lambda, float* values,
                     mir_least_squares_result_s* result);
int mir_fit_spline_batched_d(const mir_least_squares_settings_d* settings, size_t batch, size_t points, const double* points_x,
                             const double* points_y, size_t n, const double* x, const double* l, const double* u, double lambda,
                             unsigned flags, double* values, mir_least_squares_result_d* results, int device);
int mir_fit_spline_batched_s(const mir_least_squares_settings_s* settings, size_t batch, size_t points, const float* points_x,
                             const float* points_y, size_t n, const float* x, const float* l, const float* u, float lambda,
                             unsigned flags, float* values, mir_least_squares_result_s* results, int device);

/*
 * solveBoxQP (BQ:85-102, simple overload; BQ:122-379 full algorithm):
 *   argmin 1/2 x'Px + q'x  s.t.  l <= x <= u,   P n x n row-major, only the lower triangle read.
 * Single problem, host pointers; returns mir_box_qp_status, or -mir_b200_error on failure
 * to reach the device.  settings may be NULL (= BoxQPSettings.init).
 */
int mir_solve_box_qp_d(const mir_box_qp_settings_d* settings, size_t n,
                       const double* P, const double* q, const double* l, const double* u, double* x);
int mir_solve_box_qp_s(const mir_box_qp_settings_s* settings, size_t n,
                       const float* P, const float* q, const float* l, const float* u, float* x);

/* Batched BoxQP: P T[batch*n*n], q/l/u/x T[batch*n], status int32[batch] (mir_box_qp_status).
 * qp_iterations (optional, uint32[batch]) receives the BOXCQP main-loop iteration count. */
int mir_solve_box_qp_batched_d(const mir_box_qp_settings_d* settings, size_t batch, size_t n,
                               const double* P, const double* q, const double* l, const double* u,
                               double* x, int32_t* status, uint32_t* qp_iterations, int device);
int mir_solve_box_qp_batched_s(const mir_box_qp_settings_s* settings, size_t batch, size_t n,
                               const float* P, const float* q, const float* l, const float* u,
                               float* x, int32_t* status, uint32_t* qp_iterations, int device);
int mir_solve_box_qp_batched_dev_d(const mir_box_qp_settings_d* settings, size_t batch, size_t n,
                               const double* P, const double* q, const double* l, const double* u,
                               double* x, int32_t* status, uint32_t* qp_iterations, void* cuda_stream);
int mir_solve_box_qp_batched_dev_s(const mir_box_qp_settings_s* settings, size_t batch, size_t n,
                               const float* P, const float* q, const float* l, const float* u,
                               float* x, int32_t* status, uint32_t* qp_iterations, void* cuda_stream);

/*
 * One large problem, rows sharded over the ranks of an NCCL communicator (one process per
 * GPU).  Each rank passes ITS rows: model->t / model->y are DEVICE pointers to m_local
 * entries.  x (n, host) must be identical on every rank on entry and is on exit.  Every pass
 * does one all-reduce of the packed [lower(J^T J), J^T r, ||r||^2] (n(n+1)/2 + n + 1 doubles)
 * after a fresh/Broyden Jacobian and one 1-double all-reduce of the trial ||r||^2; the n x n
 * BoxQP step and the lambda/convergence control run redundantly (bit-identically) on every rank.
 *   nccl_comm  ncclComm_t, or NULL for a single-GPU run (no collective at all)
 *   stats      optional, host
 */
int mir_optimize_least_squares_sharded_d(
    const mir_least_squares_settings_d* settings, const mir_model_desc* model,
    size_t m_local, size_t n, double* x, const double* l, const double* u,
    void* nccl_comm, void* cuda_stream,
    mir_least_squares_result_d* result, mir_batch_stats* stats);

/* J^T J alone (the FP64-tensor SYRK of the large-problem path; replaces syrk at LS:1065): J is rows x ldj
 * row-major on the device (rows % 32 == 0, ldj even, n <= ldj <= 128); packed receives the lower triangle
 * by rows, n(n+1)/2 doubles (device).  Asynchronous on cuda_stream.  For roofline measurements and tests. */
int mir_b200_syrk_lower_dev_d(const double* J, size_t rows, size_t n, size_t ldj, double* packed, void* cuda_stream);

/* Diagnostics: the device restatements of LAPACK ?posvx(FACT='E', UPLO='L') -- what solveBoxQP calls at BQ:194-205
 * and BQ:310-321 -- on their own, for unit tests against the real LAPACK routine.  A T[batch*n*n] row-major (lower
 * triangle read), b / x T[batch*n], info int32[batch] (0, or k > 0: factorisation broke down at pivot k; LAPACK's
 * info = n+1 "singular to working precision", which BQ:212/323 accepts, is reported as 0), equed int32[batch]
 * (1 = the ?laqsy equilibration was applied).  variant 0: register-resident solver of the batched LM kernels
 * (n <= 8); 1: shared-memory column loop of the CTA-per-QP BoxQP kernel; 2: blocked solver of the large-problem
 * control kernel (both n <= 128); 3: one warp per system (the warp-per-QP BoxQP kernel, n <= 64); 4: one 8-lane
 * group per system (the four-problems-per-warp LM kernel, n <= 8).  Host pointers, synchronous. */
int mir_b200_posvx_batched_d(int variant, size_t batch, size_t n, const double* A, const double* b, double* x,
                             int32_t* info, int32_t* equed, int device);
int mir_b200_posvx_batched_s(int variant, size_t batch, size_t n, const float* A, const float* b, float* x,
                             int32_t* info, int32_t* equed, int device);

/* Diagnostics: the device math under every residual functor and the mux kernel's Cholesky, on its own, for unit tests
 * against the host restatement oracle/repro_math.h (bit for bit) and a high-precision reference.  y[i] = f(x[i]) for
 * i < n.  variant 0: exp_repro_tp (early returns; the large-problem evaluators and user models); 1: exp_repro (out of
 * line); 2: exp_repro_inl; 3 / 4: exp_repro_many<K>, K = 4 / 16, each thread taking K consecutive inputs; 5 / 6:
 * exp_repro_many_conv<K>, K = 4 / 16, each warp taking 32*K consecutive inputs (its fast path runs when all of them have
 * |x| < 700, |x| < 80 in float; past the end of x the warp is padded with 0); 7: mux_sqrt_rcp, sqrt(x) to y and
 * 1/sqrt(x) to y2 (y2 is ignored by the other variants).  Host pointers, synchronous. */
int mir_b200_math_hook_d(int variant, size_t n, const double* x, double* y, double* y2, int device);
int mir_b200_math_hook_s(int variant, size_t n, const float* x, float* y, float* y2, int device);

/* NCCL bootstrap helpers so that a host runtime without NCCL bindings (ctypes, D) can build the
 * communicator: rank 0 calls get_unique_id (128 bytes), shares it by any means, all call init. */
int  mir_b200_nccl_unique_id(void* id128);
int  mir_b200_nccl_comm_init(void** comm, int nranks, const void* id128, int rank);
int  mir_b200_nccl_comm_destroy(void* comm);

#ifdef __cplusplus
}
#endif
#endif /* MIR_OPTIM_B200_H */
