/*
 * models_oracle.cpp -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.
 *
 * Host residual / Jacobian callbacks (the reference's LeastSquaresFunctionBetterC /
 * LeastSquaresJacobianBetterC signatures, LS:78-80) for the built-in models named by
 * mir_model_id, plus an OpenMP driver that runs the oracle LM (lm_oracle.cpp ==
 * LS:877-1176) over a batch of independent problems.  The formulas are written here
 * independently of the CUDA functors (mir_optim_b200/csrc/models.cuh); the first five are the
 * reference's own unit-test problems (LS:217-434).  exp is oracle_math::exp_repro (repro_math.h)
 * and the file is compiled with -ffp-contract=off, so every operation rounds exactly like the
 * device functor's explicitly rounded operation sequence: CPU and GPU see identical residuals.
 */
#include "../include/mir_optim_b200.h"
#include "repro_math.h"

#include <cmath>
#include <cstdlib>
#include <cstring>
#include <vector>
#ifdef _OPENMP
#include <omp.h>
#endif

extern "C" {

/* context handed to the callbacks: one problem's data */
typedef struct oracle_model_ctx {
    int         model;
    const void* t;
    const void* y;
    const void* aux;     /* MIR_MODEL_SPLINE: the knots */
    double      param;   /* MIR_MODEL_SPLINE: lambda    */
} oracle_model_ctx;

}  // extern "C"

namespace {

using oracle_math::exp_repro;

/* ---------------------------------------------------------------------------------------------------------------
 * mir.interpolate.spline as fitSpline uses it (fit_splie.d:52, 61-64, 71-75): Spline!T over the fixed knots x with the
 * default SplineConfiguration -- SplineType.c2 (C2 cubic spline), SplineBoundaryType.notAKnot on both ends.  That module
 * lives in mir-algorithm (>= 3.7.19, dub.sdl:8; not in /root/reference), so this is a restatement of its published
 * algorithm: _computeDerivatives = first derivatives at the knots from the tridiagonal C2 system with not-a-knot end
 * rows; opCall / withTwoDerivatives = SplineKernel's Hermite form (weights w0 = (t - x0)/h, w1 = (x1 - t)/h).  The C2
 * cubic interpolant with not-a-knot ends is unique, so any correct elimination gives mir's slopes up to rounding; the
 * restatement is pinned by the reference's own golden vectors (fit_splie.d:126-137, tests/test_oracle_fit_spline.py)
 * and cross-checked against scipy.interpolate.CubicSpline.
 * ------------------------------------------------------------------------------------------------------------- */
template <class T>
void spline_slopes(size_t n, const T* x, const T* v, T* d, T* work /* 2n */)
{
    if (n == 1) { d[0] = 0; return; }
    if (n == 2) { d[0] = d[1] = (v[1] - v[0]) / (x[1] - x[0]); return; }
    if (n == 3) {                              /* not-a-knot with three knots: the parabola through them */
        const T h0 = x[1] - x[0], h1 = x[2] - x[1], s0 = (v[1] - v[0]) / h0, s1 = (v[2] - v[1]) / h1;
        const T a = (s1 - s0) / (h0 + h1);     /* second divided difference */
        d[0] = s0 - a * h0; d[1] = s0 + a * h0; d[2] = s1 + a * h1;
        return;
    }
    /* tridiagonal system lo_i d_{i-1} + di_i d_i + up_i d_{i+1} = rhs_i, Thomas elimination */
    T* cp = work; T* dp = work + n;            /* modified upper diagonal / right-hand side */
    auto h = [&](size_t i) { return x[i + 1] - x[i]; };
    auto sl = [&](size_t i) { return (v[i + 1] - v[i]) / h(i); };
    {   /* row 0: h1 d0 + (x2 - x0) d1 = ((h0 + 2 (x2 - x0)) h1 s0 + h0^2 s1) / (x2 - x0) */
        const T dd = x[2] - x[0];
        const T di = h(1), up = dd, rhs = ((h(0) + 2 * dd) * h(1) * sl(0) + h(0) * h(0) * sl(1)) / dd;
        cp[0] = up / di; dp[0] = rhs / di;
    }
    for (size_t i = 1; i + 1 < n; ++i) {       /* interior: h_i d_{i-1} + 2 (h_{i-1} + h_i) d_i + h_{i-1} d_{i+1} = 3 (h_i s_{i-1} + h_{i-1} s_i) */
        const T lo = h(i), di = 2 * (h(i - 1) + h(i)), up = h(i - 1), rhs = 3 * (h(i) * sl(i - 1) + h(i - 1) * sl(i));
        const T den = di - lo * cp[i - 1];
        cp[i] = up / den; dp[i] = (rhs - lo * dp[i - 1]) / den;
    }
    {   /* row n-1: (x_{n-1} - x_{n-3}) d_{n-2} + h_{n-3} d_{n-1} = (h_{n-2}^2 s_{n-3} + (2 (x_{n-1} - x_{n-3}) + h_{n-2}) h_{n-3} s_{n-2}) / (x_{n-1} - x_{n-3}) */
        const size_t i = n - 1;
        const T dd = x[n - 1] - x[n - 3];
        const T lo = dd, di = h(n - 3), rhs = (h(n - 2) * h(n - 2) * sl(n - 3) + (2 * dd + h(n - 2)) * h(n - 3) * sl(n - 2)) / dd;
        const T den = di - lo * cp[i - 1];
        d[i] = (rhs - lo * dp[i - 1]) / den;
    }
    for (size_t i = n - 1; i-- > 0;) d[i] = dp[i] - cp[i] * d[i + 1];
}

/* interval of t: the last knot <= t, clamped to [0, n-2] (the end polynomials extrapolate) */
template <class T> size_t spline_interval(size_t n, const T* x, T t)
{
    size_t lo = 0, hi = n;                     /* number of knots <= t by bisection */
    while (lo < hi) { const size_t mid = (lo + hi) / 2; if (x[mid] <= t) lo = mid + 1; else hi = mid; }
    size_t i = lo ? lo - 1 : 0;
    if (i + 2 > n) i = n - 2;
    return i;
}

/* value (out[0]) and first derivative (out[1]) at t: SplineKernel */
template <class T> void spline_eval(size_t n, const T* x, const T* v, const T* d, T t, T* out)
{
    if (n == 1) { out[0] = v[0]; out[1] = 0; return; }
    const size_t i = spline_interval(n, x, t);
    const T step = x[i + 1] - x[i];
    const T w0 = (t - x[i]) / step, w1 = (x[i + 1] - t) / step, wq = w0 * w1;
    const T diff = v[i + 1] - v[i];
    const T z0 = d[i] * step - diff, z1 = d[i + 1] * step - diff;
    const T pr = z0 * w1 - z1 * w0;
    const T pl = v[i] * w1 + v[i + 1] * w0;
    out[0] = pl + wq * pr;
    out[1] = (diff + ((w1 - w0) * pr - wq * (z1 + z0))) / step;
}

/* fitSpline's residual function, fit_splie.d:58-80, d = "a - b".  m = points + (lambda == 0): rows 0 .. points-1 are
 * spline(t_i) - y_i, then row m-1 is OVERWRITTEN with sqrt(integral * lambda * points / (3 n)) -- with lambda != 0 that
 * row is the last point's (the reference's `y[$ - 1] = ...` with y.length == points.length), which we reproduce. */
template <class T>
void spline_residuals(size_t m, size_t n, const T* knots, double lambda_, const T* t, const T* y, const T* p, T* r)
{
    const T lambda = (T)lambda_;
    const size_t points = (lambda != 0) ? m : m - 1;
    std::vector<T> d(n), work(2 * n);
    spline_slopes(n, knots, p, d.data(), work.data());
    T o[2];
    for (size_t i = 0; i < points; ++i) { spline_eval(n, knots, p, d.data(), t[i], o); r[i] = o[0] - y[i]; }
    T integral = 0;
    if (lambda != 0) {
        spline_eval(n, knots, p, d.data(), knots[0], o);
        T ld = o[1];
        for (size_t i = 1; i < n; ++i) {
            spline_eval(n, knots, p, d.data(), knots[i], o);
            const T rd = o[1];
            integral += (rd * rd + rd * ld + ld * ld) * (knots[i] - knots[i - 1]);
            ld = rd;
        }
    }
    r[m - 1] = std::sqrt(integral * lambda * (T)points / (T)(3 * n));
}

template <class T>
void model_f(void* vctx, size_t m, size_t n, const T* p, T* r)
{
    const oracle_model_ctx* c = static_cast<const oracle_model_ctx*>(vctx);
    const T* t = static_cast<const T*>(c->t);
    const T* y = static_cast<const T*>(c->y);
    switch (c->model) {
    case MIR_MODEL_LINEAR2:    r[0] = p[0]; r[1] = 2 - p[1]; break;                        // LS:230-234
    case MIR_MODEL_ROSENBROCK: r[0] = 10 * (p[1] - p[0] * p[0]); r[1] = 1 - p[0]; break;   // LS:261-265
    case MIR_MODEL_SQRTCIRCLE: r[0] = std::sqrt(1 - (p[0] * p[0] + p[1] * p[1])); break;   // LS:427-430
    case MIR_MODEL_EXPDECAY2:                                                               // LS:347, 360
        for (size_t i = 0; i < m; ++i) r[i] = p[0] * exp_repro(-t[i] * p[1]) - y[i];
        break;
    case MIR_MODEL_EXPTAU3:                                                                 // LS:378, 390
        for (size_t i = 0; i < m; ++i) r[i] = p[0] * exp_repro(-t[i] / p[1]) + p[2] - y[i];
        break;
    case MIR_MODEL_EXPDECAY3:
        for (size_t i = 0; i < m; ++i) r[i] = p[0] * exp_repro(-p[1] * t[i]) + p[2] - y[i];
        break;
    case MIR_MODEL_GAUSS4: {
        const T is = 1 / p[2];
        for (size_t i = 0; i < m; ++i) {
            T z = (t[i] - p[1]) * is;
            r[i] = p[0] * exp_repro((T)-0.5 * (z * z)) + p[3] - y[i];
        }
        break; }
    case MIR_MODEL_SUMEXP:
        for (size_t i = 0; i < m; ++i) {
            T acc = 0;
            for (size_t k = 0; k + 1 < n; k += 2) acc += p[k] * exp_repro(-p[k + 1] * t[i]);
            r[i] = acc - y[i];
        }
        break;
    case MIR_MODEL_GAUSSMIX:
        // (rows are independent: the OpenMP loop gives the same bits for any thread count; it only matters for the
        //  single large problem of configs[3], where the CPU baseline is meant to use all host cores)
#pragma omp parallel for schedule(static) if (m >= 65536)
        for (long long i = 0; i < (long long)m; ++i) {
            T acc = p[n - 2] + p[n - 1] * t[i];
            for (size_t k = 0; k + 3 <= n - 2; k += 3) {
                T z = (t[i] - p[k + 1]) * (1 / p[k + 2]);
                acc += p[k] * exp_repro((T)-0.5 * (z * z));
            }
            r[i] = acc - y[i];
        }
        break;
    case MIR_MODEL_SPLINE:
        spline_residuals<T>(m, n, static_cast<const T*>(c->aux), c->param, t, y, p, r);
        break;
    default: for (size_t i = 0; i < m; ++i) r[i] = NAN;
    }
}

template <class T>
void model_g(void* vctx, size_t m, size_t n, const T* p, T* J)
{
    const oracle_model_ctx* c = static_cast<const oracle_model_ctx*>(vctx);
    const T* t = static_cast<const T*>(c->t);
    switch (c->model) {
    case MIR_MODEL_LINEAR2:    J[0] = 1; J[1] = 0; J[2] = 0; J[3] = -1; break;             // LS:235-241
    case MIR_MODEL_ROSENBROCK: J[0] = -20 * p[0]; J[1] = 10; J[2] = -1; J[3] = 0; break;   // LS:295-301
    case MIR_MODEL_SQRTCIRCLE: {
        T s = std::sqrt(1 - (p[0] * p[0] + p[1] * p[1]));
        J[0] = -p[0] / s; J[1] = -p[1] / s; break; }
    case MIR_MODEL_EXPDECAY2:
        for (size_t i = 0; i < m; ++i) {
            T e = exp_repro(-t[i] * p[1]);
            J[i * n + 0] = e; J[i * n + 1] = -(p[0] * t[i]) * e;
        }
        break;
    case MIR_MODEL_EXPTAU3:
        for (size_t i = 0; i < m; ++i) {
            T e = exp_repro(-t[i] / p[1]);
            J[i * n + 0] = e; J[i * n + 1] = ((p[0] * e) * t[i]) / (p[1] * p[1]); J[i * n + 2] = 1;
        }
        break;
    case MIR_MODEL_EXPDECAY3:
        for (size_t i = 0; i < m; ++i) {
            T e = exp_repro(-p[1] * t[i]);
            J[i * n + 0] = e; J[i * n + 1] = -(p[0] * t[i]) * e; J[i * n + 2] = 1;
        }
        break;
    case MIR_MODEL_GAUSS4: {
        const T is = 1 / p[2];
        for (size_t i = 0; i < m; ++i) {
            T z = (t[i] - p[1]) * is;
            T e = exp_repro((T)-0.5 * (z * z));
            T ae = p[0] * e;
            J[i * n + 0] = e;
            J[i * n + 1] = (ae * z) * is;
            J[i * n + 2] = (ae * (z * z)) * is;
            J[i * n + 3] = 1;
        }
        break; }
    case MIR_MODEL_SUMEXP:
        for (size_t i = 0; i < m; ++i)
            for (size_t k = 0; k + 1 < n; k += 2) {
                T e = exp_repro(-p[k + 1] * t[i]);
                J[i * n + k] = e; J[i * n + k + 1] = -(p[k] * t[i]) * e;
            }
        break;
    case MIR_MODEL_GAUSSMIX:
#pragma omp parallel for schedule(static) if (m >= 65536)
        for (long long i = 0; i < (long long)m; ++i) {
            for (size_t k = 0; k + 3 <= n - 2; k += 3) {
                T is = 1 / p[k + 2];
                T z = (t[i] - p[k + 1]) * is;
                T e = exp_repro((T)-0.5 * (z * z));
                T ae = p[k] * e;
                J[i * n + k] = e; J[i * n + k + 1] = (ae * z) * is; J[i * n + k + 2] = (ae * (z * z)) * is;
            }
            J[i * n + n - 2] = 1; J[i * n + n - 1] = t[i];
        }
        break;
    default: for (size_t i = 0; i < m * n; ++i) J[i] = NAN;
    }
}

template <class T> struct API;
template <> struct API<double> {
    using S = mir_least_squares_settings_d; using R = mir_least_squares_result_d; using Sl = mir_slice_d;
    static R run(const S* s, size_t m, size_t n, double* x, const double* l, const double* u, Sl w, mir_slice_i iw,
                 void* ctx, bool fd) {
        return mir_optimize_least_squares_d(s, m, n, x, l, u, w, iw, ctx, model_f<double>, ctx,
                                            fd ? nullptr : model_g<double>, nullptr, nullptr);
    }
};
template <> struct API<float> {
    using S = mir_least_squares_settings_s; using R = mir_least_squares_result_s; using Sl = mir_slice_s;
    static R run(const S* s, size_t m, size_t n, float* x, const float* l, const float* u, Sl w, mir_slice_i iw,
                 void* ctx, bool fd) {
        return mir_optimize_least_squares_s(s, m, n, x, l, u, w, iw, ctx, model_f<float>, ctx,
                                            fd ? nullptr : model_g<float>, nullptr, nullptr);
    }
};

template <class T>
int batched(const typename API<T>::S* settings, const mir_model_desc* model, size_t batch, size_t m, size_t n,
            T* x, const T* l, const T* u, size_t bound_stride, typename API<T>::R* results, int nthreads)
{
    const bool fd = (model->flags & MIR_MODEL_FD_JACOBIAN) != 0;
    const bool per = (model->flags & MIR_MODEL_GRID_PER_PROBLEM) != 0;
    const size_t wl = mir_least_squares_work_length(m, n), iwl = mir_least_squares_iwork_length(m, n);
#ifdef _OPENMP
    if (nthreads <= 0) nthreads = omp_get_max_threads();
#else
    nthreads = 1;
#endif
    if ((size_t)nthreads > batch) nthreads = (int)(batch ? batch : 1);   // one problem: leave the threads to OpenBLAS and the row loops
#pragma omp parallel num_threads(nthreads)
    {
        std::vector<T> work(wl + 8);
        std::vector<mir_lapackint> iwork(iwl + 8);
#pragma omp for schedule(dynamic, 16)
        for (long long b = 0; b < (long long)batch; ++b) {
            oracle_model_ctx ctx;
            ctx.model = (int)model->model;
            ctx.t = model->t ? static_cast<const T*>(model->t) + (per ? (size_t)b * m : 0) : nullptr;
            ctx.y = model->y ? static_cast<const T*>(model->y) + (size_t)b * m : nullptr;
            ctx.aux = model->aux ? static_cast<const T*>(model->aux) + ((model->flags & MIR_MODEL_AUX_PER_PROBLEM) ? (size_t)b * n : 0) : nullptr;
            ctx.param = model->param;
            typename API<T>::Sl w{wl, work.data()};
            mir_slice_i iw{iwl, iwork.data()};
            results[b] = API<T>::run(settings, m, n, x + (size_t)b * n, l + (size_t)b * bound_stride,
                                     u + (size_t)b * bound_stride, w, iw, &ctx, fd);
        }
    }
    return nthreads;
}

}  // namespace

extern "C" {

void oracle_model_f_d(void* c, size_t m, size_t n, const double* x, double* y) { model_f<double>(c, m, n, x, y); }
void oracle_model_g_d(void* c, size_t m, size_t n, const double* x, double* J) { model_g<double>(c, m, n, x, J); }
void oracle_model_f_s(void* c, size_t m, size_t n, const float* x, float* y)   { model_f<float>(c, m, n, x, y); }
void oracle_model_g_s(void* c, size_t m, size_t n, const float* x, float* J)   { model_g<float>(c, m, n, x, J); }

/* The restated exp alone (unit tests: against decimal, and every device form of it bit for bit): y[i] = exp_repro(x[i]). */
void oracle_exp_repro_d(size_t n, const double* x, double* y)
{
#pragma omp parallel for schedule(static) if (n >= 65536)
    for (long long i = 0; i < (long long)n; ++i) y[i] = exp_repro(x[i]);
}
void oracle_exp_repro_s(size_t n, const float* x, float* y)
{
#pragma omp parallel for schedule(static) if (n >= 65536)
    for (long long i = 0; i < (long long)n; ++i) y[i] = exp_repro(x[i]);
}

/* The restated spline alone (unit tests: against scipy's not-a-knot CubicSpline): values and first derivatives at t[0..nt). */
void oracle_spline_eval_d(size_t n, const double* knots, const double* values, size_t nt, const double* t, double* out_v, double* out_d)
{
    std::vector<double> d(n), work(2 * n);
    spline_slopes<double>(n, knots, values, d.data(), work.data());
    for (size_t i = 0; i < nt; ++i) { double o[2]; spline_eval<double>(n, knots, values, d.data(), t[i], o); out_v[i] = o[0]; if (out_d) out_d[i] = o[1]; }
}

/* fitSpline, fit_splie.d:26-85: points (t_i, y_i), knots x, bounds on the spline values, smoothing weight lambda.
 * values (out): the fitted spline values at the knots (the reference starts from zeros, fit_splie.d:55-56, and runs
 * optimize with the finite-difference Jacobian, fit_splie.d:82).  Returns -1 for the reference's exception
 * (points < knots with lambda == 0, fit_splie.d:45-49). */
int oracle_fit_spline_d(const mir_least_squares_settings_d* s, size_t points, const double* pt, const double* py, size_t n,
                        const double* knots, const double* l, const double* u, double lambda, double* values,
                        mir_least_squares_result_d* result)
{
    if (points < n && lambda == 0) return -1;
    const size_t m = points + (lambda == 0 ? 1 : 0);
    std::vector<double> t(m, 0.0), y(m, 0.0);
    for (size_t i = 0; i < points; ++i) { t[i] = pt[i]; y[i] = py[i]; }
    for (size_t i = 0; i < n; ++i) values[i] = 0;
    oracle_model_ctx ctx{MIR_MODEL_SPLINE, t.data(), y.data(), knots, lambda};
    const size_t wl = mir_least_squares_work_length(m, n), iwl = mir_least_squares_iwork_length(m, n);
    std::vector<double> work(wl + 8);
    std::vector<mir_lapackint> iwork(iwl + 8);
    *result = mir_optimize_least_squares_d(s, m, n, values, l, u, mir_slice_d{wl, work.data()}, mir_slice_i{iwl, iwork.data()},
                                           &ctx, model_f<double>, nullptr, nullptr, nullptr, nullptr);
    return 0;
}

/* Run the oracle LM on every problem of a batch (host pointers).  Returns the thread count used. */
int oracle_batched_d(const mir_least_squares_settings_d* s, const mir_model_desc* model, size_t batch, size_t m,
                     size_t n, double* x, const double* l, const double* u, size_t bound_stride,
                     mir_least_squares_result_d* results, int nthreads)
{ return batched<double>(s, model, batch, m, n, x, l, u, bound_stride, results, nthreads); }

int oracle_batched_s(const mir_least_squares_settings_s* s, const mir_model_desc* model, size_t batch, size_t m,
                     size_t n, float* x, const float* l, const float* u, size_t bound_stride,
                     mir_least_squares_result_s* results, int nthreads)
{ return batched<float>(s, model, batch, m, n, x, l, u, bound_stride, results, nthreads); }

int oracle_solve_box_qp_d(const mir_box_qp_settings_d*, size_t, double*, const double*, const double*, const double*, double*, unsigned*);
int oracle_solve_box_qp_s(const mir_box_qp_settings_s*, size_t, float*, const float*, const float*, const float*, float*, unsigned*);

/* Batched BOXCQP (BQ:85-102 per problem).  P is copied per problem because the solver mirrors
 * the lower triangle into the upper one. */
int oracle_box_qp_batched_d(const mir_box_qp_settings_d* s, size_t batch, size_t n, const double* P, const double* q,
                            const double* l, const double* u, double* x, int32_t* status, uint32_t* iters, int nthreads)
{
#ifdef _OPENMP
    if (nthreads <= 0) nthreads = omp_get_max_threads();
#else
    nthreads = 1;
#endif
#pragma omp parallel num_threads(nthreads)
    {
        std::vector<double> Pc(n * n);
#pragma omp for schedule(dynamic, 16)
        for (long long b = 0; b < (long long)batch; ++b) {
            std::memcpy(Pc.data(), P + (size_t)b * n * n, sizeof(double) * n * n);
            unsigned it = 0;
            status[b] = oracle_solve_box_qp_d(s, n, Pc.data(), q + b * n, l + b * n, u + b * n, x + b * n, &it);
            if (iters) iters[b] = it;
        }
    }
    return nthreads;
}
int oracle_box_qp_batched_s(const mir_box_qp_settings_s* s, size_t batch, size_t n, const float* P, const float* q,
                            const float* l, const float* u, float* x, int32_t* status, uint32_t* iters, int nthreads)
{
#ifdef _OPENMP
    if (nthreads <= 0) nthreads = omp_get_max_threads();
#else
    nthreads = 1;
#endif
#pragma omp parallel num_threads(nthreads)
    {
        std::vector<float> Pc(n * n);
#pragma omp for schedule(dynamic, 16)
        for (long long b = 0; b < (long long)batch; ++b) {
            std::memcpy(Pc.data(), P + (size_t)b * n * n, sizeof(float) * n * n);
            unsigned it = 0;
            status[b] = oracle_solve_box_qp_s(s, n, Pc.data(), q + b * n, l + b * n, u + b * n, x + b * n, &it);
            if (iters) iters[b] = it;
        }
    }
    return nthreads;
}

}  // extern "C"
