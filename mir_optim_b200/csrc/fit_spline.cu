// fit_spline.cu -- fitSpline (fit_splie.d:26-85) behind the C ABI: one or many curves fitted on the device.
//
// The reference builds a residual delegate around mir.interpolate.spline and hands it to optimize() with no Jacobian
// (finite differences).  Here the residual is the device functor CtaSpline (lm_cta.cuh) and the LM loop is the general
// batched kernel, one CTA per curve; this file only reproduces fitSpline's own set-up: the argument check that throws
// in the reference (fit_splie.d:45-49), m = points + (lambda == 0) residual rows (fit_splie.d:60, 82), the start from
// zeros (fit_splie.d:55-56).
#include <vector>

#include "runtime.cuh"

namespace mirb200 {
template <class T>
int batched_host_entry(const typename Num<T>::Settings* settings, const mir_model_desc* model, size_t batch, size_t m, size_t n,
                       T* x, const T* l, const T* u, size_t bound_stride, typename Num<T>::Result* results,
                       mir_batch_stats* stats, int device);

template <class T>
static int fit_spline(const typename Num<T>::Settings* settings, size_t batch, size_t points, const T* pt, const T* py, size_t n,
                      const T* knots, const T* l, const T* u, T lambda, unsigned flags, T* values, typename Num<T>::Result* results, int device)
{
    clear_error();
    if (!settings || (batch && (!pt || !py || !knots || !l || !u || !values || !results))) { set_error("mir_fit_spline: null argument"); return MIR_B200_EINVAL; }
    if (!(lambda >= (T)0)) { set_error("mir_fit_spline: lambda must be >= 0 (fit_splie.d:36)"); return MIR_B200_EINVAL; }
    if (points < n && lambda == (T)0) {
        set_error("fitSpline: points.length has to be greater or equal x.length when lambda is 0.0");      // fit_splie.d:45-49
        return MIR_B200_EINVAL;
    }
    if (n == 0 || points == 0) { set_error("mir_fit_spline: empty input"); return MIR_B200_EINVAL; }
    if (batch == 0) return MIR_B200_OK;
    const bool per = (flags & MIR_MODEL_GRID_PER_PROBLEM) != 0;
    const size_t m = points + (lambda == (T)0 ? 1 : 0);
    mir_model_desc d{};
    d.model = MIR_MODEL_SPLINE;
    d.flags = MIR_MODEL_FD_JACOBIAN | (flags & (MIR_MODEL_GRID_PER_PROBLEM | MIR_MODEL_AUX_PER_PROBLEM | MIR_MODEL_NO_TAIL_SHORTCUT));
    d.aux = knots; d.param = (double)lambda;
    std::vector<T> tpad, ypad;
    if (m == points) { d.t = pt; d.y = py; }
    else {                                      // one extra (zero) row per curve: arrays with row stride m
        const size_t nt = per ? batch : 1;
        tpad.assign(nt * m, (T)0); ypad.assign(batch * m, (T)0);
        for (size_t b = 0; b < nt; ++b) for (size_t i = 0; i < points; ++i) tpad[b * m + i] = pt[b * points + i];
        for (size_t b = 0; b < batch; ++b) for (size_t i = 0; i < points; ++i) ypad[b * m + i] = py[b * points + i];
        d.t = tpad.data(); d.y = ypad.data();
    }
    for (size_t i = 0; i < batch * n; ++i) values[i] = (T)0;                                                 // fit_splie.d:55-56
    return batched_host_entry<T>(settings, &d, batch, m, n, values, l, u, 0, results, nullptr, device);
}
}  // namespace mirb200

using namespace mirb200;

extern "C" {

int mir_fit_spline_batched_d(const mir_least_squares_settings_d* settings, size_t batch, size_t points, const double* points_x,
                             const double* points_y, size_t n, const double* x, const double* l, const double* u, double lambda,
                             unsigned flags, double* values, mir_least_squares_result_d* results, int device)
{ return fit_spline<double>(settings, batch, points, points_x, points_y, n, x, l, u, lambda, flags, values, results, device); }

int mir_fit_spline_batched_s(const mir_least_squares_settings_s* settings, size_t batch, size_t points, const float* points_x,
                             const float* points_y, size_t n, const float* x, const float* l, const float* u, float lambda,
                             unsigned flags, float* values, mir_least_squares_result_s* results, int device)
{ return fit_spline<float>(settings, batch, points, points_x, points_y, n, x, l, u, lambda, flags, values, results, device); }

int mir_fit_spline_d(const mir_least_squares_settings_d* settings, size_t points, const double* points_x, const double* points_y,
                     size_t n, const double* x, const double* l, const double* u, double lambda, double* values,
                     mir_least_squares_result_d* result)
{ return fit_spline<double>(settings, 1, points, points_x, points_y, n, x, l, u, lambda, 0, values, result, -1); }

int mir_fit_spline_s(const mir_least_squares_settings_s* settings, size_t points, const float* points_x, const float* points_y,
                     size_t n, const float* x, const float* l, const float* u, float lambda, float* values,
                     mir_least_squares_result_s* result)
{ return fit_spline<float>(settings, 1, points, points_x, points_y, n, x, l, u, lambda, 0, values, result, -1); }

}  // extern "C"
