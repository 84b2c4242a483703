// lm_pred.cuh -- batched model prediction at new abscissae and its delta-method standard error from a covariance
// (normally mir_b200_covariance_batched_*'s output at a fit's x): one CTA per problem, any model the general batched LM
// kernel serves (lm_cta.cuh's CtaFromLarge / CtaSpline / CtaUser, used unchanged).  The definition (values, free set,
// gradient, the order of the quadratic form) is stated in include/mir_optim_b200.h next to mir_b200_predict_batched_{d,s}.
//
// Layout.  Persistent CTAs of CTA_NT threads pull problems from an atomic counter.  The k evaluation abscissae are the
// model's rows, with y = 0 read from a zero vector at the head of the per-CTA global scratch; a model with a trailing
// non-observation row (CtaTrailingRow: the spline's smoothing row) runs with m = k + 1 and param = 0 and that row is
// dropped.  Rows are dealt to the threads round-robin.  With se requested, J's free columns at the abscissae (row-major
// m x n, the fit's layout) go to the scratch behind the zero vector -- analytic rows, or cta_fd_column (the reference's
// central difference with the bound clamp, least_squares.d:1030-1047) -- C_FF is staged in shared memory as a packed
// lower triangle of doubles (n <= 128: at most 66 KB), and each thread forms q = g^T C_FF g for its rows in a fixed order.
// So every bit of a problem's output depends on its own inputs only.
#pragma once
#include "lm_cta.cuh"

namespace mirb200 {

struct PredArgs {
    const void* t;          // T[k] or T[batch*k] (MIR_MODEL_GRID_PER_PROBLEM); may be null for user models
    const void* x;          // T[batch*n]
    const void* l;          // T[n] or T[batch*bound_stride]
    const void* u;
    const void* aux;        // T[n] or T[batch*n] (MIR_MODEL_AUX_PER_PROBLEM) or null
    double param;
    const void* cov;        // T[batch*n*n], lower triangle read; null when se is null
    void* value;            // T[batch*k] or null
    void* se;               // T[batch*k] or null
    unsigned int* counter;  // work queue, zero on entry
    void* scratch;          // per CTA: zeros (k + 1) | J ((k + 1) * n, with se)
    unsigned long long scratch_stride;   // elements of T per CTA
    unsigned long long batch;
    unsigned k, n, bound_stride, flags;  // flags: the model's MIR_MODEL_* flags
};

template <class Model, class T, bool FD>
__global__ void __launch_bounds__(CTA_NT)
lm_pred_cta_kernel(const T jacEps, const PredArgs pa)
{
    constexpr int NT = CTA_NT;
    constexpr bool useFD = FD || !Model::kAnalytic;       // no analytic Jacobian: central differences whatever was asked for
    const int tid = threadIdx.x;
    const int n = (int)pa.n, k = (int)pa.k;
    const int m = k + (CtaTrailingRow<Model>::value ? 1 : 0);
    const bool wantSe = pa.se != nullptr;

    extern __shared__ __align__(16) unsigned char pred_smem_raw[];
    double* const Cf = reinterpret_cast<double*>(pred_smem_raw);  // packed lower: C_FF by free position (with se)
    T* const x = reinterpret_cast<T*>(Cf + (wantSe ? n * (n + 1) / 2 : 0));
    T* const lo = x + n; T* const up = lo + n; T* const pp = up + n;
    T* const prep = pp + n;
    int* const fidx = reinterpret_cast<int*>(prep + Model::prep_elems(n));   // free position -> parameter
    __shared__ unsigned int s_idx;
    __shared__ int s_nf;

    T* const zeros = static_cast<T*>(pa.scratch) + (size_t)blockIdx.x * pa.scratch_stride;   // y = 0 for every row
    T* const J = zeros + (size_t)k + 1;                                                      // m x n row-major
    for (int r = tid; r < m; r += NT) zeros[r] = (T)0;

    for (;;) {
        __syncthreads();
        if (tid == 0) s_idx = atomicAdd(pa.counter, 1u);
        __syncthreads();
        const unsigned long long prob = s_idx;
        if (prob >= pa.batch) break;

        CtaProblem<T> pb = cta_problem<T>(pa.t, nullptr, pa.aux, pa.param, pa.flags, k, n, prob, nullptr);   // t: k per problem
        pb.m = m;
        pb.y = zeros;
        if constexpr (CtaTrailingRow<Model>::value) pb.param = (T)0;
        for (int i = tid; i < n; i += NT) {
            x[i] = static_cast<const T*>(pa.x)[prob * n + i];
            lo[i] = static_cast<const T*>(pa.l)[prob * pa.bound_stride + i];
            up[i] = static_cast<const T*>(pa.u)[prob * pa.bound_stride + i];
        }
        __syncthreads();
        if (tid == 0) {                                   // free set F = { i : l_i < x_i < u_i }, in parameter order
            int nf = 0;
            for (int i = 0; i < n; ++i)
                if ((lo[i] < x[i]) && (x[i] < up[i])) fidx[nf++] = i;
            s_nf = nf;
        }
        Model::prepare(pb, x, prep);                      // (ends with a barrier: s_nf and fidx are visible)
        const int nf = s_nf;

        if (pa.value) {
            T* const vg = static_cast<T*>(pa.value) + prob * k;
            for (int r = tid; r < k; r += NT) vg[r] = Model::residual(pb, x, prep, r);
        }
        if (!wantSe) continue;

        // the free columns of J at the abscissae, as the fit's fresh-Jacobian step computes them (lm_cta_kernel, LS:1011-1049)
        if (nf > 0) {
            if constexpr (!useFD) {
                for (int r = tid; r < m; r += NT) Model::jacobian_row(pb, x, prep, r, J + (size_t)r * n);
            } else {
                for (int c = 0; c < nf; ++c) cta_fd_column<Model, T>(pb, x, lo, up, pp, prep, J, fidx[c], jacEps);
            }
        }
        // C_FF from the lower triangle of cov: free positions i >= j are parameters fidx[i] >= fidx[j]
        const T* const cg = static_cast<const T*>(pa.cov) + prob * (unsigned long long)n * n;
        const int NPF = nf * (nf + 1) / 2;
        for (int e = tid; e < NPF; e += NT) {
            int i, j; cta_untri(e, i, j);
            Cf[e] = (double)cg[(size_t)fidx[i] * n + fidx[j]];
        }
        __syncthreads();
        // q = sum_a g_a (sum_c C(a,c) g_c), a and c ascending, every step an fma in double
        T* const sg = static_cast<T*>(pa.se) + prob * k;
        for (int r = tid; r < k; r += NT) {
            const T* const Jr = J + (size_t)r * n;
            double q = 0.0;
            for (int a = 0; a < nf; ++a) {
                const double* const Ca = Cf + tri(a, 0);
                double acc = 0.0;
                for (int c = 0; c <= a; ++c) acc = fma(Ca[c], (double)Jr[fidx[c]], acc);
                for (int c = a + 1; c < nf; ++c) acc = fma(Cf[tri(c, a)], (double)Jr[fidx[c]], acc);
                q = fma((double)Jr[fidx[a]], acc, q);
            }
            sg[r] = (T)sqrt(q);
        }
    }
}

#ifndef __CUDACC_RTC__
// lm_pred_cta_kernel (`kern`: built in or compiled at run time) over pa.batch problems, for a model with `prepElems`
// prepared values
template <class T, class K> int launch_pred(const K& kern, T jacEps, PredArgs pa, int prepElems, cudaStream_t stream)
{
    const size_t n = pa.n, np = pa.se ? n * (n + 1) / 2 : 0;
    const size_t smem = sizeof(double) * np + sizeof(T) * (4 * n + prepElems) + sizeof(int) * n + 16;
    const unsigned long long rows = (unsigned long long)pa.k + 1;
    pa.scratch_stride = rows + (pa.se ? rows * pa.n : 0) + 2;
    void* params[] = {&jacEps, &pa};
    return launch_persistent<T>(kern, smem, "mir_optim_b200: n too large for the shared memory of the prediction kernel", pa.batch,
                                pa.scratch_stride, pa.scratch, params, stream);
}

// prediction of the built-in models (lm_pred.cu) and of models compiled at run time (lm_nvrtc.cu).  `pa` is complete
// except for scratch / scratch_stride, which launch_pred fills; the caller has checked the arguments.
template <class T>
int launch_pred_model(const mir_model_desc& model, T jacEps, PredArgs pa, cudaStream_t stream);
template <class T>
int launch_user_pred(const mir_model_desc& model, T jacEps, PredArgs pa, cudaStream_t stream);
#endif

}  // namespace mirb200
