// lm_cov.cuh -- parameter covariance and standard errors at a given point (normally a fit's output), batched: one CTA
// per problem, any model the general batched LM kernel serves (lm_cta.cuh's CtaFromLarge / CtaSpline / CtaUser, used
// unchanged).  The definition (free set, Jacobian, Jacobi-scaled Cholesky inverse, scale, info codes) is stated in
// include/mir_optim_b200.h next to mir_b200_covariance_batched_{d,s}.
//
// Layout.  Persistent CTAs of CTA_NT threads pull problems from an atomic counter.  Residuals and J (row-major m x n, the
// fit's layout) go to a per-CTA global scratch; rows are dealt to the threads round-robin, and J is evaluated by the
// fresh-Jacobian step of lm_cta_kernel (analytic rows, or cta_fd_column: the reference's central difference with the
// bound clamp of least_squares.d:1030-1047), over the free columns only.  A = J_F^T J_F is built in double, one thread per
// packed entry over the rows in row order; ||r||^2 is a cta_sum_all of per-thread partial sums in row order.  So every
// bit of a problem's output depends on its own inputs only.  The scaled block, its Cholesky factor L, L^-1 and S^-1
// live in shared memory as packed lower triangles (n <= 128: at most 2 x 66 KB).
#pragma once
#include "lm_cta.cuh"

namespace mirb200 {

struct CovArgs {
    const void* t;          // T[m] or T[batch*m] (MIR_MODEL_GRID_PER_PROBLEM); may be null for user models
    const void* y;          // T[batch*m]; may be null for user models
    const void* x;          // T[batch*n]
    const void* l;          // T[n] or T[batch*bound_stride]
    const void* u;
    const void* aux;        // T[n] or T[batch*n] (MIR_MODEL_AUX_PER_PROBLEM) or null
    double param;
    void* cov;              // T[batch*n*n] or null
    void* stddev;           // T[batch*n] or null
    int* info;              // int32[batch]
    unsigned int* counter;  // work queue, zero on entry
    void* scratch;          // per CTA: J (m*n) | r (m)
    unsigned long long scratch_stride;   // elements of T per CTA
    unsigned long long batch;
    unsigned m, n, bound_stride, flags;  // flags: the model's MIR_MODEL_* flags
    unsigned unscaled;      // MIR_COV_UNSCALED: s^2 = 1
};

template <class T> __device__ __forceinline__ bool cov_finite(T v) { return t_abs(v) < Num<T>::inf(); }

template <class Model, class T, bool FD>
__global__ void __launch_bounds__(CTA_NT)
lm_cov_cta_kernel(const T jacEps, const CovArgs ca)
{
    constexpr int NT = CTA_NT;
    constexpr bool useFD = FD || !Model::kAnalytic;       // no analytic Jacobian: central differences whatever was asked for
    const int tid = threadIdx.x;
    const int n = (int)ca.n, m = (int)ca.m;
    const int NP = n * (n + 1) / 2;

    extern __shared__ __align__(16) unsigned char cov_smem_raw[];
    double* const A = reinterpret_cast<double*>(cov_smem_raw);   // packed lower: A, then S, then L, then S^-1
    double* const W = A + NP;                                    // packed lower: L^-1
    double* const sc = W + NP;                                   // D^-1/2 by free position
    double* const red = sc + n;                                  // 8 doubles for cta_sum_all
    T* const x = reinterpret_cast<T*>(red + 8);
    T* const lo = x + n; T* const up = lo + n; T* const pp = up + n;
    T* const prep = pp + n;
    const int pe = Model::prep_elems(n);
    int* const fidx = reinterpret_cast<int*>(prep + pe);         // free position -> parameter
    int* const fpos = fidx + n;                                  // parameter -> free position, or -1
    __shared__ unsigned int s_idx;
    __shared__ int s_nf;

    T* const J = static_cast<T*>(ca.scratch) + (size_t)blockIdx.x * ca.scratch_stride;   // m x n row-major
    T* const rv = J + (size_t)m * n;

    for (;;) {
        __syncthreads();
        if (tid == 0) s_idx = atomicAdd(ca.counter, 1u);
        __syncthreads();
        const unsigned long long prob = s_idx;
        if (prob >= ca.batch) break;

        const CtaProblem<T> pb = cta_problem<T>(ca.t, ca.y, ca.aux, ca.param, ca.flags, m, n, prob);
        bool bad = false;
        for (int i = tid; i < n; i += NT) {
            const T v = static_cast<const T*>(ca.x)[prob * n + i];
            x[i] = v;
            lo[i] = static_cast<const T*>(ca.l)[prob * ca.bound_stride + i];
            up[i] = static_cast<const T*>(ca.u)[prob * ca.bound_stride + i];
            bad = bad || !cov_finite(v);
        }
        __syncthreads();
        if (tid == 0) {                                   // free set F = { i : l_i < x_i < u_i }, in parameter order
            int nf = 0;
            for (int i = 0; i < n; ++i) {
                const bool fr = (lo[i] < x[i]) && (x[i] < up[i]);
                fpos[i] = fr ? nf : -1;
                if (fr) fidx[nf++] = i;
            }
            s_nf = nf;
        }
        bad = cta_any_all(bad);                           // (a barrier: s_nf, fpos, fidx are visible)
        const int nf = s_nf;
        int info = 0;
        double s2 = 1.0;

        if (bad) {
            info = -2;
        } else {
            // residuals at x and ||r||^2 in double
            Model::prepare(pb, x, prep);
            double part = 0.0;
            for (int r = tid; r < m; r += NT) {
                const T v = Model::residual(pb, x, prep, r);
                rv[r] = v;
                part = fma((double)v, (double)v, part);
                bad = bad || !cov_finite(v);
            }
            const double rr = cta_sum_all(part, red);
            // the free columns of J, as the fit's fresh-Jacobian step computes them (lm_cta_kernel, LS:1011-1049)
            if (nf > 0) {
                if constexpr (!useFD) {
                    for (int r = tid; r < m; r += NT) Model::jacobian_row(pb, x, prep, r, J + (size_t)r * n);
                } else {
                    for (int k = 0; k < nf; ++k) cta_fd_column<Model, T>(pb, x, lo, up, pp, prep, J, fidx[k], jacEps);
                }
                for (int r = tid; r < m; r += NT)
                    for (int k = 0; k < nf; ++k) bad = bad || !cov_finite(J[(size_t)r * n + fidx[k]]);
            }
            bad = cta_any_all(bad);
            if (bad) info = -2;
            else if (!ca.unscaled && m <= nf) info = -1;
            else {
                if (!ca.unscaled) s2 = rr / (double)(m - nf);
                const int NPF = nf * (nf + 1) / 2;
                // A = J_F^T J_F: one thread per entry, rows in order
                for (int e = tid; e < NPF; e += NT) {
                    int i, j; cta_untri(e, i, j);
                    const T* Ji = J + fidx[i];
                    const T* Jj = J + fidx[j];
                    double acc = 0.0;
                    for (int r = 0; r < m; ++r) acc = fma((double)Ji[(size_t)r * n], (double)Jj[(size_t)r * n], acc);
                    A[e] = acc;
                }
                __syncthreads();
                // S = D^-1/2 A D^-1/2; a zero diagonal gives a zero row and column, so its pivot stops the factorisation
                for (int i = tid; i < nf; i += NT) { const double d = A[tri(i, i)]; sc[i] = d > 0.0 ? 1.0 / sqrt(d) : 0.0; }
                __syncthreads();
                for (int e = tid; e < NPF; e += NT) { int i, j; cta_untri(e, i, j); A[e] = (A[e] * sc[i]) * sc[j]; }
                __syncthreads();
                // S = L L^T, column by column (LAPACK ?potf2, lower)
                int fail = -1;
                for (int j = 0; j < nf; ++j) {
                    const double d = A[tri(j, j)];
                    if (!(d > 0.0)) { fail = j; break; }                     // (the same shared value on every thread)
                    const double ljj = sqrt(d), rl = 1.0 / ljj;
                    __syncthreads();
                    if (tid == 0) A[tri(j, j)] = ljj;
                    for (int i = j + 1 + tid; i < nf; i += NT) A[tri(i, j)] *= rl;
                    __syncthreads();
                    const int tr = nf - j - 1;
                    for (int e = tid; e < tr * (tr + 1) / 2; e += NT) {      // trailing update, each entry once per column
                        int i, k; cta_untri(e, i, k);
                        i += j + 1; k += j + 1;
                        A[tri(i, k)] = fma(-A[tri(i, j)], A[tri(k, j)], A[tri(i, k)]);
                    }
                    __syncthreads();
                }
                if (fail >= 0) {
                    info = fidx[fail] + 1;
                } else {
                    // W = L^-1 (?trtri): thread j forms column j
                    for (int j = tid; j < nf; j += NT) {
                        W[tri(j, j)] = 1.0 / A[tri(j, j)];
                        for (int i = j + 1; i < nf; ++i) {
                            double acc = 0.0;
                            for (int k = j; k < i; ++k) acc = fma(A[tri(i, k)], W[tri(k, j)], acc);
                            W[tri(i, j)] = -acc / A[tri(i, i)];
                        }
                    }
                    __syncthreads();
                    // S^-1 = W^T W (?lauum), lower triangle, into A
                    for (int e = tid; e < NPF; e += NT) {
                        int i, j; cta_untri(e, i, j);
                        double acc = 0.0;
                        for (int k = i; k < nf; ++k) acc = fma(W[tri(k, i)], W[tri(k, j)], acc);
                        A[e] = acc;
                    }
                    __syncthreads();
                }
            }
        }

        // outputs: cov = s^2 D^-1/2 S^-1 D^-1/2 on F x F (lower triangle computed, mirrored), zero elsewhere
        const double fill = info == -1 ? (double)Num<T>::inf() : (info != 0 ? __longlong_as_double(0x7ff8000000000000LL) : 0.0);
        auto cov_at = [&](int pi, int pj) -> double {
            if (info != 0) return fill;
            const int hi = pi > pj ? pi : pj, lw = pi > pj ? pj : pi;
            return ((A[tri(hi, lw)] * sc[hi]) * sc[lw]) * s2;
        };
        if (ca.cov) {
            T* const cg = static_cast<T*>(ca.cov) + prob * (unsigned long long)n * n;
            for (int e = tid; e < n * n; e += NT) {
                const int i = e / n, j = e - i * n;
                const int pi = fpos[i], pj = fpos[j];
                cg[e] = (pi >= 0 && pj >= 0) ? (T)cov_at(pi, pj) : (T)0;
            }
        }
        if (ca.stddev) {
            T* const sg = static_cast<T*>(ca.stddev) + prob * n;
            for (int i = tid; i < n; i += NT) {
                const int pi = fpos[i];
                sg[i] = pi >= 0 ? (T)sqrt(cov_at(pi, pi)) : (T)0;
            }
        }
        if (tid == 0) ca.info[prob] = info;
    }
}

#ifndef __CUDACC_RTC__
// lm_cov_cta_kernel (`kern`: built in or compiled at run time) over ca.batch problems, for a model with `prepElems`
// prepared values
template <class T, class K> int launch_cov(const K& kern, T jacEps, CovArgs ca, int prepElems, cudaStream_t stream)
{
    const size_t n = ca.n, np = n * (n + 1) / 2;
    const size_t smem = sizeof(double) * (2 * np + n + 8) + sizeof(T) * (4 * n + prepElems) + sizeof(int) * 2 * n + 16;
    ca.scratch_stride = (unsigned long long)ca.m * ca.n + ca.m + 2;
    void* params[] = {&jacEps, &ca};
    return launch_persistent<T>(kern, smem, "mir_optim_b200: n too large for the shared memory of the covariance kernel", ca.batch,
                                ca.scratch_stride, ca.scratch, params, stream);
}

// covariance of the built-in models (lm_cov.cu) and of models compiled at run time (lm_nvrtc.cu).  `ca` is complete
// except for scratch / scratch_stride, which launch_cov fills; the caller has checked the arguments.
template <class T>
int launch_cov_model(const mir_model_desc& model, T jacEps, CovArgs ca, cudaStream_t stream);
template <class T>
int launch_user_cov(const mir_model_desc& model, T jacEps, CovArgs ca, cudaStream_t stream);
#endif

}  // namespace mirb200
