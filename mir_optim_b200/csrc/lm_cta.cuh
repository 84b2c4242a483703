// lm_cta.cuh -- batched Levenberg-Marquardt for ANY model with a run-time number of parameters (n <= 128) and
// residuals: one CTA per problem.  Follows optimizeLeastSquaresImplGeneric!T, least_squares.d:877-1176 (cites inline);
// the box-constrained step is cta_boxqp (boxqp_cta.cuh <- solveBoxQP, boxcqp.d:122-379, LAPACK ?posvx restated).
//
// The specialised batched kernels (lm_tpp: one thread per problem, n <= 4; lm_mux: four problems per warp, n <= 8,
// m <= 128; lm_small: one lane group per problem, compile-time n) cover the BASELINE configs.  This kernel is the general
// path behind the same entry points: the reference accepts any n (least_squares.d:911) and any residual function
// (least_squares.d:78-80), so shapes and models the specialised kernels do not instantiate run here instead of
// returning "unsupported" -- fitSpline's residual (fit_splie.d:58-80, n = number of knots), sums of exponentials or
// Gaussian mixtures with any number of components, and models compiled at run time (NVRTC, lm_nvrtc.cpp).
//
// Samples by TMA: when they fit beside the QP scratch (and m is even: 16-byte granularity), each problem's abscissae and
// observations are staged into shared memory with cp.async.bulk + an mbarrier when the CTA picks the problem up, so the
// 2n evaluations of a finite-difference Jacobian and every trial evaluation read them from shared memory.
//
// Layout.  Persistent CTAs of 128 threads pull problems from an atomic counter.  The n-sized state (x, trial point,
// bounds, step, J^T y, QP bounds) and the QP scratch live in shared memory; J (row-major m x n, LS:154), J^T J and the two
// residual vectors live in a per-CTA global scratch that stays in L1/L2.  Rows are dealt to the threads round-robin;
// every scalar of the LM state is kept by all threads in registers and stays bit-identical (the CTA reductions hand
// every thread the same bits), so control flow is CTA-uniform without a broadcast per branch.
//
// A model is a class with
//     static bool   valid(int n, int m)                       shape check (host and device)
//     static int    prep_elems(int n)                         shared-memory scratch of one prepared parameter vector
//     static void   prepare(pb, p, prep)                      CTA-cooperative set-up for the parameter vector p (ends with a barrier)
//     static T      residual(pb, p, prep, row)                r_row(p)
//     static constexpr bool kAnalytic; static void jacobian_row(pb, p, prep, row, Jrow)   dr_row / dp (row of J)
// (the GPU counterparts of LeastSquaresFunction / LeastSquaresJacobian, least_squares.d:73-80).
#pragma once
#include "boxqp_cta.cuh"
#include "lm_small.cuh"
#include "models_large.cuh"
#ifndef __CUDACC_RTC__
#include "runtime.cuh"
#endif

namespace mirb200 {

constexpr int CTA_NT = 128;

template <class T> struct CtaProblem {
    int m, n;
    const T* t;      // abscissa of this problem (m values) or null
    const T* y;      // observations of this problem (m values) or null
    const T* aux;    // model constants of this problem (n values) or null
    T param;
    const T* w;      // observation weights of this problem (m values) with MIR_MODEL_WEIGHTED, else null
};

struct CtaBatchArgs {
    SmallBatchArgs b;
    const void* aux;        // T[n] or T[batch*n]
    double param;
    void* scratch;          // per CTA: J (m*n) | JJ (n*n) | vec0 (m) | vec1 (m)
    unsigned long long scratch_stride;   // elements per CTA
    unsigned n;
    unsigned stage_m;       // != 0: shared memory holds room for the problem's samples (t, y: 2 * stage_m values) staged by TMA
    const void* w;          // T[batch*m] observation weights (MIR_MODEL_WEIGHTED) or null
};

// ---- TMA bulk copy + mbarrier (as in syrk_dmma.cuh) ------------------------------------------------------------------------
__device__ __forceinline__ unsigned cta_smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void cta_mbar_init(unsigned long long* bar, unsigned count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(cta_smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void cta_mbar_expect_tx(unsigned long long* bar, unsigned bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(cta_smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void cta_mbar_wait(unsigned long long* bar, unsigned parity)
{
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(cta_smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void cta_tma_g2s(void* dst, const void* src, unsigned bytes, unsigned long long* bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(cta_smem_u32(dst)), "l"(src), "r"(bytes), "r"(cta_smem_u32(bar)) : "memory");
}

// ---- deterministic CTA reductions: every thread receives the same bits --------------------------------------------------
template <class T> __device__ __forceinline__ T cta_sum_all(T v, T* red4)
{
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
    __syncthreads();                                   // (red4 may still be read from the previous reduction)
    if ((threadIdx.x & 31) == 0) red4[threadIdx.x >> 5] = v;
    __syncthreads();
    return (red4[0] + red4[1]) + (red4[2] + red4[3]);
}
template <class T> __device__ __forceinline__ T cta_max_all(T v, T* red4)
{
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) v = t_max(v, __shfl_xor_sync(0xffffffffu, v, off));
    __syncthreads();
    if ((threadIdx.x & 31) == 0) red4[threadIdx.x >> 5] = v;
    __syncthreads();
    return t_max(t_max(red4[0], red4[1]), t_max(red4[2], red4[3]));
}
__device__ __forceinline__ bool cta_any_all(bool p) { return __syncthreads_or(p ? 1 : 0) != 0; }

// ---- adapters: the run-time-n functors of the large-problem path (models_large.cuh) as lm_cta models -----------------
template <class L, class T> struct CtaFromLarge {
    static constexpr bool kAnalytic = true;
    __host__ __device__ static bool valid(int n, int) { return L::valid_n(n); }
    __host__ __device__ static int prep_elems(int n) { return n; }
    __device__ static void prepare(const CtaProblem<T>& pb, const T* p, T* prep)
    {
        for (int k = threadIdx.x; k < pb.n; k += CTA_NT) prep[k] = L::aux_of(k, pb.n, p[k]);
        __syncthreads();
    }
    __device__ static T residual(const CtaProblem<T>& pb, const T* p, const T* prep, int row)
    {
        const ParamView<T> pv{p, prep, -1, (T)0, (T)0};
        return L::residual(pv, pb.n, pb.t[row], pb.y[row]);
    }
    __device__ static void jacobian_row(const CtaProblem<T>& pb, const T* p, const T* prep, int row, T* Jrow)
    {
        const ParamView<T> pv{p, prep, -1, (T)0, (T)0};
        const int items = L::jac_items(pb.n);
        for (int it = 0; it < items; ++it) L::jac_item(pv, pb.n, it, pb.t[row], Jrow);
    }
};

// ---- fitSpline's residual (fit_splie.d:58-80): p = values at the knots pb.aux of a C2 cubic spline with not-a-knot ends
// (mir.interpolate.spline with the default SplineConfiguration; restated as in oracle/models_oracle.cpp).  prep = first
// derivatives at the knots (n) | penalty row value (1) | elimination scratch (2n).  Rows 0 .. m-2 are spline(t_i) - y_i
// and row m-1 is sqrt(integral * lambda * points / (3 n)), which with lambda != 0 REPLACES the last point's residual
// (the reference writes y[$ - 1] with y.length == points.length) and with lambda == 0 is an extra zero row.
template <class T> struct CtaSpline {
    static constexpr bool kAnalytic = false;
    __host__ __device__ static bool valid(int n, int m) { return n >= 1 && m >= 1; }
    __host__ __device__ static int prep_elems(int n) { return 3 * n + 2; }
    __device__ static int interval(int n, const T* x, T t)
    {
        int lo = 0, hi = n;
        while (lo < hi) { const int mid = (lo + hi) >> 1; if (x[mid] <= t) lo = mid + 1; else hi = mid; }
        int i = lo ? lo - 1 : 0;
        if (i + 2 > n) i = n - 2;
        return i;
    }
    __device__ static void eval(int n, const T* x, const T* v, const T* d, T t, T& val, T& der)
    {
        if (n == 1) { val = v[0]; der = (T)0; return; }
        const int i = interval(n, x, t);
        const T step = x[i + 1] - x[i];
        const T w0 = div_ni(t - x[i], step), w1 = div_ni(x[i + 1] - t, step), wq = mul_rn(w0, w1);
        const T diff = v[i + 1] - v[i];
        const T z0 = sub_rn(mul_rn(d[i], step), diff), z1 = sub_rn(mul_rn(d[i + 1], step), diff);
        const T pr = sub_rn(mul_rn(z0, w1), mul_rn(z1, w0));
        const T pl = add_rn(mul_rn(v[i], w1), mul_rn(v[i + 1], w0));
        val = add_rn(pl, mul_rn(wq, pr));
        der = div_ni(add_rn(diff, sub_rn(mul_rn(sub_rn(w1, w0), pr), mul_rn(wq, add_rn(z1, z0)))), step);
    }
    __device__ static void prepare(const CtaProblem<T>& pb, const T* v, T* prep)
    {
        const int n = pb.n;
        const T* x = pb.aux;
        T* d = prep; T* cp = prep + n + 1; T* dp = cp + n;
        if (threadIdx.x == 0) {                           // n <= 128: the tridiagonal sweep is a serial chain anyway
            auto h = [&](int i) { return x[i + 1] - x[i]; };
            auto sl = [&](int i) { return div_ni(v[i + 1] - v[i], h(i)); };
            if (n == 1) d[0] = (T)0;
            else if (n == 2) { d[0] = d[1] = sl(0); }
            else if (n == 3) {
                const T h0 = h(0), h1 = h(1), s0 = sl(0), s1 = sl(1);
                const T a = div_ni(s1 - s0, h0 + h1);
                d[0] = sub_rn(s0, mul_rn(a, h0)); d[1] = add_rn(s0, mul_rn(a, h0)); d[2] = add_rn(s1, mul_rn(a, h1));
            } else {
                {
                    const T dd = x[2] - x[0];
                    const T di = h(1), up = dd;
                    const T rhs = div_ni(add_rn(mul_rn(mul_rn(add_rn(h(0), mul_rn((T)2, dd)), h(1)), sl(0)), mul_rn(mul_rn(h(0), h(0)), sl(1))), dd);
                    cp[0] = div_ni(up, di); dp[0] = div_ni(rhs, di);
                }
                for (int i = 1; i + 1 < n; ++i) {
                    const T lo = h(i), di = mul_rn((T)2, add_rn(h(i - 1), h(i))), up = h(i - 1);
                    const T rhs = mul_rn((T)3, add_rn(mul_rn(h(i), sl(i - 1)), mul_rn(h(i - 1), sl(i))));
                    const T den = sub_rn(di, mul_rn(lo, cp[i - 1]));
                    cp[i] = div_ni(up, den); dp[i] = div_ni(sub_rn(rhs, mul_rn(lo, dp[i - 1])), den);
                }
                {
                    const int i = n - 1;
                    const T dd = x[n - 1] - x[n - 3];
                    const T lo = dd, di = h(n - 3);
                    const T rhs = div_ni(add_rn(mul_rn(mul_rn(h(n - 2), h(n - 2)), sl(n - 3)),
                                                mul_rn(mul_rn(add_rn(mul_rn((T)2, dd), h(n - 2)), h(n - 3)), sl(n - 2))), dd);
                    const T den = sub_rn(di, mul_rn(lo, cp[i - 1]));
                    d[i] = div_ni(sub_rn(rhs, mul_rn(lo, dp[i - 1])), den);
                }
                for (int i = n - 2; i >= 0; --i) d[i] = sub_rn(dp[i], mul_rn(cp[i], d[i + 1]));
            }
            // penalty row, fit_splie.d:67-80
            const T lambda = pb.param;
            const int points = (lambda != (T)0) ? pb.m : pb.m - 1;
            T integral = (T)0;
            if (lambda != (T)0) {
                T val, ld, rd;
                eval(n, x, v, d, x[0], val, ld);
                for (int i = 1; i < n; ++i) {
                    eval(n, x, v, d, x[i], val, rd);
                    const T q = add_rn(add_rn(mul_rn(rd, rd), mul_rn(rd, ld)), mul_rn(ld, ld));
                    integral = add_rn(integral, mul_rn(q, x[i] - x[i - 1]));
                    ld = rd;
                }
            }
            d[n] = sqrt_ni(div_ni(mul_rn(mul_rn(integral, lambda), (T)points), (T)(3 * n)));
        }
        __syncthreads();
    }
    __device__ static T residual(const CtaProblem<T>& pb, const T* v, const T* prep, int row)
    {
        if (row == pb.m - 1) return prep[pb.n];
        T val, der;
        eval(pb.n, pb.aux, v, prep, pb.t[row], val, der);
        return sub_rn(val, pb.y[row]);
    }
    __device__ static void jacobian_row(const CtaProblem<T>&, const T*, const T*, int, T*) {}
};

// ---- a model compiled at run time (mir_b200_model_compile, lm_nvrtc.cu): the user's UserModel<REAL> behind the interface
template <class U, class T> struct CtaUser {
    static constexpr bool kAnalytic = U::kAnalytic;
    __host__ __device__ static bool valid(int, int) { return true; }
    __host__ __device__ static int prep_elems(int) { return 1; }
    __device__ static void prepare(const CtaProblem<T>&, const T*, T*) { __syncthreads(); }
    __device__ static T residual(const CtaProblem<T>& pb, const T* p, const T*, int row)
    {
        return U::residual(p, pb.n, pb.m, row, pb.t ? pb.t[row] : (T)0, pb.y ? pb.y[row] : (T)0, pb.aux, pb.param);
    }
    __device__ static void jacobian_row(const CtaProblem<T>& pb, const T* p, const T*, int row, T* Jrow)
    {
        if constexpr (U::kAnalytic) U::jacobian(p, pb.n, pb.m, row, pb.t ? pb.t[row] : (T)0, pb.y ? pb.y[row] : (T)0, pb.aux, pb.param, Jrow);
    }
};

// ---- weighted least squares (MIR_MODEL_WEIGHTED): the model M with every row scaled by its weight, r~_i = w_i r_i and
// J~_ij = w_i J_ij, each rounded once; a finite-difference Jacobian (cta_fd_column) differentiates r~ itself.  The weights
// are read from global memory (pb.w), where the problem's rows stay in L1/L2.
template <class M, class T> struct CtaWeighted {
    static constexpr bool kAnalytic = M::kAnalytic;
    __host__ __device__ static bool valid(int n, int m) { return M::valid(n, m); }
    __host__ __device__ static int prep_elems(int n) { return M::prep_elems(n); }
    __device__ static void prepare(const CtaProblem<T>& pb, const T* p, T* prep) { M::prepare(pb, p, prep); }
    __device__ static T residual(const CtaProblem<T>& pb, const T* p, const T* prep, int row)
    {
        return mul_rn(pb.w[row], M::residual(pb, p, prep, row));
    }
    __device__ static void jacobian_row(const CtaProblem<T>& pb, const T* p, const T* prep, int row, T* Jrow)
    {
        M::jacobian_row(pb, p, prep, row, Jrow);
        const T w = pb.w[row];
        for (int k = 0; k < pb.n; ++k) Jrow[k] = mul_rn(w, Jrow[k]);
    }
};
template <class M> struct CtaIsWeighted { static constexpr bool value = false; };
template <class M, class T> struct CtaIsWeighted<CtaWeighted<M, T>> { static constexpr bool value = true; };

// ---- pieces shared by lm_cta_kernel and lm_cov_cta_kernel (lm_cov.cuh) ----------------------------------------------------
// problem `prob` of a batch: t (m or batch*m, MIR_MODEL_GRID_PER_PROBLEM), y (batch*m), aux (n or batch*n,
// MIR_MODEL_AUX_PER_PROBLEM), w (batch*m, read with MIR_MODEL_WEIGHTED only); null arrays stay null
template <class T>
__device__ __forceinline__ CtaProblem<T> cta_problem(const void* t, const void* y, const void* aux, double param, unsigned flags,
                                                     int m, int n, unsigned long long prob, const void* w)
{
    CtaProblem<T> pb;
    pb.m = m; pb.n = n;
    pb.t = t ? static_cast<const T*>(t) + ((flags & MIR_MODEL_GRID_PER_PROBLEM) ? prob * m : 0) : nullptr;
    pb.y = y ? static_cast<const T*>(y) + prob * m : nullptr;
    pb.aux = aux ? static_cast<const T*>(aux) + ((flags & MIR_MODEL_AUX_PER_PROBLEM) ? prob * n : 0) : nullptr;
    pb.param = (T)param;
    pb.w = (w && (flags & MIR_MODEL_WEIGHTED)) ? static_cast<const T*>(w) + prob * m : nullptr;
    return pb;
}

// Column j of the central-difference Jacobian at x into J (m x n row-major), the step clamped to the bounds, or a zero
// column where the clamped step is empty (LS:1030-1047).  pp (n values) and prep are shared scratch.  Returns whether the
// model was evaluated (twice).
template <class Model, class T>
__device__ __forceinline__ bool cta_fd_column(const CtaProblem<T>& pb, const T* x, const T* lo, const T* up, T* pp, T* prep,
                                              T* J, int j, T eps)
{
    const int tid = threadIdx.x, n = pb.n, m = pb.m;
    const T xmh = t_max(x[j] - eps, lo[j]);                                                         // LS:1030-1033
    const T xph = t_min(x[j] + eps, up[j]);
    const T twh = xph - xmh;
    if (twh != (T)0) {
        const T rt = rcp_ni(twh);
        __syncthreads();
        for (int i = tid; i < n; i += CTA_NT) pp[i] = (i == j) ? xph : x[i];
        __syncthreads();
        Model::prepare(pb, pp, prep);
        for (int r = tid; r < m; r += CTA_NT) J[(size_t)r * n + j] = Model::residual(pb, pp, prep, r);   // f(x + h e_j), parked in its column
        __syncthreads();
        if (tid == 0) pp[j] = xmh;
        __syncthreads();
        Model::prepare(pb, pp, prep);
        for (int r = tid; r < m; r += CTA_NT) {
            const T fm = Model::residual(pb, pp, prep, r);
            J[(size_t)r * n + j] = (J[(size_t)r * n + j] - fm) * rt;                                // LS:1040-1042
        }
        return true;
    }
    for (int r = tid; r < m; r += CTA_NT) J[(size_t)r * n + j] = (T)0;                              // LS:1045-1047
    return false;
}

// (i, j), i >= j, of the packed lower-triangular entry e (tri(i, j) == e)
__device__ __forceinline__ void cta_untri(int e, int& i, int& j)
{
    i = (int)((sqrtf(8.0f * (float)e + 1.0f) - 1.0f) * 0.5f);
    while ((i + 1) * (i + 2) / 2 <= e) ++i;
    while (i * (i + 1) / 2 > e) --i;
    j = e - i * (i + 1) / 2;
}

template <class Model, class T, bool FD>
__global__ void __launch_bounds__(CTA_NT)
lm_cta_kernel(const typename Num<T>::Settings st, const CtaBatchArgs ca)
{
    constexpr int NT = CTA_NT;
    constexpr bool useFD = FD || !Model::kAnalytic;       // no analytic Jacobian: g == null semantics whatever was asked for
    using Result = typename Num<T>::Result;
    const SmallBatchArgs& args = ca.b;
    const int tid = threadIdx.x;
    const int n = (int)ca.n, m = (int)args.m;
    const bool tailShortcut = (args.flags & MIR_MODEL_NO_TAIL_SHORTCUT) == 0;

    extern __shared__ __align__(16) unsigned char cta_smem_raw[];
    T* sp = reinterpret_cast<T*>(cta_smem_raw);
    T* x = sp; sp += n;  T* xt = sp; sp += n;  T* lo = sp; sp += n;  T* up = sp; sp += n;
    T* dX = sp; sp += n; T* Jy = sp; sp += n;  T* qpl = sp; sp += n; T* qpu = sp; sp += n;
    T* pp = sp; sp += n; T* tmp = sp; sp += n;
    T* red4 = sp; sp += 8;
    const int pe = Model::prep_elems(n);
    T* prepA = sp; sp += pe;                      // prepared data of the point being evaluated
    sp += (reinterpret_cast<uintptr_t>(sp) & 8) ? 1 : 0;
    CtaQPScratch<T> qw;
    qw.carve(sp, n);
    __shared__ unsigned int s_idx, s_staged;
    // sample staging area (TMA destination), 16-byte aligned, behind the QP scratch
    __shared__ __align__(8) unsigned long long s_bar;
    const int stageM = (int)ca.stage_m;
    T* const sT = reinterpret_cast<T*>((reinterpret_cast<uintptr_t>(reinterpret_cast<unsigned char*>(sp) + CtaQPScratch<T>::bytes(n)) + 15) & ~(uintptr_t)15);
    T* const sY = sT + stageM;
    unsigned stageParity = 0;
    bool tStaged = false;
    if (stageM) {
        if (tid == 0) cta_mbar_init(&s_bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        __syncthreads();
    }

    T* const scr = static_cast<T*>(ca.scratch) + (size_t)blockIdx.x * ca.scratch_stride;
    T* const J = scr;                             // m x n row-major (LS:154)
    T* const JJ = J + (size_t)m * n;              // n x n, lower triangle valid
    T* const vec0 = JJ + (size_t)n * n;
    T* const vec1 = vec0 + m;

    unsigned long long sPasses = 0, sAccepted = 0, sFresh = 0, sBroyden = 0, sEvals = 0, sSolves = 0, sQPIt = 0, sProblems = 0;

    for (;;) {
        __syncthreads();
        if (tid == 0) {
            const unsigned int idx = atomicAdd(args.counter, 1u);
            s_idx = idx;
            s_staged = (idx < args.batch) ? (wait_staged(args.ready, idx, args.spin_limit) ? 1u : 0u) : 1u;
        }
        __syncthreads();
        const unsigned long long prob = s_idx;
        if (prob >= args.batch) break;
        ++sProblems;
        if (!s_staged) {                          // inputs never arrived: the host discards this launch (flag ready[1])
            if (tid == 0) {
                Result bad;
                bad.status = mir_ls_numericError; bad.iterations = 0; bad.fCalls = 0; bad.gCalls = 0; bad.residual = Num<T>::inf(); bad.lambda = (T)0;
                static_cast<Result*>(args.results)[prob] = bad;
            }
            continue;
        }
        CtaProblem<T> pb = cta_problem<T>(args.t, args.y, ca.aux, ca.param, args.flags, m, n, prob, ca.w);
        if (stageM && pb.y != nullptr && (reinterpret_cast<uintptr_t>(pb.y) & 15) == 0 && (pb.t == nullptr || (reinterpret_cast<uintptr_t>(pb.t) & 15) == 0)) {
            const bool perGrid = (args.flags & MIR_MODEL_GRID_PER_PROBLEM) != 0;
            const bool needT = pb.t != nullptr && (perGrid || !tStaged);
            const unsigned bytes = (unsigned)(m * sizeof(T));
            if (tid == 0) {
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");       // the previous problem's generic reads before the async writes
                cta_mbar_expect_tx(&s_bar, bytes * (needT ? 2u : 1u));
                cta_tma_g2s(sY, pb.y, bytes, &s_bar);
                if (needT) cta_tma_g2s(sT, pb.t, bytes, &s_bar);
            }
            cta_mbar_wait(&s_bar, stageParity);
            stageParity ^= 1u;
            if (pb.t != nullptr) { pb.t = sT; tStaged = true; }
            pb.y = sY;
        }
        T* const xg = static_cast<T*>(args.x) + prob * n;
        for (int i = tid; i < n; i += NT) {
            x[i] = xg[i];
            lo[i] = static_cast<const T*>(args.l)[prob * args.bound_stride + i];
            up[i] = static_cast<const T*>(args.u)[prob * args.bound_stride + i];
        }
        __syncthreads();

        Result ret;
        ret.status = mir_ls_numericError; ret.iterations = 0; ret.fCalls = 0; ret.gCalls = 0; ret.residual = Num<T>::inf(); ret.lambda = (T)0;
        // ---- validation, LS:930-943 (first failure wins)
        {
            bool nonfinite = false, outb = false;
            for (int i = tid; i < n; i += NT) {
                nonfinite = nonfinite || !(-Num<T>::inf() < x[i] && x[i] < Num<T>::inf());
                outb = outb || !((lo[i] <= x[i]) && (x[i] <= up[i]));
            }
            nonfinite = cta_any_all(nonfinite); outb = cta_any_all(outb);
            int vs = 0;
            if (m == 0 || n == 0 || nonfinite) vs = mir_ls_badGuess;
            else if (outb) vs = mir_ls_badBounds;
            else if (!((T)0 <= st.minStepQuality && st.minStepQuality < (T)1)) vs = mir_ls_badMinStepQuality;
            else if (!((T)0 <= st.goodStepQuality && st.goodStepQuality <= (T)1)) vs = mir_ls_badGoodStepQuality;
            else if (!(st.minStepQuality < st.goodStepQuality)) vs = mir_ls_badStepQuality;
            else if (!((T)1 <= st.lambdaIncrease && st.lambdaIncrease <= Num<T>::sqrt_max())) vs = mir_ls_badLambdaParams;
            else if (!(Num<T>::sqrt_min_normal() <= st.lambdaDecrease && st.lambdaDecrease <= (T)1)) vs = mir_ls_badLambdaParams;
            if (vs) {
                ret.status = vs;
                if (tid == 0) static_cast<Result*>(args.results)[prob] = ret;          // x is left untouched
                continue;
            }
        }

        // evaluates f at the n-vector `at` (shared memory) into `out` (global), returns ||f||^2
        auto eval = [&](const T* at, T* out) -> T {
            Model::prepare(pb, at, prepA);
            T part = (T)0;
            for (int r = tid; r < m; r += NT) { const T v = Model::residual(pb, at, prepA, r); out[r] = v; part += v * v; }
            ++sEvals;
            return cta_sum_all(part, red4);
        };

        const unsigned maxAge = st.maxAge ? st.maxAge : (useFD ? 2u * (unsigned)n : 3u);               // LS:945
        T* y = vec0; T* mb = vec1;
        ret.fCalls = 1;
        ret.residual = eval(x, y);                                                                  // LS:953-955
        bool fConverged = ret.residual <= st.maxGoodResidual;                                       // LS:956
        bool needJacobian = true;
        unsigned age = maxAge;
        T lambda = warm_lambda<T>(args, prob), mu = (T)1, deltaX_dot = (T)0;
        ret.status = mir_ls_maxIterations;                                                          // LS:959-971
        bool jjValid = false;

        do {
            ++sPasses;
            if (fConverged) { ret.status = mir_ls_fConverged; break; }                              // LS:974-978
            if (!(lambda <= st.maxLambda)) { ret.status = mir_ls_furtherImprovement; break; }       // LS:979-983
            if (mu > (T)16 && age) { needJacobian = true; age = maxAge; mu = (T)1; }                // LS:984-989
            {
                bool nan = false;
                for (int i = tid; i < n; i += NT) nan = nan || !(x[i] <= x[i]);
                if (cta_any_all(nan)) { ret.status = mir_ls_numericError; break; }                  // LS:990-995
            }
            // the provably inert lambda-overflow tail (lm_small.cuh, tail_is_inert; here only for x strictly inside its bounds)
            if (!needJacobian && age == 0 && tailShortcut && jjValid) {
                T q2p = (T)0, xminp = Num<T>::inf();
                bool notStrict = false;
                for (int i = tid; i < n; i += NT) {
                    q2p += Jy[i] * Jy[i]; xminp = t_min(xminp, t_abs(x[i]));
                    notStrict = notStrict || !((lo[i] < x[i]) && (x[i] < up[i]));
                }
                const T q2 = cta_sum_all(q2p, red4);
                const T xmin = -cta_max_all(-xminp, red4);
                notStrict = cta_any_all(notStrict);
                if (!notStrict && xmin > (T)0 && st.maxStep > (T)0 && sqrt_ni(q2) < lambda * (xmin * (Num<T>::lapack_eps() * (T)0.125))) {
                    for (;;) {                     // replay LS:1112, 1125-1130 and the next pass's LS:979-983
                        ++ret.fCalls;
                        lambda *= st.lambdaIncrease * mu; mu *= (T)2;
                        ++sPasses;
                        if (!(lambda <= st.maxLambda)) break;
                    }
                    ret.status = mir_ls_furtherImprovement; break;
                }
            }
            if (needJacobian) {                                                                     // LS:996-998
                needJacobian = false;
                if (age < maxAge) {                                                                 // Broyden, LS:999-1007
                    ++age; ++sBroyden;
                    const T negd = -rcp_ni(deltaX_dot);
                    for (int r = tid; r < m; r += NT) {              // here y = f_new, mBuffer = f_old (after the swap, LS:1136)
                        T* Jr = J + (size_t)r * n;
                        T acc = (T)0;
                        for (int i = 0; i < n; ++i) acc = fma(Jr[i], dX[i], acc);                   // gemv(1, J, deltaX, 1, mBuffer)
                        const T v = ((mb[r] - y[r]) + acc) * negd;                                  // axpy(-1, y, mBuffer); scal(-d, mBuffer)
                        for (int i = 0; i < n; ++i) Jr[i] = fma(v, dX[i], Jr[i]);                   // ger(1, mBuffer, deltaX, J)
                    }
                } else {
                    age = 0; ++sFresh;                                                              // LS:1010
                    if constexpr (!useFD) {                                                         // LS:1011-1015
                        ++ret.gCalls;
                        Model::prepare(pb, x, prepA);
                        for (int r = tid; r < m; r += NT) Model::jacobian_row(pb, x, prepA, r, J + (size_t)r * n);
                    } else {                                                                        // LS:1018-1049
                        ret.fCalls += (unsigned)n;                                                  // (counts tasks, LS:1049)
                        for (int j = 0; j < n; ++j)
                            if (cta_fd_column<Model, T>(pb, x, lo, up, pp, prepA, J, j, st.jacobianEpsilon)) sEvals += 2;
                    }
                }
                __syncthreads();
                // J^T y (LS:1052) and J^T J (syrk, LS:1065; rebuilt only when J changed): one entry per thread at a time, rows in order
                const int NP = n * (n + 1) / 2;
                for (int e = tid; e < NP + n; e += NT) {
                    if (e < NP) {
                        int i, j; cta_untri(e, i, j);
                        T acc = (T)0;
                        for (int r = 0; r < m; ++r) acc = fma(J[(size_t)r * n + i], J[(size_t)r * n + j], acc);
                        JJ[(size_t)i * n + j] = acc;
                    } else {
                        const int j = e - NP;
                        T acc = (T)0;
                        for (int r = 0; r < m; ++r) acc = fma(J[(size_t)r * n + j], y[r], acc);
                        Jy[j] = acc;
                    }
                }
                jjValid = true;
                __syncthreads();
                // g-test, LS:1053-1062
                T gp = (T)0;
                for (int i = tid; i < n; i += NT) gp = t_max(gp, t_abs(Jy[i]));
                T gsel = cta_max_all(gp, red4);
                if (!(Jy[0] == Jy[0])) gsel = Jy[0];           // BLAS: a NaN wins iamax only as the first element
                if (!(gsel > st.gradTolerance)) {
                    if (age == 0) { ret.status = mir_ls_gConverged; break; }
                    age = maxAge; continue;
                }
            }
            if (!(lambda >= st.minLambda)) {                                                        // LS:1067-1072
                T dp_ = (T)0;
                for (int i = tid; i < n; i += NT) dp_ = t_max(dp_, JJ[(size_t)i * n + i]);
                const T dmax = cta_max_all(dp_, red4);
                lambda = (T)(0.001 * (double)dmax);
                if (!(lambda >= st.minLambda)) lambda = (T)1;
            }
            for (int i = tid; i < n; i += NT) { qpl[i] = lo[i] - x[i]; qpu[i] = up[i] - x[i]; }     // LS:1074-1077
            __syncthreads();
            {
                const T lam = lambda;
                const T* JJc = JJ;
                const int nn = n;
                auto P = [=](int i, int j) -> T { const T v = JJc[(size_t)i * nn + j]; return (i == j) ? v + lam : v; };   // LS:1078-1079
                unsigned qit = 0, qsolves = 0;
                const int qps = cta_boxqp<T, NT, false>(st.qpSettings, n, P, Jy, qpl, qpu, dX, qw, qit, qsolves);         // LS:1080
                sSolves += qsolves; sQPIt += qit;
                __syncthreads();
                bool nan = false;
                for (int i = tid; i < n; i += NT) nan = nan || !(dX[i] <= dX[i]);
                nan = cta_any_all(nan);
                if (qps != mir_qp_solved || nan) { ret.status = mir_ls_numericError; break; }       // LS:1080-1092
            }
            T ndp = (T)0;
            for (int i = tid; i < n; i += NT) { const T d = add_rn(add_rn(dX[i], x[i]), -x[i]); dX[i] = d; ndp += d * d; }   // LS:1096-1099
            const T nd = cta_sum_all(ndp, red4);
            if (!(sqrt_ni(nd) < st.maxStep)) { lambda *= st.lambdaIncrease * mu; mu *= (T)2; continue; }   // LS:1101-1106
            bool differs = false;
            for (int i = tid; i < n; i += NT) {
                const T v = t_max(t_min(add_rn(dX[i], x[i]), up[i]), lo[i]);                        // LS:1108-1110
                xt[i] = v;
                differs = differs || !((v == x[i]) && (signbit(v) == signbit(x[i])));
            }
            differs = cta_any_all(differs);
            ++ret.fCalls;                                                                           // LS:1112
            T trial;
            if (!differs) trial = ret.residual;     // f(xt) == y bit for bit: evaluation skipped, a rejection follows
            else trial = eval(xt, mb);                                                              // LS:1113-1115
            if (!(trial <= Num<T>::inf())) { ret.status = mir_ls_numericError; break; }             // LS:1117-1122
            const T improvement = ret.residual - trial;                                             // LS:1124
            if (!(improvement > (T)0)) { lambda *= st.lambdaIncrease * mu; mu *= (T)2; continue; }  // LS:1125-1130
            needJacobian = true; mu = (T)1; ++ret.iterations; ++sAccepted;                          // LS:1132-1139
            __syncthreads();
            for (int i = tid; i < n; i += NT) x[i] = xt[i];
            { T* sw = y; y = mb; mb = sw; }
            ret.residual = trial;
            fConverged = ret.residual <= st.maxGoodResidual;
            deltaX_dot = nd;
            __syncthreads();
            T pp_ = (T)0, xmaxp = (T)0;
            for (int i = tid; i < n; i += NT) {                                                     // symv(Lower, 1, JJ, deltaX, 2, Jy), LS:1141
                T acc = (T)0;
                for (int j = 0; j < n; ++j) acc = fma((i >= j) ? JJ[(size_t)i * n + j] : JJ[(size_t)j * n + i], dX[j], acc);
                const T v = acc + (T)2 * Jy[i];
                tmp[i] = v;
                pp_ += v * dX[i];
                xmaxp = t_max(xmaxp, t_abs(x[i]));
            }
            const T pred = -cta_sum_all(pp_, red4);                                                 // LS:1142
            for (int i = tid; i < n; i += NT) Jy[i] = tmp[i];                                       // (scratch from here, as in the reference)
            jjValid = false;                            // Jy no longer holds J^T y: the tail test waits for the next Jacobian step
            if (!(pred > (T)0)) { ret.status = mir_ls_furtherImprovement; break; }                  // LS:1144-1148
            const T rho = div_ni(pred, improvement);                                                // LS:1150
            if (rho < st.minStepQuality) { lambda *= st.lambdaIncrease * mu; mu *= (T)2; }          // LS:1152-1156
            else if (rho >= st.goodStepQuality) lambda = t_max(st.lambdaDecrease * lambda * mu, st.minLambda);   // LS:1158-1161
            const T xmax = cta_max_all(xmaxp, red4);                                                // LS:1164 (nrm2, scaled)
            T xn = (T)0;
            if (xmax > (T)0) {
                const T ri = rcp_ni(xmax);
                T ssp = (T)0;
                for (int i = tid; i < n; i += NT) { const T v = x[i] * ri; ssp += v * v; }
                xn = xmax * sqrt_ni(cta_sum_all(ssp, red4));
            }
            const T sd = sqrt_ni(deltaX_dot);
            if (!(sd > st.absTolerance && xn > sd * st.relTolerance)) {                             // LS:1164-1173
                if (age == 0) { ret.status = mir_ls_xConverged; break; }
                age = maxAge; continue;
            }
        } while (ret.iterations < st.maxIterations);                                               // LS:1175

        ret.lambda = lambda;
        __syncthreads();
        for (int i = tid; i < n; i += NT) xg[i] = x[i];
        if (tid == 0) static_cast<Result*>(args.results)[prob] = ret;
    }

    if (args.stats && tid == 0 && sProblems) {
        atomicAdd((unsigned long long*)&args.stats->problems, sProblems);
        atomicAdd((unsigned long long*)&args.stats->passes, sPasses);
        atomicAdd((unsigned long long*)&args.stats->accepted, sAccepted);
        atomicAdd((unsigned long long*)&args.stats->fresh_jacobians, sFresh);
        atomicAdd((unsigned long long*)&args.stats->broyden_updates, sBroyden);
        atomicAdd((unsigned long long*)&args.stats->model_evals, sEvals);
        atomicAdd((unsigned long long*)&args.stats->qp_solves, sSolves);
        atomicAdd((unsigned long long*)&args.stats->qp_iterations, sQPIt);
    }
}

// ---- host side -----------------------------------------------------------------------------------------------------------
#ifndef __CUDACC_RTC__
// The per-CTA scratch (J, J^T J, two residual vectors) is sized by m n: keep the resident wave within a few GB, fewer CTAs
// if need be (they are persistent and pull problems from a queue, so any grid size solves the batch).
inline unsigned long long cta_cap_grid(unsigned long long grid, unsigned long long bytesPerCta)
{
    const unsigned long long budget = 6ull << 30;
    const unsigned long long fit = bytesPerCta ? budget / bytesPerCta : grid;
    if (fit < grid) grid = fit ? fit : 1;
    return grid;
}

// a kernel of this library, for launch_persistent (runtime API); `what` names the launch in its error
struct RuntimeKernel {
    const void* fn; const char* what;
    int set_smem(size_t smem) const { return check_cuda(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem), "cudaFuncSetAttribute"); }
    int occupancy(int* blocks, size_t smem) const { return check_cuda(cudaOccupancyMaxActiveBlocksPerMultiprocessor(blocks, fn, CTA_NT, smem), "cudaOccupancyMaxActiveBlocksPerMultiprocessor"); }
    int launch(unsigned grid, size_t smem, cudaStream_t s, void** params) const
    {
        cudaLaunchKernel(fn, dim3(grid), dim3(CTA_NT), params, smem, s);
        return check_cuda(cudaGetLastError(), what);
    }
};

// Launch policy of the persistent-CTA kernels (lm_cta_kernel, lm_cov_cta_kernel; built in or compiled at run time): up to
// 8 resident CTAs per SM, no more CTAs than problems, and `stride` elements of T of global scratch per CTA, freed in stream
// order behind the kernel; its address goes to `scratch`, a field of the argument struct `params` points to.  `kern` makes
// the calls that differ between the runtime API (RuntimeKernel) and the driver API (lm_nvrtc.cu): set_smem, occupancy
// and launch, each returning MIR_B200_OK or an error code with the error set.
template <class T, class K>
int launch_persistent(const K& kern, size_t smem, const char* tooBig, unsigned long long batch, unsigned long long stride,
                      void*& scratch, void** params, cudaStream_t stream)
{
    if (smem > 220 * 1024) { set_error(tooBig); return MIR_B200_EUNSUPPORTED; }
    if (int rc = kern.set_smem(smem)) return rc;
    int blocksPerSM = 0;
    if (int rc = kern.occupancy(&blocksPerSM, smem)) return rc;
    if (blocksPerSM < 1) blocksPerSM = 1;
    if (blocksPerSM > 8) blocksPerSM = 8;
    unsigned long long grid = (unsigned long long)sm_count() * blocksPerSM;
    if (batch < grid) grid = batch ? batch : 1;
    grid = cta_cap_grid(grid, stride * sizeof(T));
    T* buf = nullptr;
    MIRB200_CUDA(cudaMallocAsync((void**)&buf, sizeof(T) * stride * grid, stream));
    scratch = buf;
    const int rc = kern.launch((unsigned)grid, smem, stream, params);
    count_launch();
    cudaFreeAsync(buf, stream);
    return rc;
}

// lm_cta_kernel (`kern`: built in or compiled at run time) over a batch.  One problem's samples (t and y, m values each) are
// staged in shared memory behind everything else where there is room: m even keeps the TMA copies at 16-byte
// granularity; the budget leaves at least two CTAs per SM for the small shapes this kernel usually sees.
template <class T, class K>
int launch_cta_fit(const K& kern, const typename Num<T>::Settings& st, const SmallBatchArgs& args, const mir_model_desc& model,
                   size_t n, int prepElems, cudaStream_t stream)
{
    const size_t smem = sizeof(T) * (10 * n + 8 + prepElems + 1) + CtaQPScratch<T>::bytes((int)n) + 16;
    const size_t stage = 2 * (size_t)args.m * sizeof(T) + 32;
    const bool staged = args.m > 0 && (args.m * sizeof(T)) % 16 == 0 && stage <= 48 * 1024 && smem + stage <= 200 * 1024;
    CtaBatchArgs ca;
    ca.b = args; ca.aux = model.aux; ca.param = model.param; ca.n = (unsigned)n; ca.stage_m = staged ? args.m : 0u;
    ca.w = (model.flags & MIR_MODEL_WEIGHTED) ? model.w : nullptr;
    ca.scratch_stride = (unsigned long long)args.m * n + (unsigned long long)n * n + 2ull * args.m + 4;
    void* params[] = {(void*)&st, &ca};
    return launch_persistent<T>(kern, staged ? smem + stage : smem, "mir_optim_b200: n too large for the shared memory of the general batched kernel",
                                args.batch, ca.scratch_stride, ca.scratch, params, stream);
}

// The built-in models of the persistent-CTA kernels: f(ModelTag<M>{}) with the lm_cta model M of model.model; EINVAL for a
// spline without its knots, EUNSUPPORTED with the error `unknown` for an id without a model.
template <class T, class F> int visit_cta_model(const mir_model_desc& model, const char* unknown, F&& f)
{
    if (model.model == MIR_MODEL_SPLINE) {
        if (!model.aux) { set_error("mir_optim_b200: MIR_MODEL_SPLINE needs the knots in model->aux"); return MIR_B200_EINVAL; }
        return f(ModelTag<CtaSpline<T>>{});
    }
    return visit_large_model<T>(model.model, [&](auto tag) { return f(ModelTag<CtaFromLarge<typename decltype(tag)::type, T>>{}); },
                                [&] { set_error(unknown); return (int)MIR_B200_EUNSUPPORTED; });
}

// The built-in models on lm_cta_kernel, as they are (W = false) or behind CtaWeighted (W = true; lm_cta_w_inst.cu)
template <class T, bool W>
int launch_cta_builtin(const mir_model_desc& model, size_t n, const typename Num<T>::Settings& st, const SmallBatchArgs& args, cudaStream_t stream)
{
    return visit_cta_model<T>(model, "mir_optim_b200: model id not available in the batched path", [&](auto tag) {
        using M = typename decltype(tag)::type;
        if (n > 128) { set_error("mir_optim_b200: the batched path supports n <= 128"); return (int)MIR_B200_EUNSUPPORTED; }
        if (!M::valid((int)n, (int)args.m)) { set_error("mir_optim_b200: (m, n) not valid for this model"); return (int)MIR_B200_EINVAL; }
        const bool fd = (args.flags & MIR_MODEL_FD_JACOBIAN) || !M::kAnalytic;
        const void* fn;
        if constexpr (W) fn = fd ? (const void*)lm_cta_kernel<CtaWeighted<M, T>, T, true> : (const void*)lm_cta_kernel<CtaWeighted<M, T>, T, false>;
        else fn = fd ? (const void*)lm_cta_kernel<M, T, true> : (const void*)lm_cta_kernel<M, T, false>;
        return launch_cta_fit<T>(RuntimeKernel{fn, "lm_cta_kernel launch"}, st, args, model, n, M::prep_elems((int)n), stream);
    });
}

// general batched path by model id; MIR_B200_EUNSUPPORTED if the model has no run-time-n functor
template <class T>
int launch_cta_model(const mir_model_desc& model, size_t n, const typename Num<T>::Settings& st, const SmallBatchArgs& args, cudaStream_t stream);
// models compiled at run time (lm_nvrtc.cu)
template <class T>
int launch_user_model(const mir_model_desc& model, size_t n, const typename Num<T>::Settings& st, const SmallBatchArgs& args, cudaStream_t stream);
#endif  // !__CUDACC_RTC__

}  // namespace mirb200
