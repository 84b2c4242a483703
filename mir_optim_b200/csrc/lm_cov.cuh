// lm_cov.cuh -- parameter covariance and standard errors at a given point (normally a fit's output), batched: one CTA
// per problem, any model the general batched LM kernel serves (lm_cta.cuh's CtaFromLarge / CtaSpline / CtaUser, used
// unchanged; behind CtaWeighted in lm_cov_cta_weighted_kernel).  The definition (free set, Jacobian, Jacobi-scaled
// Cholesky inverse, scale, info codes) is stated in include/mir_optim_b200.h next to mir_b200_covariance_batched_{d,s}.
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
    const void* w;          // T[batch*m] observation weights (MIR_MODEL_WEIGHTED) or null
};

template <class T> __device__ __forceinline__ bool cov_finite(T v) { return t_abs(v) < Num<T>::inf(); }

// The kernel, from one body (lm_cov_kernel.inl) under two names: lm_cov_cta_kernel<Model, T, FD> for the models as they
// are, and lm_cov_cta_weighted_kernel<CtaWeighted<M, T>, T, FD> for weighted least squares (MIR_MODEL_WEIGHTED).  The
// second name keeps the set of lm_cov_cta_kernel instantiations the unweighted one (the kernel inventory of
// tests/test_covariance_cpu.py counts it per model); defining the body in place, rather than in a shared inline function,
// keeps the unweighted kernels' code what it was.
#define MIRB200_COV_KERNEL lm_cov_cta_kernel
#include "lm_cov_kernel.inl"
#undef MIRB200_COV_KERNEL
#define MIRB200_COV_KERNEL lm_cov_cta_weighted_kernel
#include "lm_cov_kernel.inl"
#undef MIRB200_COV_KERNEL

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

// the built-in models on lm_cov_cta_kernel (W = false) or lm_cov_cta_weighted_kernel (W = true; lm_cov_w_inst.cu);
// EUNSUPPORTED with the error `unknown` for an id without a model
template <class T, bool W>
int launch_cov_builtin(const mir_model_desc& model, T jacEps, CovArgs ca, const char* unknown, cudaStream_t stream)
{
    return visit_cta_model<T>(model, unknown, [&](auto tag) {
        using M = typename decltype(tag)::type;
        const bool fd = (model.flags & MIR_MODEL_FD_JACOBIAN) || !M::kAnalytic;
        const void* fn;
        if constexpr (W) fn = fd ? (const void*)lm_cov_cta_weighted_kernel<CtaWeighted<M, T>, T, true> : (const void*)lm_cov_cta_weighted_kernel<CtaWeighted<M, T>, T, false>;
        else fn = fd ? (const void*)lm_cov_cta_kernel<M, T, true> : (const void*)lm_cov_cta_kernel<M, T, false>;
        return launch_cov<T>(RuntimeKernel{fn, "lm_cov_cta_kernel launch"}, jacEps, ca, M::prep_elems((int)ca.n), stream);
    });
}

// covariance of the built-in models (lm_cov.cu) and of models compiled at run time (lm_nvrtc.cu).  `ca` is complete
// except for scratch / scratch_stride, which launch_cov fills; the caller has checked the arguments.
template <class T>
int launch_cov_model(const mir_model_desc& model, T jacEps, CovArgs ca, cudaStream_t stream);
template <class T>
int launch_user_cov(const mir_model_desc& model, T jacEps, CovArgs ca, cudaStream_t stream);
#endif

}  // namespace mirb200
