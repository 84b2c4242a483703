// lm_large.cu -- host side of the single-large-problem LM engine and the C ABI built on it:
//   mir_optimize_least_squares_sharded_d      rows sharded over the ranks of an NCCL communicator
//   mir_optimize_least_squares_{d,s}          the reference's own entry points (least_squares.d:705-748)
//   mir_b200_syrk_lower_dev_d                 the J^T J kernel alone (roofline measurements)
// Kernels: lm_large.cuh, syrk_dmma.cuh.  No CPU fallback anywhere: without a device every entry
// point reports an error (legacy entries: status numericError + mir_b200_last_error()).
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <mutex>
#include <string>
#include <vector>

#include "lm_large.cuh"
#include "nccl_dl.h"
#include "runtime.cuh"

namespace mirb200 {

// batched small-problem path (lm_batched.cu), used by the legacy entry for shapes it covers
template <class T>
int batched_host_entry(const typename Num<T>::Settings* settings, const mir_model_desc* model, size_t batch, size_t m, size_t n,
                       T* x, const T* l, const T* u, size_t bound_stride, typename Num<T>::Result* results,
                       mir_batch_stats* stats, int device);

// ---------------------------------------------------------------------------------------------
// CUDA-core J^T J for float (the FP64 tensor kernel is double only).  Same partial-image format.
// 256 threads = 16 x 16 grid of 8 x 8 sub-blocks, lower blocks only.
// ---------------------------------------------------------------------------------------------
template <class T>
__global__ void __launch_bounds__(256) syrk_simple_kernel(const T* __restrict__ J, long long rows, int ldj, T* __restrict__ partial,
                                                          const int* gate, const int* done)
{
    if (*done || *gate == 0) return;
    __shared__ T tile[LARGE_TILE][SYRK_NPAD + 4];
    const int tid = threadIdx.x, ti = tid >> 4, tj = tid & 15;
    T acc[8][8];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = (T)0;
    for (int e = tid; e < LARGE_TILE * (SYRK_NPAD + 4); e += 256) (&tile[0][0])[e] = (T)0;
    const long long tiles = (rows + LARGE_TILE - 1) / LARGE_TILE;
    const long long per = (tiles + gridDim.x - 1) / gridDim.x;
    const long long t0 = (long long)blockIdx.x * per, t1 = (t0 + per < tiles) ? t0 + per : tiles;
    for (long long tl = t0; tl < t1; ++tl) {
        __syncthreads();
        for (int e = tid; e < LARGE_TILE * ldj; e += 256) {
            const int r = e / ldj, k = e - r * ldj;
            const long long row = tl * LARGE_TILE + r;
            tile[r][k] = row < rows ? J[(size_t)row * ldj + k] : (T)0;
        }
        __syncthreads();
        if (tj <= ti && tj * 8 < ldj) {
#pragma unroll 4
            for (int r = 0; r < LARGE_TILE; ++r) {
                T a[8], b[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) { a[i] = tile[r][8 * ti + i]; b[i] = tile[r][8 * tj + i]; }
#pragma unroll
                for (int i = 0; i < 8; ++i)
#pragma unroll
                    for (int j = 0; j < 8; ++j) acc[i][j] += a[i] * b[j];
            }
        }
    }
    T* out = partial + (size_t)blockIdx.x * (SYRK_NPAD * SYRK_NPAD);
    if (tj <= ti) {
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
            for (int j = 0; j < 8; ++j) out[(size_t)(8 * ti + i) * SYRK_NPAD + 8 * tj + j] = acc[i][j];
    }
}

template <class T>
__global__ void __launch_bounds__(256) syrk_reduce_kernel_t(const T* __restrict__ partial, int nparts, int n, T* __restrict__ packed,
                                                            const int* gate, const int* done)
{
    if (*done || *gate == 0) return;
    const int np = n * (n + 1) / 2;
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < np; e += gridDim.x * blockDim.x) {
        int i = (int)((sqrt(8.0 * e + 1.0) - 1.0) * 0.5);
        while (i * (i + 1) / 2 > e) --i;
        while ((i + 1) * (i + 2) / 2 <= e) ++i;
        const int j = e - i * (i + 1) / 2;
        const T* p = partial + (size_t)i * SYRK_NPAD + j;
        T s = (T)0;
        for (int c = 0; c < nparts; ++c) s += p[(size_t)c * (SYRK_NPAD * SYRK_NPAD)];
        packed[e] = s;
    }
}

// ---------------------------------------------------------------------------------------------
// model dispatch
// ---------------------------------------------------------------------------------------------
template <class T> struct LargeKernels {
    void (*eval)(const EvalArgs<T>);
    void (*jac)(const JacArgs<T>);
    void (*jacfd)(const JacArgs<T>);
    bool (*valid_n)(int);
};
template <class Model, class T> LargeKernels<T> kernels_of()
{
    return {large_eval_kernel<Model, T>, large_jac_kernel<Model, T, false>, large_jac_kernel<Model, T, true>, &Model::valid_n};
}
template <class T> bool large_model_kernels(unsigned model, LargeKernels<T>& k)
{
    return visit_large_model<T>(model, [&](auto tag) { k = kernels_of<typename decltype(tag)::type, T>(); return true; },
                                [] { return false; });
}

// argument validation, least_squares.d:930-943 (first failure wins).  Returns 0 when valid.
template <class T>
static int validate_args(const typename Num<T>::Settings& st, bool haveRows, size_t n, const T* x, const T* l, const T* u)
{
    bool finite = true, inb = true;
    for (size_t i = 0; i < n; ++i) {
        finite = finite && (-Num<T>::inf() < x[i] && x[i] < Num<T>::inf());
        inb = inb && (l[i] <= x[i]) && (x[i] <= u[i]);
    }
    if (!haveRows || n == 0 || !finite) return mir_ls_badGuess;
    if (!inb) return mir_ls_badBounds;
    if (!((T)0 <= st.minStepQuality && st.minStepQuality < (T)1)) return mir_ls_badMinStepQuality;
    if (!((T)0 <= st.goodStepQuality && st.goodStepQuality <= (T)1)) return mir_ls_badGoodStepQuality;
    if (!(st.minStepQuality < st.goodStepQuality)) return mir_ls_badStepQuality;
    if (!((T)1 <= st.lambdaIncrease && st.lambdaIncrease <= Num<T>::sqrt_max())) return mir_ls_badLambdaParams;
    if (!(Num<T>::sqrt_min_normal() <= st.lambdaDecrease && st.lambdaDecrease <= (T)1)) return mir_ls_badLambdaParams;
    return 0;
}

// Host callbacks of the reference's C API (least_squares.d:78-80, 672-678)
template <class T> struct HostCallbacks {
    void* fCtx = nullptr; void (*f)(void*, size_t, size_t, const T*, T*) = nullptr;
    void* gCtx = nullptr; void (*g)(void*, size_t, size_t, const T*, T*) = nullptr;
    void* tmCtx = nullptr; mir_ls_thread_manager tm = nullptr;
};

// one finite-difference column, least_squares.d:1022-1047 (run through the user's thread manager when given)
template <class T> struct FDTaskCtx {
    const HostCallbacks<T>* cb; size_t m, n; const T* x; const T* l; const T* u; T eps; T* J; size_t ldj;
};
template <class T> static void fd_task(mir_ls_task task, unsigned, unsigned, unsigned j)
{
    const FDTaskCtx<T>& c = *static_cast<const FDTaskCtx<T>*>(task.context);
    std::vector<T> p(c.x, c.x + c.n), fp(c.m), fm(c.m);          // private scratch per task (the reference shares mBuffer, a latent race)
    const T save = p[j];
    const T xmh = std::fmax(save - c.eps, c.l[j]);
    const T xph = std::fmin(save + c.eps, c.u[j]);
    const T twh = xph - xmh;
    if (twh != 0) {
        p[j] = xph; c.cb->f(c.cb->fCtx, c.m, c.n, p.data(), fp.data());
        p[j] = xmh; c.cb->f(c.cb->fCtx, c.m, c.n, p.data(), fm.data());
        const T rt = 1 / twh;
        for (size_t i = 0; i < c.m; ++i) c.J[i * c.ldj + j] = (fp[i] - fm[i]) * rt;
    } else {
        for (size_t i = 0; i < c.m; ++i) c.J[i * c.ldj + j] = 0;
    }
}

// ---------------------------------------------------------------------------------------------
// the engine
// ---------------------------------------------------------------------------------------------
template <class T>
static int large_solve(const typename Num<T>::Settings& st, unsigned model, unsigned modelFlags, long long rows, size_t n_,
                       const T* d_t, const T* d_yobs, const HostCallbacks<T>* cb,
                       T* x, const T* l, const T* u, void* comm, cudaStream_t stream,
                       typename Num<T>::Result* result, mir_batch_stats* stats)
{
    using Ctl = LargeCtl<T>;
    constexpr bool kDouble = std::is_same<T, double>::value;
    const bool fdJacobian = (modelFlags & MIR_MODEL_FD_JACOBIAN) != 0;
    result->status = mir_ls_numericError; result->iterations = 0; result->fCalls = 0; result->gCalls = 0;
    result->residual = Num<T>::inf(); result->lambda = 0;
    if (stats) std::memset(stats, 0, sizeof *stats);

    const int vs = validate_args<T>(st, rows > 0 || comm != nullptr, n_, x, l, u);
    if (vs) { result->status = vs; return MIR_B200_OK; }
    if (n_ > (size_t)LARGE_NMAX) {
        set_error("mir_optim_b200: the single-problem GPU path supports n <= 128 parameters");
        return MIR_B200_EUNSUPPORTED;
    }
    const int n = (int)n_;
    LargeKernels<T> K{};
    if (!cb) {
        if (!large_model_kernels<T>(model, K)) { set_error("mir_optim_b200: model id not available in the single-problem path"); return MIR_B200_EUNSUPPORTED; }
        if (!K.valid_n(n)) { set_error("mir_optim_b200: n does not match the model"); return MIR_B200_EINVAL; }
    }
    int rc = require_device(-1);
    if (rc) return rc;
    if (comm && (rc = nccl_available())) return rc;

    // All work runs on an internal stream ordered after the caller's stream: the pass loop is replayed as a CUDA graph,
    // and the legacy default stream (what a caller may well hand in) cannot be captured.  The call is blocking anyway.
    struct WorkStream {
        cudaStream_t s = nullptr; cudaEvent_t e = nullptr;
        ~WorkStream() { if (e) cudaEventDestroy(e); if (s) cudaStreamDestroy(s); }
    } work;
    MIRB200_CUDA(cudaStreamCreateWithFlags(&work.s, cudaStreamNonBlocking));
    MIRB200_CUDA(cudaEventCreateWithFlags(&work.e, cudaEventDisableTiming));
    MIRB200_CUDA(cudaEventRecord(work.e, stream));
    MIRB200_CUDA(cudaStreamWaitEvent(work.s, work.e, 0));
    stream = work.s;

    // double: the Broyden update runs inside the SYRK ring (syrk_dmma.cuh); float keeps the separate kernel
    const bool fuseBroyden = kDouble;
    static const bool trace = [] { const char* e = std::getenv("MIRB200_TRACE"); return e && *e == '1'; }();
    const auto tr0 = std::chrono::steady_clock::now();
    auto TR = [&](const char* what) { if (trace) { cudaStreamSynchronize(stream); fprintf(stderr, "[trace] %-28s %8.3f ms\n", what, std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - tr0).count()); } };
    const int ldj = (n + 1) & ~1;
    const long long rowsPad = (rows + SYRK_KT - 1) / SYRK_KT * SYRK_KT;
    const int sms = sm_count();
    const bool hasG = cb ? (cb->g != nullptr) : !fdJacobian;
    const int np = n * (n + 1) / 2;

    auto clampGrid = [](long long want, long long cap) { long long g = want < cap ? want : cap; return (unsigned)(g < 1 ? 1 : g); };
    const unsigned gridEval = clampGrid((rows + 255) / 256, (long long)sms * 4);
    const unsigned gridJac = clampGrid((rows + LARGE_TILE - 1) / LARGE_TILE, (long long)sms * 4);
    const unsigned gridBro = clampGrid((rows + 7) / 8, (long long)sms * 8);
    const unsigned gridSyrk = clampGrid(rowsPad / SYRK_KT, kDouble ? sms : (long long)sms * 2);
    const unsigned gridJyMax = gridJac > gridBro ? gridJac : gridBro;

    // ---- device memory (stream ordered) ----
    auto align = [](size_t v) { return (v + 255) & ~(size_t)255; };
    const size_t bCtl = align(sizeof(Ctl)), bJ = align(sizeof(T) * (size_t)rowsPad * ldj), bV = align(sizeof(T) * (size_t)(rows > 0 ? rows : 1));
    const size_t bRR = align(sizeof(T) * gridEval), bJy = align(sizeof(T) * (size_t)gridJyMax * LARGE_NMAX);
    const size_t bPart = align(sizeof(T) * (size_t)gridSyrk * SYRK_NPAD * SYRK_NPAD);
    char* base = nullptr;
    MIRB200_CUDA(cudaMallocAsync((void**)&base, bCtl + bJ + 2 * bV + bRR + bJy + bPart, stream));
    struct Free { char* p; cudaStream_t s; ~Free() { cudaFreeAsync(p, s); } } freer{base, stream};
    char* p = base;
    Ctl* d_ctl = (Ctl*)p; p += bCtl;
    T* d_J = (T*)p; p += bJ;
    T* d_b0 = (T*)p; p += bV;
    T* d_b1 = (T*)p; p += bV;
    T* d_partRR = (T*)p; p += bRR;
    T* d_partJy = (T*)p; p += bJy;
    T* d_part = (T*)p;
    if (rowsPad > rows) MIRB200_CUDA(cudaMemsetAsync(d_J + (size_t)rows * ldj, 0, sizeof(T) * (size_t)(rowsPad - rows) * ldj, stream));
    if (ldj > n && cb) MIRB200_CUDA(cudaMemsetAsync(d_J, 0, sizeof(T) * (size_t)rows * ldj, stream));   // pad column (host J has pitch n)

    TR("alloc");
    // ---- control block ----
    std::unique_ptr<Ctl> h(new Ctl);
    std::memset(h.get(), 0, sizeof(Ctl));
    h->st = st; h->n = n; h->ldj = ldj; h->hasG = hasG ? 1 : 0;
    h->tailShortcut = (modelFlags & MIR_MODEL_NO_TAIL_SHORTCUT) ? 0 : 1;
    h->maxAge = st.maxAge ? st.maxAge : (hasG ? 3u : 2u * (unsigned)n);                           // LS:945
    h->status = mir_ls_maxIterations; h->residual = Num<T>::inf();
    h->initPhase = 1; h->doEval = 1; h->ysel = 0; h->mu = 1; h->chunkSeq = 0; h->doneChunk = -1;
    for (int i = 0; i < n; ++i) { h->x[i] = x[i]; h->xt[i] = x[i]; h->l[i] = l[i]; h->u[i] = u[i]; }
    MIRB200_CUDA(cudaMemcpyAsync(d_ctl, h.get(), sizeof(Ctl), cudaMemcpyHostToDevice, stream));

    const size_t ctlSmem = ((CtaQPScratch<T>::bytes(n) + 15) & ~(size_t)15) + sizeof(T) * (4 * (size_t)n + (size_t)np);   // + packed lower J^T J
    MIRB200_CUDA(cudaFuncSetAttribute(large_ctl_mid_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ctlSmem));
    const size_t jacSmem = sizeof(T) * LARGE_TILE * (size_t)(ldj + 1);
    if (kDouble) MIRB200_CUDA(cudaFuncSetAttribute(syrk_dmma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SYRK_SMEM_BYTES));

    EvalArgs<T> ea{d_ctl, d_t, d_yobs, d_b0, d_b1, d_partRR, rows};
    JacArgs<T> ja{d_ctl, d_t, d_yobs, d_b0, d_b1, d_J, d_partJy, rows};

    // host-callback staging
    std::vector<T> hx, hy, hJ;
    struct Mail { int jacMode, doEval, skipRest, done, ysel, initPhase; };
    if (cb) { hx.resize(n); hy.resize((size_t)rows); }
    auto fetch = [&](Mail& m, bool wantXt) -> int {
        MIRB200_CUDA(cudaMemcpyAsync(&m, (char*)d_ctl + offsetof(Ctl, jacMode), sizeof(Mail), cudaMemcpyDeviceToHost, stream));
        MIRB200_CUDA(cudaMemcpyAsync(hx.data(), (char*)d_ctl + (wantXt ? offsetof(Ctl, xt) : offsetof(Ctl, x)), sizeof(T) * n, cudaMemcpyDeviceToHost, stream));
        MIRB200_CUDA(cudaStreamSynchronize(stream));
        return MIR_B200_OK;
    };

    auto allreduce = [&](void* buf, size_t count) -> int { return comm ? nccl_allreduce_sum(buf, count, kDouble, comm, stream) : (int)MIR_B200_OK; };

    auto step_eval = [&]() -> int {
        if (!cb) {
            K.eval<<<gridEval, 256, 0, stream>>>(ea); count_launch();
        } else {
            Mail m; if (int r = fetch(m, true)) return r;
            if (!m.done && m.doEval) {
                cb->f(cb->fCtx, (size_t)rows, (size_t)n, hx.data(), hy.data());                    // LS:953, 1113
                MIRB200_CUDA(cudaMemcpyAsync(m.ysel ? d_b0 : d_b1, hy.data(), sizeof(T) * (size_t)rows, cudaMemcpyHostToDevice, stream));
            }
            large_rr_kernel<T><<<gridEval, 256, 0, stream>>>(ea); count_launch();
        }
        MIRB200_CUDA(cudaGetLastError());
        return allreduce((char*)d_ctl + offsetof(Ctl, rr), 1);
    };

    auto step_jacobian = [&]() -> int {
        if (!cb) {
            auto jk = fdJacobian ? K.jacfd : K.jac;
            jk<<<gridJac, 256, jacSmem, stream>>>(ja); count_launch();
            if (!fuseBroyden) { large_broyden_kernel<T, true><<<gridBro, 256, 0, stream>>>(ja); count_launch(); }   // else: fused into the SYRK ring
        } else {
            Mail m; if (int r = fetch(m, false)) return r;
            if (!m.done && m.jacMode == JAC_FRESH) {
                hJ.resize((size_t)rows * n);
                if (cb->g) cb->g(cb->gCtx, (size_t)rows, (size_t)n, hx.data(), hJ.data());         // LS:1013
                else {                                                                             // LS:1018-1049
                    FDTaskCtx<T> fc{cb, (size_t)rows, (size_t)n, hx.data(), l, u, st.jacobianEpsilon, hJ.data(), (size_t)n};
                    mir_ls_task task{&fc, nullptr};
                    if (cb->tm) cb->tm(cb->tmCtx, (unsigned)n, task, &fd_task<T>);
                    else for (unsigned j = 0; j < (unsigned)n; ++j) fd_task<T>(task, 1, 0, j);
                }
                MIRB200_CUDA(cudaMemcpy2DAsync(d_J, sizeof(T) * ldj, hJ.data(), sizeof(T) * n, sizeof(T) * n, (size_t)rows, cudaMemcpyHostToDevice, stream));
            }
            large_broyden_kernel<T, false><<<gridBro, 256, 0, stream>>>(ja); count_launch();
            if (!fuseBroyden) { large_broyden_kernel<T, true><<<gridBro, 256, 0, stream>>>(ja); count_launch(); }
        }
        if (kDouble) {
            SyrkBroyden sb{fuseBroyden ? 1 : 0, (double*)d_J, (const double*)d_b0, (const double*)d_b1, &d_ctl->ysel, (const double*)d_ctl->dX,
                           (const double*)&d_ctl->deltaX_dot, rows, (double*)d_partJy, &d_ctl->ticket[1], (double*)d_ctl->packed + np, n};
            SyrkArgs sa{(const double*)d_J, rowsPad / SYRK_KT, ldj, (n + 7) / 8, (double*)d_part, &d_ctl->jacMode, &d_ctl->done, sb};
            syrk_dmma_kernel<<<gridSyrk, SYRK_THREADS, SYRK_SMEM_BYTES, stream>>>(sa); count_launch();
            syrk_reduce_kernel<<<(np + 255) / 256, 256, 0, stream>>>((const double*)d_part, (int)gridSyrk, n, (double*)d_ctl->packed, &d_ctl->jacMode, &d_ctl->done);
            count_launch();
        } else {
            syrk_simple_kernel<T><<<gridSyrk, 256, 0, stream>>>(d_J, rows, ldj, d_part, &d_ctl->jacMode, &d_ctl->done); count_launch();
            syrk_reduce_kernel_t<T><<<(np + 255) / 256, 256, 0, stream>>>(d_part, (int)gridSyrk, n, d_ctl->packed, &d_ctl->jacMode, &d_ctl->done);
            count_launch();
        }
        MIRB200_CUDA(cudaGetLastError());
        return allreduce(d_ctl->packed, (size_t)np + n);
    };

    auto step_mid = [&]() -> int {
        large_ctl_mid_kernel<T><<<1, LARGE_CTL_THREADS, ctlSmem, stream>>>(d_ctl); count_launch();
        return check_cuda(cudaGetLastError(), "large_ctl_mid_kernel");
    };
    auto step_post = [&]() -> int {
        large_ctl_post_kernel<T><<<1, LARGE_CTL_THREADS, 0, stream>>>(d_ctl); count_launch();
        return check_cuda(cudaGetLastError(), "large_ctl_post_kernel");
    };

    TR("setup");
    // ---- initial residual, LS:953-956 ----
    if ((rc = step_eval())) return rc;
    if ((rc = step_post())) return rc;

    TR("initial residual");
    // ---- passes: enqueued in chunks, `done` polled one chunk behind ----
    int* h_done = static_cast<int*>(pinned_scratch(2 * sizeof(int)));
    if (!h_done) { set_error("mir_optim_b200: cannot allocate pinned host scratch"); return MIR_B200_ECUDA; }
    h_done[0] = h_done[1] = -1;
    cudaEvent_t ev[2];
    MIRB200_CUDA(cudaEventCreateWithFlags(&ev[0], cudaEventDisableTiming));
    MIRB200_CUDA(cudaEventCreateWithFlags(&ev[1], cudaEventDisableTiming));
    struct FreeEv { cudaEvent_t* e; ~FreeEv() { cudaEventDestroy(e[0]); cudaEventDestroy(e[1]); } } fe{ev};
    const int chunk = cb ? 1 : 4;
    auto enqueue_chunk = [&]() -> int {
        for (int k = 0; k < chunk; ++k) {
            if (int r = step_jacobian()) return r;
            if (int r = step_mid()) return r;
            if (int r = step_eval()) return r;
            if (int r = step_post()) return r;
        }
        // The mailbox carries the index of the chunk in which the solve finished (-1 while it runs), see
        // large_chunk_end_kernel: one host slot serves every chunk and the stop decision below is the same on every
        // rank no matter how late its host reads the slot.
        large_chunk_end_kernel<T><<<1, 1, 0, stream>>>(d_ctl); count_launch();
        return check_cuda(cudaMemcpyAsync(&h_done[0], (char*)d_ctl + offsetof(Ctl, doneChunk), sizeof(int), cudaMemcpyDeviceToHost, stream), "D2H done");
    };
    // Every kernel of a pass takes its arguments from the device-resident control block, so a chunk of passes is the
    // same ~40 launches (+ all-reduces) every time: captured once and replayed as a CUDA graph, the host issues one
    // call per chunk and its scheduling jitter no longer reaches the GPU (measured on shared B200 hosts: the same solve
    // took 0.17 - 0.99 s with direct launches).  Host callbacks need the host between kernels: direct launches.
    struct GraphHolder {
        cudaGraph_t g = nullptr; cudaGraphExec_t x = nullptr;
        ~GraphHolder() { if (x) cudaGraphExecDestroy(x); if (g) cudaGraphDestroy(g); }
    } graph;
    static const bool noGraph = [] { const char* e = std::getenv("MIRB200_NO_GRAPH"); return e && *e == '1'; }();
    unsigned launchesPerChunk = 0;
    if (!cb && !noGraph) {
        const unsigned long long l0 = mir_b200_kernel_launches();
        if (cudaStreamBeginCapture(stream, cudaStreamCaptureModeThreadLocal) == cudaSuccess) {
            const int rcap = enqueue_chunk();
            const cudaError_t ec = cudaStreamEndCapture(stream, &graph.g);
            if (rcap != MIR_B200_OK || ec != cudaSuccess || cudaGraphInstantiate(&graph.x, graph.g, 0) != cudaSuccess) {
                cudaGetLastError(); clear_error();
                if (graph.x) { cudaGraphExecDestroy(graph.x); graph.x = nullptr; }
            }
        } else cudaGetLastError();
        launchesPerChunk = (unsigned)(mir_b200_kernel_launches() - l0);
        count_launch(-(long long)launchesPerChunk);     // the capture pass launched nothing
    }
    bool finished = false;
    for (unsigned long long c = 0; !finished; ++c) {
        if (graph.x) { MIRB200_CUDA(cudaGraphLaunch(graph.x, stream)); count_launch(launchesPerChunk); }
        else if ((rc = enqueue_chunk())) return rc;
        const int slot = (int)(c & 1);
        MIRB200_CUDA(cudaEventRecord(ev[slot], stream));
        // decide from the state at the end of the chunk that was synchronised on, and from nothing later: every rank
        // of a sharded run then enqueues exactly doneChunk + 2 chunks (the last one a no-op whose all-reduces still pair up)
        if (cb) { MIRB200_CUDA(cudaEventSynchronize(ev[slot])); finished = h_done[0] >= 0; }
        else if (c >= 1) {
            MIRB200_CUDA(cudaEventSynchronize(ev[slot ^ 1]));
            const int dc = *(volatile int*)&h_done[0];
            finished = dc >= 0 && (unsigned long long)dc <= c - 1;
        }
    }

    TR("passes");
    // ---- results ----
    MIRB200_CUDA(cudaMemcpyAsync(h.get(), d_ctl, offsetof(Ctl, JJ), cudaMemcpyDeviceToHost, stream));
    MIRB200_CUDA(cudaStreamSynchronize(stream));
    TR("results");
    for (int i = 0; i < n; ++i) x[i] = h->x[i];
    result->status = h->status; result->iterations = h->iterations; result->fCalls = h->fCalls; result->gCalls = h->gCalls;
    result->residual = h->residual; result->lambda = h->lambda;
    if (stats) {
        stats->problems = 1; stats->passes = h->passes; stats->accepted = h->accepted; stats->fresh_jacobians = h->fresh;
        stats->broyden_updates = h->broyden; stats->model_evals = h->evals; stats->qp_solves = h->qpSolves; stats->qp_iterations = h->qpIters;
    }
    return MIR_B200_OK;
}

// ---------------------------------------------------------------------------------------------
// legacy entry points, least_squares.d:705-748
// ---------------------------------------------------------------------------------------------
template <class T> struct Sentinels;
template <> struct Sentinels<double> { static void* f() { return (void*)&mir_b200_device_model_d; } static void* g() { return (void*)&mir_b200_device_model_jac_d; } };
template <> struct Sentinels<float>  { static void* f() { return (void*)&mir_b200_device_model_s; } static void* g() { return (void*)&mir_b200_device_model_jac_s; } };

template <class T, class F, class G>
static typename Num<T>::Result legacy_entry(const typename Num<T>::Settings* settings, size_t m, size_t n, T* x, const T* l, const T* u,
                                            void* fContext, F f, void* gContext, G g, void* tmContext, mir_ls_thread_manager tm)
{
    using Result = typename Num<T>::Result;
    clear_error();
    Result ret;
    ret.status = mir_ls_numericError; ret.iterations = 0; ret.fCalls = 0; ret.gCalls = 0; ret.residual = Num<T>::inf(); ret.lambda = 0;
    if (!settings || !f || (n && (!x || !l || !u))) { set_error("mir_optim_b200: null argument"); return ret; }

    if ((void*)f == Sentinels<T>::f()) {
        // device-functor mode: fContext is a mir_model_desc with HOST arrays; g selects analytic vs finite differences
        const mir_model_desc* desc = static_cast<const mir_model_desc*>(fContext);
        if (!desc) { set_error("mir_optim_b200: device-model mode needs fContext = mir_model_desc*"); return ret; }
        if (g && (void*)g != Sentinels<T>::g()) { set_error("mir_optim_b200: device-model mode takes g = NULL (finite differences) or mir_b200_device_model_jac_*"); return ret; }
        // (the flags are masked below: without these checks a weighted or robust desc would run as a plain one)
        if (desc->flags & MIR_MODEL_WEIGHTED) {
            set_error("mir_optim_b200: MIR_MODEL_WEIGHTED is supported by the batched and covariance entry points, not by device-model mode");
            return ret;
        }
        if (desc->flags & (MIR_MODEL_LOSS_SOFT_L1 | MIR_MODEL_LOSS_HUBER)) {
            set_error("mir_optim_b200: robust losses (MIR_MODEL_LOSS_*) are supported by the batched entry points, not by device-model mode");
            return ret;
        }
        mir_model_desc d = *desc;
        d.flags = (d.flags & (uint32_t)MIR_MODEL_NO_TAIL_SHORTCUT) | (g ? 0u : (uint32_t)MIR_MODEL_FD_JACOBIAN);
        // small shapes, fitSpline's residual and models compiled at run time: the batched kernels with a batch of one;
        // many rows of a model the row-parallel engine knows: that engine
        const bool rowEngineModel = d.model == MIR_MODEL_EXPDECAY2 || d.model == MIR_MODEL_EXPTAU3 || d.model == MIR_MODEL_EXPDECAY3 ||
                                    d.model == MIR_MODEL_GAUSS4 || d.model == MIR_MODEL_SUMEXP || d.model == MIR_MODEL_GAUSSMIX;
        int rc = MIR_B200_EUNSUPPORTED;
        if (!(rowEngineModel && m > 128)) {
            d.aux = desc->aux; d.param = desc->param;
            rc = batched_host_entry<T>(settings, &d, 1, m, n, x, l, u, 0, &ret, nullptr, -1);
            if (rc == MIR_B200_OK) return ret;
            if (rc != MIR_B200_EUNSUPPORTED || !rowEngineModel) { ret.status = mir_ls_numericError; return ret; }
        }
        clear_error();
        if (require_device(-1)) return ret;
        cudaStream_t stream = nullptr;
        if (check_cuda(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking), "cudaStreamCreate")) return ret;
        T *dt = nullptr, *dy = nullptr;
        const size_t bytes = sizeof(T) * (m ? m : 1);
        if (check_cuda(cudaMallocAsync((void**)&dt, bytes, stream), "cudaMallocAsync") || check_cuda(cudaMallocAsync((void**)&dy, bytes, stream), "cudaMallocAsync")) {
            cudaStreamDestroy(stream); return ret;
        }
        if (m && d.t) cudaMemcpyAsync(dt, d.t, sizeof(T) * m, cudaMemcpyHostToDevice, stream);
        if (m && d.y) cudaMemcpyAsync(dy, d.y, sizeof(T) * m, cudaMemcpyHostToDevice, stream);
        rc = large_solve<T>(*settings, d.model, d.flags, (long long)m, n, dt, dy, nullptr, x, l, u, nullptr, stream, &ret, nullptr);
        cudaFreeAsync(dt, stream); cudaFreeAsync(dy, stream);
        cudaStreamSynchronize(stream); cudaStreamDestroy(stream);
        if (rc) ret.status = mir_ls_numericError;
        return ret;
    }

    // host-callback mode: f / g run on the host exactly when the reference would call them; everything else on the GPU
    HostCallbacks<T> cb;
    cb.fCtx = fContext; cb.f = f; cb.gCtx = gContext; cb.g = g; cb.tmCtx = tmContext; cb.tm = tm;
    if (n > (size_t)LARGE_NMAX) { set_error("mir_optim_b200: the single-problem GPU path supports n <= 128 parameters"); return ret; }
    {
        const int vs = validate_args<T>(*settings, m > 0, n, x, l, u);
        if (vs) { ret.status = vs; return ret; }
    }
    if (require_device(-1)) return ret;
    cudaStream_t stream = nullptr;
    if (check_cuda(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking), "cudaStreamCreate")) return ret;
    const int rc = large_solve<T>(*settings, 0, g ? 0u : (unsigned)MIR_MODEL_FD_JACOBIAN, (long long)m, n, nullptr, nullptr, &cb, x, l, u, nullptr, stream, &ret, nullptr);
    cudaStreamSynchronize(stream); cudaStreamDestroy(stream);
    if (rc) ret.status = mir_ls_numericError;
    return ret;
}

}  // namespace mirb200

using namespace mirb200;

extern "C" {

// Sentinels: never meant to be called; they mark "evaluate the built-in model on the device".
void mir_b200_device_model_d(void*, size_t, size_t, const double*, double*) {}
void mir_b200_device_model_jac_d(void*, size_t, size_t, const double*, double*) {}
void mir_b200_device_model_s(void*, size_t, size_t, const float*, float*) {}
void mir_b200_device_model_jac_s(void*, size_t, size_t, const float*, float*) {}

mir_least_squares_result_d mir_optimize_least_squares_d(const mir_least_squares_settings_d* settings, size_t m, size_t n, double* x,
    const double* l, const double* u, mir_slice_d work, mir_slice_i iwork, void* fContext, mir_ls_function_d f, void* gContext,
    mir_ls_jacobian_d g, void* tmContext, mir_ls_thread_manager tm)
{
    (void)work; (void)iwork;      // caller scratch of the CPU implementation; the engine's state lives in device memory
    return legacy_entry<double>(settings, m, n, x, l, u, fContext, f, gContext, g, tmContext, tm);
}

mir_least_squares_result_s mir_optimize_least_squares_s(const mir_least_squares_settings_s* settings, size_t m, size_t n, float* x,
    const float* l, const float* u, mir_slice_s work, mir_slice_i iwork, void* fContext, mir_ls_function_s f, void* gContext,
    mir_ls_jacobian_s g, void* tmContext, mir_ls_thread_manager tm)
{
    (void)work; (void)iwork;
    return legacy_entry<float>(settings, m, n, x, l, u, fContext, f, gContext, g, tmContext, tm);    // real m (the reference passes 2, LS:629)
}

int mir_optimize_least_squares_sharded_d(const mir_least_squares_settings_d* settings, const mir_model_desc* model, size_t m_local,
    size_t n, double* x, const double* l, const double* u, void* nccl_comm, void* cuda_stream, mir_least_squares_result_d* result,
    mir_batch_stats* stats)
{
    clear_error();
    if (!settings || !model || !x || !l || !u || !result) { set_error("mir_optim_b200: null argument"); return MIR_B200_EINVAL; }
    if (m_local && (!model->t || !model->y)) { set_error("mir_optim_b200: sharded solve needs device pointers model->t / model->y"); return MIR_B200_EINVAL; }
    if (model->flags & MIR_MODEL_WEIGHTED) { set_error("mir_optim_b200: the sharded solve does not support MIR_MODEL_WEIGHTED"); return MIR_B200_EUNSUPPORTED; }
    if (model->flags & (MIR_MODEL_LOSS_SOFT_L1 | MIR_MODEL_LOSS_HUBER)) { set_error("mir_optim_b200: the sharded solve does not support robust losses (MIR_MODEL_LOSS_*)"); return MIR_B200_EUNSUPPORTED; }
    return large_solve<double>(*settings, model->model, model->flags, (long long)m_local, n,
                               (const double*)model->t, (const double*)model->y, nullptr, x, l, u, nccl_comm, (cudaStream_t)cuda_stream,
                               result, stats);
}

// J^T J alone: J is rows x ldj row-major on the device (rows % 32 == 0, ldj even, n <= ldj <= 128),
// packed receives the lower triangle by rows (n(n+1)/2 doubles, device).  scratch: >= grid*128*128 doubles or NULL.
int mir_b200_syrk_lower_dev_d(const double* J, size_t rows, size_t n, size_t ldj, double* packed, void* cuda_stream)
{
    clear_error();
    if (!J || !packed || n == 0 || n > 128 || ldj < n || ldj > 128 || (ldj & 1) || rows % SYRK_KT) {
        set_error("mir_optim_b200: syrk needs rows % 32 == 0, even ldj, n <= ldj <= 128"); return MIR_B200_EINVAL;
    }
    int rc = require_device(-1);
    if (rc) return rc;
    cudaStream_t stream = (cudaStream_t)cuda_stream;
    const long long tiles = (long long)(rows / SYRK_KT);
    unsigned grid = (unsigned)(tiles < sm_count() ? (tiles ? tiles : 1) : sm_count());
    double* part = nullptr; int* flags = nullptr;
    MIRB200_CUDA(cudaMallocAsync((void**)&part, sizeof(double) * (size_t)grid * SYRK_NPAD * SYRK_NPAD + 64, stream));
    flags = (int*)(part + (size_t)grid * SYRK_NPAD * SYRK_NPAD);
    const int hf[2] = {1, 0};
    MIRB200_CUDA(cudaMemcpyAsync(flags, hf, sizeof hf, cudaMemcpyHostToDevice, stream));
    MIRB200_CUDA(cudaFuncSetAttribute(syrk_dmma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SYRK_SMEM_BYTES));
    SyrkArgs sa{J, tiles, (int)ldj, (int)((n + 7) / 8), part, flags, flags + 1, SyrkBroyden{}};
    syrk_dmma_kernel<<<grid, SYRK_THREADS, SYRK_SMEM_BYTES, stream>>>(sa); count_launch();
    const int np = (int)(n * (n + 1) / 2);
    syrk_reduce_kernel<<<(np + 255) / 256, 256, 0, stream>>>(part, (int)grid, (int)n, packed, flags, flags + 1); count_launch();
    rc = check_cuda(cudaGetLastError(), "syrk launch");
    cudaFreeAsync(part, stream);
    return rc;
}

}  // extern "C"
