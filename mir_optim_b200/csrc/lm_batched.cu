// lm_batched.cu -- C ABI of the batched LM entry points (header part 2): argument checks,
// staging of host buffers, stream-ordered scratch, launch of the warp-per-problem kernel.
#include <cstdlib>
#include <cstring>
#include <string>

#include "lm_small_launch.cuh"
#include "runtime.cuh"

namespace mirb200 {
// general batched kernel, one CTA per problem, any n <= 128 (lm_cta.cuh / lm_cta_inst.cu)
template <class T>
int launch_cta_model(const mir_model_desc& model, size_t n, const typename Num<T>::Settings& st, const SmallBatchArgs& args, cudaStream_t stream);
}

extern char** environ;

namespace mirb200 {

// Models that read samples need both arrays (t: m or batch*m abscissae, y: batch*m observations -- the lengths are the
// caller's contract, stated in the header); only LINEAR2, ROSENBROCK and SQRTCIRCLE are data-free.
static bool model_data_free(unsigned model)
{
    return model == MIR_MODEL_LINEAR2 || model == MIR_MODEL_ROSENBROCK || model == MIR_MODEL_SQRTCIRCLE;
}
static bool model_needs_data(unsigned model)
{
    return !(model_data_free(model) || model >= (unsigned)MIR_MODEL_USER_BASE);
}
// Shapes the specialised kernels (lm_tpp / lm_mux / lm_small) instantiate; everything else goes to the general kernel.
static bool specialised_shape(unsigned model, size_t n)
{
    switch (model) {
    case MIR_MODEL_LINEAR2: case MIR_MODEL_ROSENBROCK: case MIR_MODEL_SQRTCIRCLE: case MIR_MODEL_EXPDECAY2: return n == 2;
    case MIR_MODEL_EXPTAU3: case MIR_MODEL_EXPDECAY3: return n == 3;
    case MIR_MODEL_GAUSS4: return n == 4;
    case MIR_MODEL_SUMEXP: return n == 4 || n == 8;
    default: return false;
    }
}
// the samples and weights check of the batched fit and of the covariance (lm_cov.cu)
int check_model_data(const mir_model_desc* model, size_t batch, size_t m)
{
    if (batch && m && model_needs_data(model->model) && (!model->t || !model->y)) {
        set_error("mir_optim_b200: this model reads samples: model->t and model->y must not be NULL");
        return MIR_B200_EINVAL;
    }
    if (model->flags & MIR_MODEL_WEIGHTED) {
        if (model_data_free(model->model)) {
            set_error("mir_optim_b200: MIR_MODEL_WEIGHTED needs a model with observation rows (not LINEAR2, ROSENBROCK or SQRTCIRCLE)");
            return MIR_B200_EUNSUPPORTED;
        }
        if (batch && m && !model->w) { set_error("mir_optim_b200: MIR_MODEL_WEIGHTED: model->w must not be NULL"); return MIR_B200_EINVAL; }
    }
    return MIR_B200_OK;
}

template <class T>
static int batched_dev(const typename Num<T>::Settings* settings, const mir_model_desc* model, size_t batch, size_t m, size_t n,
                       T* x, const T* l, const T* u, size_t bound_stride, typename Num<T>::Result* results,
                       mir_batch_stats* stats, cudaStream_t stream, const unsigned int* ready = nullptr, unsigned spinLimit = 0)
{
    clear_error();
    if (!settings || !model || (batch && (!x || !l || !u || !results))) { set_error("mir_optim_b200: null argument"); return MIR_B200_EINVAL; }
    if (int rcm = check_model_data(model, batch, m)) return rcm;
    if (n == 0) { set_error("mir_optim_b200: n must be > 0 for the batched entry point"); return MIR_B200_EINVAL; }
    if (bound_stride != 0 && bound_stride < n) { set_error("mir_optim_b200: bound_stride must be 0 or >= n"); return MIR_B200_EINVAL; }
    if (batch == 0) return MIR_B200_OK;
    int rc = require_device(-1);
    if (rc) return rc;

    if (batch >= 0xffffffffull) { set_error("mir_optim_b200: at most 2^32 - 2 problems per launch"); return MIR_B200_EINVAL; }
    unsigned int* counter = nullptr;
    MIRB200_CUDA(cudaMallocAsync((void**)&counter, sizeof(unsigned int), stream));
    MIRB200_CUDA(cudaMemsetAsync(counter, 0, sizeof(unsigned int), stream));

    SmallBatchArgs a;
    a.t = model->t; a.y = model->y; a.x = x; a.l = l; a.u = u; a.results = results;
    a.counter = counter; a.ready = ready; a.spin_limit = spinLimit; a.stats = stats; a.batch = batch; a.m = (unsigned)m;
    a.bound_stride = (unsigned)bound_stride; a.flags = model->flags;
    static const bool forceGeneral = [] { const char* e = std::getenv("MIRB200_BATCH_KERNEL"); return e && !std::strcmp(e, "cta"); }();   // tests / experiments
    // weights are an adapter of the general kernel's models (CtaWeighted): the specialised kernels never see them
    if (specialised_shape(model->model, n) && !forceGeneral && !(model->flags & MIR_MODEL_WEIGHTED)) {
        rc = launch_small_model<T>(model->model, n, *settings, a, stream);
        // a shape the specialised kernels do not cover after all (m beyond their rows-per-lane instantiations): general kernel
        if (rc == MIR_B200_EUNSUPPORTED && model_needs_data(model->model) && batch > 1) { clear_error(); rc = launch_cta_model<T>(*model, n, *settings, a, stream); }
    } else {
        rc = launch_cta_model<T>(*model, n, *settings, a, stream);
    }
    cudaFreeAsync(counter, stream);
    return rc;
}

// True when something in the environment serialises kernel launches against copies (or makes launches blocking), so a
// kernel running beside the copies that feed it cannot be relied on: CUDA_LAUNCH_BLOCKING, an injected tool library
// (Nsight Compute / Systems, compute-sanitizer and CUPTI tools all enter through CUDA_INJECTION64_PATH), or the
// profilers' own variables.  MIRB200_NO_STAGING=1 forces the same plain path by hand.
static bool launches_may_serialise()
{
    auto set = [](const char* name) { const char* e = std::getenv(name); return e && *e && std::strcmp(e, "0") != 0; };
    if (set("MIRB200_NO_STAGING") || set("CUDA_LAUNCH_BLOCKING") || set("CUDA_INJECTION64_PATH") || set("CUDA_INJECTION32_PATH")) return true;
    for (char** e = ::environ; e && *e; ++e)
        if (!std::strncmp(*e, "NV_COMPUTE_PROFILER_", 20) || !std::strncmp(*e, "NV_NSIGHT_", 10) || !std::strncmp(*e, "NSYS_", 5) ||
            !std::strncmp(*e, "NV_SANITIZER_", 13)) return true;
    return false;
}

template <class T>
static int batched_host(const typename Num<T>::Settings* settings, const mir_model_desc* model, size_t batch, size_t m, size_t n,
                        T* x, const T* l, const T* u, size_t bound_stride, typename Num<T>::Result* results,
                        mir_batch_stats* stats, int device)
{
    using Result = typename Num<T>::Result;
    clear_error();
    if (!settings || !model || (batch && (!x || !l || !u || !results))) { set_error("mir_optim_b200: null argument"); return MIR_B200_EINVAL; }
    if (int rcm = check_model_data(model, batch, m)) return rcm;
    int rc = require_device(device);
    if (rc) return rc;
    if (batch == 0) return MIR_B200_OK;

    const bool per = (model->flags & MIR_MODEL_GRID_PER_PROBLEM) != 0;
    const size_t tBytes = model->t ? sizeof(T) * (per ? batch * m : m) : 0;
    const size_t yBytes = model->y ? sizeof(T) * batch * m : 0;
    const size_t wBytes = (model->flags & MIR_MODEL_WEIGHTED) ? sizeof(T) * batch * m : 0;
    const size_t xBytes = sizeof(T) * batch * n;
    const size_t bBytes = sizeof(T) * (bound_stride ? batch * bound_stride : n);
    const size_t rBytes = sizeof(Result) * batch;
    const size_t aBytes = model->aux ? sizeof(T) * ((model->flags & MIR_MODEL_AUX_PER_PROBLEM) ? batch * n : n) : 0;

    // Pipeline ("staged").  ONE kernel launch for the whole batch (chunked launches lose ~15 % to queue drain at this grid
    // size) that runs BESIDE the copies feeding it: the per-problem inputs go to the device on a copy stream in chunks of
    // 65536 problems, each followed by a 4-byte watermark copy, and a thread that pulls problem i from the work queue
    // waits until the watermark has passed i (wait_staged).  The copy engine runs ~3x ahead of the solve, so only the
    // first chunk's transfer is exposed.  Every copy is enqueued BEFORE the launch and the launch is ordered after the
    // first chunk, so a launch call that blocks the host cannot starve the kernel of its inputs; where launches may be
    // serialised against copies anyway (launches_may_serialise) the plain order copy -> kernel -> copy is used, and if
    // the kernel still times out waiting (flag d_ready[1]) its results are discarded and the batch is re-run plainly.
    static const bool plainOnly = launches_may_serialise();
    static const unsigned spinLimit = [] {
        const char* e = std::getenv("MIRB200_STAGING_SPINS");
        const long long v = e ? std::atoll(e) : 0;
        return (unsigned)(v > 0 ? v : 2000000);                  // ~5 s without any progress of the watermark
    }();
    static const bool testStall = [] { const char* e = std::getenv("MIRB200_TEST_STALL_STAGING"); return e && *e == '1'; }();   // tests: withhold the watermark
    const bool staged = !plainOnly;
    const size_t chunk = 65536;
    const size_t nchunks = (batch + chunk - 1) / chunk;
    cudaStream_t cs = nullptr, ps = nullptr;
    cudaEvent_t ev = nullptr, ev0 = nullptr;
    unsigned int* h_wm = nullptr;
    rc = MIR_B200_OK;
    auto CK = [&](cudaError_t err, const char* what) { if (rc == MIR_B200_OK) rc = check_cuda(err, what); };
    CK(cudaStreamCreateWithFlags(&cs, cudaStreamNonBlocking), "cudaStreamCreate");
    CK(cudaStreamCreateWithFlags(&ps, cudaStreamNonBlocking), "cudaStreamCreate");
    CK(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming), "cudaEventCreate");
    CK(cudaEventCreateWithFlags(&ev0, cudaEventDisableTiming), "cudaEventCreate");
    h_wm = static_cast<unsigned int*>(pinned_scratch(sizeof(unsigned int) * (nchunks + 4)));
    if (!h_wm && rc == MIR_B200_OK) { set_error("mir_optim_b200: cannot allocate pinned host scratch"); rc = MIR_B200_ECUDA; }
    auto cleanup = [&]() {
        if (cs) cudaStreamDestroy(cs);
        if (ps) cudaStreamDestroy(ps);
        if (ev) cudaEventDestroy(ev);
        if (ev0) cudaEventDestroy(ev0);
    };
    if (rc != MIR_B200_OK) { cleanup(); return rc; }
    unsigned int* const h_flag = h_wm + nchunks + 1;              // time-out flag read back from the device
    *h_flag = 0;

    auto align = [](size_t v) { return (v + 255) & ~(size_t)255; };
    const size_t total = align(tBytes) + align(yBytes) + align(xBytes) + 2 * align(bBytes) + align(rBytes) + align(sizeof(mir_batch_stats)) + align(aBytes) + 256
                         + align(wBytes);
    char* base = nullptr;
    cudaError_t e = cudaMallocAsync((void**)&base, total, cs);
    if (e != cudaSuccess) { cleanup(); return check_cuda(e, "cudaMallocAsync(batch buffers)"); }
    char* p = base;
    T* dt = (T*)p; p += align(tBytes);
    T* dy = (T*)p; p += align(yBytes);
    T* dx = (T*)p; p += align(xBytes);
    T* dl = (T*)p; p += align(bBytes);
    T* du = (T*)p; p += align(bBytes);
    Result* dr = (Result*)p; p += align(rBytes);
    mir_batch_stats* ds = (mir_batch_stats*)p; p += align(sizeof(mir_batch_stats));
    T* da = (T*)p; p += align(aBytes);
    unsigned int* d_ready = (unsigned int*)p; p += 256;           // {watermark, time-out flag}
    T* dw = (T*)p;

    // shared inputs, counters and the watermark (0 = nothing staged) on the compute stream; the copy stream starts behind them
    if (tBytes && !per) CK(cudaMemcpyAsync(dt, model->t, tBytes, cudaMemcpyHostToDevice, cs), "H2D t");
    if (!bound_stride) {
        CK(cudaMemcpyAsync(dl, l, bBytes, cudaMemcpyHostToDevice, cs), "H2D l");
        CK(cudaMemcpyAsync(du, u, bBytes, cudaMemcpyHostToDevice, cs), "H2D u");
    }
    if (aBytes) CK(cudaMemcpyAsync(da, model->aux, aBytes, cudaMemcpyHostToDevice, cs), "H2D aux");
    if (stats) CK(cudaMemsetAsync(ds, 0, sizeof(mir_batch_stats), cs), "memset stats");
    CK(cudaMemsetAsync(d_ready, 0, 2 * sizeof(unsigned int), cs), "memset watermark");
    CK(cudaEventRecord(ev, cs), "cudaEventRecord");
    CK(cudaStreamWaitEvent(ps, ev, 0), "cudaStreamWaitEvent");
    // the per-problem inputs, chunk by chunk
    size_t c = 0;
    for (size_t lo = 0; lo < batch && rc == MIR_B200_OK; lo += chunk, ++c) {
        const size_t nb = (lo + chunk <= batch) ? chunk : batch - lo;
        if (tBytes && per) CK(cudaMemcpyAsync(dt + lo * m, static_cast<const T*>(model->t) + lo * m, sizeof(T) * nb * m, cudaMemcpyHostToDevice, ps), "H2D t");
        if (yBytes) CK(cudaMemcpyAsync(dy + lo * m, static_cast<const T*>(model->y) + lo * m, sizeof(T) * nb * m, cudaMemcpyHostToDevice, ps), "H2D y");
        if (wBytes) CK(cudaMemcpyAsync(dw + lo * m, static_cast<const T*>(model->w) + lo * m, sizeof(T) * nb * m, cudaMemcpyHostToDevice, ps), "H2D w");
        CK(cudaMemcpyAsync(dx + lo * n, x + lo * n, sizeof(T) * nb * n, cudaMemcpyHostToDevice, ps), "H2D x");
        if (model->flags & MIR_MODEL_WARM_START) CK(cudaMemcpyAsync(dr + lo, results + lo, sizeof(Result) * nb, cudaMemcpyHostToDevice, ps), "H2D results (warm start)");
        if (bound_stride) {
            CK(cudaMemcpyAsync(dl + lo * bound_stride, l + lo * bound_stride, sizeof(T) * nb * bound_stride, cudaMemcpyHostToDevice, ps), "H2D l");
            CK(cudaMemcpyAsync(du + lo * bound_stride, u + lo * bound_stride, sizeof(T) * nb * bound_stride, cudaMemcpyHostToDevice, ps), "H2D u");
        }
        if (staged) {
            h_wm[c] = (unsigned int)(lo + nb);
            if (!testStall || c == 0) CK(cudaMemcpyAsync(d_ready, &h_wm[c], sizeof(unsigned int), cudaMemcpyHostToDevice, ps), "H2D watermark");
            if (c == 0) CK(cudaEventRecord(ev0, ps), "cudaEventRecord");
        }
    }
    auto launch = [&](const unsigned int* ready) {
        mir_model_desc dm = *model;
        dm.t = tBytes ? dt : nullptr; dm.y = yBytes ? dy : nullptr; dm.aux = aBytes ? da : nullptr; dm.w = wBytes ? dw : nullptr;
        if (rc == MIR_B200_OK) rc = batched_dev<T>(settings, &dm, batch, m, n, dx, dl, du, bound_stride, dr, stats ? ds : nullptr, cs, ready, spinLimit);
    };
    if (staged) {
        CK(cudaStreamWaitEvent(cs, ev0, 0), "cudaStreamWaitEvent");         // the first chunk is resident before the kernel starts
        launch(d_ready);
        CK(cudaMemcpyAsync(h_flag, d_ready + 1, sizeof(unsigned int), cudaMemcpyDeviceToHost, cs), "D2H staging flag");
    } else {
        CK(cudaEventRecord(ev0, ps), "cudaEventRecord");
        CK(cudaStreamWaitEvent(cs, ev0, 0), "cudaStreamWaitEvent");
        launch(nullptr);
    }
    auto copy_back = [&]() {
        CK(cudaMemcpyAsync(x, dx, xBytes, cudaMemcpyDeviceToHost, cs), "D2H x");
        CK(cudaMemcpyAsync(results, dr, rBytes, cudaMemcpyDeviceToHost, cs), "D2H results");
        if (stats) CK(cudaMemcpyAsync(stats, ds, sizeof(mir_batch_stats), cudaMemcpyDeviceToHost, cs), "D2H stats");
    };
    // x and results are caller memory: they are only overwritten once the launch is known to be good, so the staged
    // path reads the flag first (the copy engine is idle by then; the D2H of 40 B per fit costs ~1 ms per 2^20 fits)
    cudaError_t se = cudaStreamSynchronize(ps);
    if (rc == MIR_B200_OK) rc = check_cuda(se, "batched LM input staging");
    if (!staged) copy_back();
    se = cudaStreamSynchronize(cs);
    if (rc == MIR_B200_OK) rc = check_cuda(se, "batched LM kernel");
    if (staged && rc == MIR_B200_OK) {
        if (*h_flag) {
            // the kernel gave up waiting for its inputs (the copies could not run beside it): every input is resident
            // now, x was partly overwritten by the problems that did run -- restore it and run the batch plainly
            CK(cudaMemcpyAsync(dx, x, xBytes, cudaMemcpyHostToDevice, cs), "H2D x (re-run)");
            if (model->flags & MIR_MODEL_WARM_START) CK(cudaMemcpyAsync(dr, results, rBytes, cudaMemcpyHostToDevice, cs), "H2D results (re-run)");
            if (stats) CK(cudaMemsetAsync(ds, 0, sizeof(mir_batch_stats), cs), "memset stats");
            launch(nullptr);
        }
        copy_back();
        se = cudaStreamSynchronize(cs);
        if (rc == MIR_B200_OK) rc = check_cuda(se, "batched LM kernel");
    }
    cudaFreeAsync(base, cs);
    cudaStreamSynchronize(cs);
    cleanup();
    return rc;
}

// used by the legacy single-problem entry (lm_large.cu) for shapes the register-resident kernel covers
template <class T>
int batched_host_entry(const typename Num<T>::Settings* settings, const mir_model_desc* model, size_t batch, size_t m, size_t n,
                       T* x, const T* l, const T* u, size_t bound_stride, typename Num<T>::Result* results,
                       mir_batch_stats* stats, int device)
{ return batched_host<T>(settings, model, batch, m, n, x, l, u, bound_stride, results, stats, device); }
template int batched_host_entry<double>(const mir_least_squares_settings_d*, const mir_model_desc*, size_t, size_t, size_t, double*, const double*,
                                        const double*, size_t, mir_least_squares_result_d*, mir_batch_stats*, int);
template int batched_host_entry<float>(const mir_least_squares_settings_s*, const mir_model_desc*, size_t, size_t, size_t, float*, const float*,
                                       const float*, size_t, mir_least_squares_result_s*, mir_batch_stats*, int);

}  // namespace mirb200

using namespace mirb200;

extern "C" {

int mir_optimize_least_squares_batched_d(const mir_least_squares_settings_d* s, const mir_model_desc* model, size_t batch, size_t m,
    size_t n, double* x, const double* l, const double* u, size_t bound_stride, mir_least_squares_result_d* results,
    mir_batch_stats* stats, int device)
{ return batched_host<double>(s, model, batch, m, n, x, l, u, bound_stride, results, stats, device); }

int mir_optimize_least_squares_batched_s(const mir_least_squares_settings_s* s, const mir_model_desc* model, size_t batch, size_t m,
    size_t n, float* x, const float* l, const float* u, size_t bound_stride, mir_least_squares_result_s* results,
    mir_batch_stats* stats, int device)
{ return batched_host<float>(s, model, batch, m, n, x, l, u, bound_stride, results, stats, device); }

int mir_optimize_least_squares_batched_dev_d(const mir_least_squares_settings_d* s, const mir_model_desc* model, size_t batch, size_t m,
    size_t n, double* x, const double* l, const double* u, size_t bound_stride, mir_least_squares_result_d* results,
    mir_batch_stats* stats, void* stream)
{ return batched_dev<double>(s, model, batch, m, n, x, l, u, bound_stride, results, stats, (cudaStream_t)stream); }

int mir_optimize_least_squares_batched_dev_s(const mir_least_squares_settings_s* s, const mir_model_desc* model, size_t batch, size_t m,
    size_t n, float* x, const float* l, const float* u, size_t bound_stride, mir_least_squares_result_s* results,
    mir_batch_stats* stats, void* stream)
{ return batched_dev<float>(s, model, batch, m, n, x, l, u, bound_stride, results, stats, (cudaStream_t)stream); }

}  // extern "C"
