// lm_cov.cu -- C ABI of the batched covariance entry points (mir_b200_covariance_batched_*): argument checks, staging of
// host buffers, and the launch of lm_cov_cta_kernel (lm_cov.cuh) for the built-in models, with the model table
// (visit_cta_model) and the launch policy (launch_persistent) of the general batched LM kernel.
#include "lm_cov.cuh"
#include "runtime.cuh"

namespace mirb200 {

extern template int launch_cov_builtin<double, true>(const mir_model_desc&, double, CovArgs, const char*, cudaStream_t);
extern template int launch_cov_builtin<float, true>(const mir_model_desc&, float, CovArgs, const char*, cudaStream_t);

int check_model_data(const mir_model_desc* model, size_t batch, size_t m);   // lm_batched.cu

namespace {

constexpr const char* kNoCovModel = "mir_optim_b200: model id not available for the covariance (it has no run-time-n functor)";

// argument checks shared by both forms (batch may be 0; data pointers are checked by the caller when batch > 0)
template <class T>
int cov_check(const mir_model_desc* model, size_t m, size_t n, const void* cov, const void* stddev)
{
    if (!model) { set_error("mir_optim_b200: null model"); return MIR_B200_EINVAL; }
    if (!cov && !stddev) { set_error("mir_optim_b200: cov and stddev are both NULL: nothing to compute"); return MIR_B200_EINVAL; }
    if (n == 0 || m == 0) { set_error("mir_optim_b200: m and n must be > 0"); return MIR_B200_EINVAL; }
    if (n > 128) { set_error("mir_optim_b200: the covariance supports n <= 128"); return MIR_B200_EUNSUPPORTED; }
    if (m >= 0x7fffffffull) { set_error("mir_optim_b200: m too large"); return MIR_B200_EUNSUPPORTED; }
    if (model->model >= (uint32_t)MIR_MODEL_USER_BASE) return MIR_B200_OK;      // checked when the model is loaded
    return visit_cta_model<T>(*model, kNoCovModel, [&](auto tag) {
        using M = typename decltype(tag)::type;
        if (!M::valid((int)n, (int)m)) { set_error("mir_optim_b200: (m, n) not valid for this model"); return (int)MIR_B200_EINVAL; }
        return (int)MIR_B200_OK;
    });
}

template <class T>
int cov_check_data(const mir_model_desc* model, size_t batch, size_t m, const T* x, const T* l, const T* u, size_t n, size_t bound_stride,
                   const int32_t* info)
{
    if (!x || !l || !u || !info) { set_error("mir_optim_b200: null argument"); return MIR_B200_EINVAL; }
    if (int rc = check_model_data(model, batch, m)) return rc;
    if (bound_stride != 0 && bound_stride < n) { set_error("mir_optim_b200: bound_stride must be 0 or >= n"); return MIR_B200_EINVAL; }
    return MIR_B200_OK;
}

template <class T>
int covariance_dev(const typename Num<T>::Settings* settings, const mir_model_desc* model, size_t batch, size_t m, size_t n,
                   const T* x, const T* l, const T* u, size_t bound_stride, unsigned covFlags, T* cov, T* stddev, int32_t* info,
                   cudaStream_t stream)
{
    clear_error();
    if (int rc = cov_check<T>(model, m, n, cov, stddev)) return rc;
    if (batch == 0) return MIR_B200_OK;
    if (int rc = cov_check_data<T>(model, batch, m, x, l, u, n, bound_stride, info)) return rc;
    if (batch >= 0xffffffffull) { set_error("mir_optim_b200: at most 2^32 - 2 problems per launch"); return MIR_B200_EINVAL; }
    if (int rc = require_device(-1)) return rc;
    typename Num<T>::Settings defaults;
    if (!settings) {
        if constexpr (sizeof(T) == 8) mir_least_squares_init_d(&defaults); else mir_least_squares_init_s(&defaults);
        settings = &defaults;
    }
    unsigned int* counter = nullptr;
    MIRB200_CUDA(cudaMallocAsync((void**)&counter, sizeof(unsigned int), stream));
    MIRB200_CUDA(cudaMemsetAsync(counter, 0, sizeof(unsigned int), stream));
    CovArgs ca;
    ca.t = model->t; ca.y = model->y; ca.x = x; ca.l = l; ca.u = u; ca.aux = model->aux; ca.param = model->param;
    ca.cov = cov; ca.stddev = stddev; ca.info = info; ca.counter = counter; ca.scratch = nullptr; ca.scratch_stride = 0;
    ca.batch = batch; ca.m = (unsigned)m; ca.n = (unsigned)n; ca.bound_stride = (unsigned)bound_stride;
    ca.flags = model->flags; ca.unscaled = (covFlags & MIR_COV_UNSCALED) ? 1u : 0u;
    ca.w = (model->flags & MIR_MODEL_WEIGHTED) ? model->w : nullptr;
    const int rc = launch_cov_model<T>(*model, settings->jacobianEpsilon, ca, stream);
    cudaFreeAsync(counter, stream);
    return rc;
}

template <class T>
int covariance_host(const typename Num<T>::Settings* settings, const mir_model_desc* model, size_t batch, size_t m, size_t n,
                    const T* x, const T* l, const T* u, size_t bound_stride, unsigned covFlags, T* cov, T* stddev, int32_t* info,
                    int device)
{
    clear_error();
    if (int rc = cov_check<T>(model, m, n, cov, stddev)) return rc;
    if (batch) { if (int rc = cov_check_data<T>(model, batch, m, x, l, u, n, bound_stride, info)) return rc; }
    if (int rc = require_device(device)) return rc;
    if (batch == 0) return MIR_B200_OK;

    const bool per = (model->flags & MIR_MODEL_GRID_PER_PROBLEM) != 0;
    const size_t tBytes = model->t ? sizeof(T) * (per ? batch * m : m) : 0;
    const size_t yBytes = model->y ? sizeof(T) * batch * m : 0;
    const size_t wBytes = (model->flags & MIR_MODEL_WEIGHTED) ? sizeof(T) * batch * m : 0;
    const size_t aBytes = model->aux ? sizeof(T) * ((model->flags & MIR_MODEL_AUX_PER_PROBLEM) ? batch * n : n) : 0;
    const size_t xBytes = sizeof(T) * batch * n;
    const size_t bBytes = sizeof(T) * (bound_stride ? batch * bound_stride : n);
    const size_t cBytes = cov ? sizeof(T) * batch * n * n : 0;
    const size_t sBytes = stddev ? sizeof(T) * batch * n : 0;
    const size_t iBytes = sizeof(int32_t) * batch;
    auto align = [](size_t v) { return (v + 255) & ~(size_t)255; };
    const size_t total = align(tBytes) + align(yBytes) + align(wBytes) + align(aBytes) + align(xBytes) + 2 * align(bBytes) + align(cBytes) + align(sBytes) + align(iBytes);

    cudaStream_t s = nullptr;
    MIRB200_CUDA(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
    int rc = MIR_B200_OK;
    auto CK = [&](cudaError_t err, const char* what) { if (rc == MIR_B200_OK) rc = check_cuda(err, what); };
    char* base = nullptr;
    CK(cudaMallocAsync((void**)&base, total, s), "cudaMallocAsync(covariance buffers)");
    if (rc == MIR_B200_OK) {
        char* p = base;
        T* dt = (T*)p; p += align(tBytes);
        T* dy = (T*)p; p += align(yBytes);
        T* dw = (T*)p; p += align(wBytes);
        T* da = (T*)p; p += align(aBytes);
        T* dx = (T*)p; p += align(xBytes);
        T* dl = (T*)p; p += align(bBytes);
        T* du = (T*)p; p += align(bBytes);
        T* dc = (T*)p; p += align(cBytes);
        T* ds = (T*)p; p += align(sBytes);
        int32_t* di = (int32_t*)p;
        if (tBytes) CK(cudaMemcpyAsync(dt, model->t, tBytes, cudaMemcpyHostToDevice, s), "H2D t");
        if (yBytes) CK(cudaMemcpyAsync(dy, model->y, yBytes, cudaMemcpyHostToDevice, s), "H2D y");
        if (wBytes) CK(cudaMemcpyAsync(dw, model->w, wBytes, cudaMemcpyHostToDevice, s), "H2D w");
        if (aBytes) CK(cudaMemcpyAsync(da, model->aux, aBytes, cudaMemcpyHostToDevice, s), "H2D aux");
        CK(cudaMemcpyAsync(dx, x, xBytes, cudaMemcpyHostToDevice, s), "H2D x");
        CK(cudaMemcpyAsync(dl, l, bBytes, cudaMemcpyHostToDevice, s), "H2D l");
        CK(cudaMemcpyAsync(du, u, bBytes, cudaMemcpyHostToDevice, s), "H2D u");
        mir_model_desc dm = *model;
        dm.t = tBytes ? dt : nullptr; dm.y = yBytes ? dy : nullptr; dm.aux = aBytes ? da : nullptr; dm.w = wBytes ? dw : nullptr;
        if (rc == MIR_B200_OK)
            rc = covariance_dev<T>(settings, &dm, batch, m, n, dx, dl, du, bound_stride, covFlags, cov ? dc : nullptr, stddev ? ds : nullptr, di, s);
        if (rc == MIR_B200_OK) {
            if (cBytes) CK(cudaMemcpyAsync(cov, dc, cBytes, cudaMemcpyDeviceToHost, s), "D2H cov");
            if (sBytes) CK(cudaMemcpyAsync(stddev, ds, sBytes, cudaMemcpyDeviceToHost, s), "D2H stddev");
            CK(cudaMemcpyAsync(info, di, iBytes, cudaMemcpyDeviceToHost, s), "D2H info");
        }
        cudaFreeAsync(base, s);
    }
    const cudaError_t se = cudaStreamSynchronize(s);
    if (rc == MIR_B200_OK) rc = check_cuda(se, "covariance kernel");
    cudaStreamDestroy(s);
    return rc;
}

}  // namespace

template <class T>
int launch_cov_model(const mir_model_desc& model, T jacEps, CovArgs ca, cudaStream_t stream)
{
    if (model.model >= (uint32_t)MIR_MODEL_USER_BASE) return launch_user_cov<T>(model, jacEps, ca, stream);
    if (model.flags & MIR_MODEL_WEIGHTED) return launch_cov_builtin<T, true>(model, jacEps, ca, kNoCovModel, stream);
    return launch_cov_builtin<T, false>(model, jacEps, ca, kNoCovModel, stream);
}
template int launch_cov_model<double>(const mir_model_desc&, double, CovArgs, cudaStream_t);
template int launch_cov_model<float>(const mir_model_desc&, float, CovArgs, cudaStream_t);

}  // namespace mirb200

using namespace mirb200;

extern "C" {

int mir_b200_covariance_batched_d(const mir_least_squares_settings_d* settings, const mir_model_desc* model, size_t batch, size_t m,
    size_t n, const double* x, const double* l, const double* u, size_t bound_stride, unsigned cov_flags, double* cov, double* stddev,
    int32_t* info, int device)
{ return covariance_host<double>(settings, model, batch, m, n, x, l, u, bound_stride, cov_flags, cov, stddev, info, device); }

int mir_b200_covariance_batched_s(const mir_least_squares_settings_s* settings, const mir_model_desc* model, size_t batch, size_t m,
    size_t n, const float* x, const float* l, const float* u, size_t bound_stride, unsigned cov_flags, float* cov, float* stddev,
    int32_t* info, int device)
{ return covariance_host<float>(settings, model, batch, m, n, x, l, u, bound_stride, cov_flags, cov, stddev, info, device); }

int mir_b200_covariance_batched_dev_d(const mir_least_squares_settings_d* settings, const mir_model_desc* model, size_t batch, size_t m,
    size_t n, const double* x, const double* l, const double* u, size_t bound_stride, unsigned cov_flags, double* cov, double* stddev,
    int32_t* info, void* cuda_stream)
{ return covariance_dev<double>(settings, model, batch, m, n, x, l, u, bound_stride, cov_flags, cov, stddev, info, (cudaStream_t)cuda_stream); }

int mir_b200_covariance_batched_dev_s(const mir_least_squares_settings_s* settings, const mir_model_desc* model, size_t batch, size_t m,
    size_t n, const float* x, const float* l, const float* u, size_t bound_stride, unsigned cov_flags, float* cov, float* stddev,
    int32_t* info, void* cuda_stream)
{ return covariance_dev<float>(settings, model, batch, m, n, x, l, u, bound_stride, cov_flags, cov, stddev, info, (cudaStream_t)cuda_stream); }

}  // extern "C"
