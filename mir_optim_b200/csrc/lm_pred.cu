// lm_pred.cu -- C ABI of the batched prediction entry points (mir_b200_predict_batched_*): argument checks, staging of
// host buffers, and the launch of lm_pred_cta_kernel (lm_pred.cuh) for the built-in models, with the model table
// (visit_cta_model) and the launch policy (launch_persistent) of the general batched LM kernel.
#include "lm_pred.cuh"
#include "runtime.cuh"

namespace mirb200 {

namespace {

constexpr const char* kNoPredModel = "mir_optim_b200: model id not available for the prediction (it has no run-time-n functor)";

// argument checks shared by both forms (batch may be 0; data pointers are checked by the caller when batch > 0), in the
// order of the covariance's (lm_cov.cu)
template <class T>
int pred_check(const mir_model_desc* model, size_t k, size_t n, const void* cov, const void* value, const void* se)
{
    if (!model) { set_error("mir_optim_b200: null model"); return MIR_B200_EINVAL; }
    if (!value && !se) { set_error("mir_optim_b200: value and se are both NULL: nothing to compute"); return MIR_B200_EINVAL; }
    if (se && !cov) { set_error("mir_optim_b200: se needs cov"); return MIR_B200_EINVAL; }
    if (n == 0 || k == 0) { set_error("mir_optim_b200: k and n must be > 0"); return MIR_B200_EINVAL; }
    if (n > 128) { set_error("mir_optim_b200: the prediction supports n <= 128"); return MIR_B200_EUNSUPPORTED; }
    if (k >= 0x7fffffffull) { set_error("mir_optim_b200: k too large"); return MIR_B200_EUNSUPPORTED; }
    if (model->model >= (uint32_t)MIR_MODEL_USER_BASE) return MIR_B200_OK;      // checked when the model is loaded
    return visit_cta_model<T>(*model, kNoPredModel, [&](auto tag) {
        using M = typename decltype(tag)::type;
        if (!M::valid((int)n, (int)k + (CtaTrailingRow<M>::value ? 1 : 0))) { set_error("mir_optim_b200: (k, n) not valid for this model"); return (int)MIR_B200_EINVAL; }
        return (int)MIR_B200_OK;
    });
}

template <class T>
int pred_check_data(const mir_model_desc* model, const T* x, const T* l, const T* u, size_t n, size_t bound_stride)
{
    if (!x || !l || !u) { set_error("mir_optim_b200: null argument"); return MIR_B200_EINVAL; }
    if (model->model < (uint32_t)MIR_MODEL_USER_BASE && !model->t) {    // (the data-free built-in models are rejected above)
        set_error("mir_optim_b200: this model reads abscissae: model->t must not be NULL"); return MIR_B200_EINVAL;
    }
    if (bound_stride != 0 && bound_stride < n) { set_error("mir_optim_b200: bound_stride must be 0 or >= n"); return MIR_B200_EINVAL; }
    return MIR_B200_OK;
}

template <class T>
int predict_dev(const typename Num<T>::Settings* settings, const mir_model_desc* model, size_t batch, size_t k, size_t n,
                const T* x, const T* l, const T* u, size_t bound_stride, const T* cov, T* value, T* se, cudaStream_t stream)
{
    clear_error();
    if (int rc = pred_check<T>(model, k, n, cov, value, se)) return rc;
    if (batch == 0) return MIR_B200_OK;
    if (int rc = pred_check_data<T>(model, x, l, u, n, bound_stride)) return rc;
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
    PredArgs pa;
    pa.t = model->t; pa.x = x; pa.l = l; pa.u = u; pa.aux = model->aux; pa.param = model->param;
    pa.cov = se ? cov : nullptr; pa.value = value; pa.se = se; pa.counter = counter; pa.scratch = nullptr; pa.scratch_stride = 0;
    pa.batch = batch; pa.k = (unsigned)k; pa.n = (unsigned)n; pa.bound_stride = (unsigned)bound_stride;
    pa.flags = model->flags & (MIR_MODEL_FD_JACOBIAN | MIR_MODEL_GRID_PER_PROBLEM | MIR_MODEL_AUX_PER_PROBLEM);   // y and w are not read
    const int rc = launch_pred_model<T>(*model, settings->jacobianEpsilon, pa, stream);
    cudaFreeAsync(counter, stream);
    return rc;
}

template <class T>
int predict_host(const typename Num<T>::Settings* settings, const mir_model_desc* model, size_t batch, size_t k, size_t n,
                 const T* x, const T* l, const T* u, size_t bound_stride, const T* cov, T* value, T* se, int device)
{
    clear_error();
    if (int rc = pred_check<T>(model, k, n, cov, value, se)) return rc;
    if (batch) { if (int rc = pred_check_data<T>(model, x, l, u, n, bound_stride)) return rc; }
    if (int rc = require_device(device)) return rc;
    if (batch == 0) return MIR_B200_OK;

    const bool per = (model->flags & MIR_MODEL_GRID_PER_PROBLEM) != 0;
    const size_t tBytes = model->t ? sizeof(T) * (per ? batch * k : k) : 0;
    const size_t aBytes = model->aux ? sizeof(T) * ((model->flags & MIR_MODEL_AUX_PER_PROBLEM) ? batch * n : n) : 0;
    const size_t xBytes = sizeof(T) * batch * n;
    const size_t bBytes = sizeof(T) * (bound_stride ? batch * bound_stride : n);
    const size_t cBytes = se ? sizeof(T) * batch * n * n : 0;
    const size_t vBytes = value ? sizeof(T) * batch * k : 0;
    const size_t sBytes = se ? sizeof(T) * batch * k : 0;
    auto align = [](size_t v) { return (v + 255) & ~(size_t)255; };
    const size_t total = align(tBytes) + align(aBytes) + align(xBytes) + 2 * align(bBytes) + align(cBytes) + align(vBytes) + align(sBytes);

    cudaStream_t s = nullptr;
    MIRB200_CUDA(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
    int rc = MIR_B200_OK;
    auto CK = [&](cudaError_t err, const char* what) { if (rc == MIR_B200_OK) rc = check_cuda(err, what); };
    char* base = nullptr;
    CK(cudaMallocAsync((void**)&base, total, s), "cudaMallocAsync(prediction buffers)");
    if (rc == MIR_B200_OK) {
        char* p = base;
        T* dt = (T*)p; p += align(tBytes);
        T* da = (T*)p; p += align(aBytes);
        T* dx = (T*)p; p += align(xBytes);
        T* dl = (T*)p; p += align(bBytes);
        T* du = (T*)p; p += align(bBytes);
        T* dc = (T*)p; p += align(cBytes);
        T* dv = (T*)p; p += align(vBytes);
        T* ds = (T*)p;
        if (tBytes) CK(cudaMemcpyAsync(dt, model->t, tBytes, cudaMemcpyHostToDevice, s), "H2D t");
        if (aBytes) CK(cudaMemcpyAsync(da, model->aux, aBytes, cudaMemcpyHostToDevice, s), "H2D aux");
        CK(cudaMemcpyAsync(dx, x, xBytes, cudaMemcpyHostToDevice, s), "H2D x");
        CK(cudaMemcpyAsync(dl, l, bBytes, cudaMemcpyHostToDevice, s), "H2D l");
        CK(cudaMemcpyAsync(du, u, bBytes, cudaMemcpyHostToDevice, s), "H2D u");
        if (cBytes) CK(cudaMemcpyAsync(dc, cov, cBytes, cudaMemcpyHostToDevice, s), "H2D cov");
        mir_model_desc dm = *model;
        dm.t = tBytes ? dt : nullptr; dm.y = nullptr; dm.aux = aBytes ? da : nullptr; dm.w = nullptr;
        if (rc == MIR_B200_OK)
            rc = predict_dev<T>(settings, &dm, batch, k, n, dx, dl, du, bound_stride, se ? dc : nullptr, value ? dv : nullptr, se ? ds : nullptr, s);
        if (rc == MIR_B200_OK) {
            if (vBytes) CK(cudaMemcpyAsync(value, dv, vBytes, cudaMemcpyDeviceToHost, s), "D2H value");
            if (sBytes) CK(cudaMemcpyAsync(se, ds, sBytes, cudaMemcpyDeviceToHost, s), "D2H se");
        }
        cudaFreeAsync(base, s);
    }
    const cudaError_t serr = cudaStreamSynchronize(s);
    if (rc == MIR_B200_OK) rc = check_cuda(serr, "prediction kernel");
    cudaStreamDestroy(s);
    return rc;
}

}  // namespace

template <class T>
int launch_pred_model(const mir_model_desc& model, T jacEps, PredArgs pa, cudaStream_t stream)
{
    if (model.model >= (uint32_t)MIR_MODEL_USER_BASE) return launch_user_pred<T>(model, jacEps, pa, stream);
    return visit_cta_model<T>(model, kNoPredModel, [&](auto tag) {
        using M = typename decltype(tag)::type;
        const bool fd = (model.flags & MIR_MODEL_FD_JACOBIAN) || !M::kAnalytic;
        const void* fn = fd ? (const void*)lm_pred_cta_kernel<M, T, true> : (const void*)lm_pred_cta_kernel<M, T, false>;
        return launch_pred<T>(RuntimeKernel{fn, "lm_pred_cta_kernel launch"}, jacEps, pa, M::prep_elems((int)pa.n), stream);
    });
}
template int launch_pred_model<double>(const mir_model_desc&, double, PredArgs, cudaStream_t);
template int launch_pred_model<float>(const mir_model_desc&, float, PredArgs, cudaStream_t);

}  // namespace mirb200

using namespace mirb200;

extern "C" {

int mir_b200_predict_batched_d(const mir_least_squares_settings_d* settings, const mir_model_desc* model, size_t batch, size_t k,
    size_t n, const double* x, const double* l, const double* u, size_t bound_stride, const double* cov, double* value, double* se,
    int device)
{ return predict_host<double>(settings, model, batch, k, n, x, l, u, bound_stride, cov, value, se, device); }

int mir_b200_predict_batched_s(const mir_least_squares_settings_s* settings, const mir_model_desc* model, size_t batch, size_t k,
    size_t n, const float* x, const float* l, const float* u, size_t bound_stride, const float* cov, float* value, float* se,
    int device)
{ return predict_host<float>(settings, model, batch, k, n, x, l, u, bound_stride, cov, value, se, device); }

int mir_b200_predict_batched_dev_d(const mir_least_squares_settings_d* settings, const mir_model_desc* model, size_t batch, size_t k,
    size_t n, const double* x, const double* l, const double* u, size_t bound_stride, const double* cov, double* value, double* se,
    void* cuda_stream)
{ return predict_dev<double>(settings, model, batch, k, n, x, l, u, bound_stride, cov, value, se, (cudaStream_t)cuda_stream); }

int mir_b200_predict_batched_dev_s(const mir_least_squares_settings_s* settings, const mir_model_desc* model, size_t batch, size_t k,
    size_t n, const float* x, const float* l, const float* u, size_t bound_stride, const float* cov, float* value, float* se,
    void* cuda_stream)
{ return predict_dev<float>(settings, model, batch, k, n, x, l, u, bound_stride, cov, value, se, (cudaStream_t)cuda_stream); }

}  // extern "C"
