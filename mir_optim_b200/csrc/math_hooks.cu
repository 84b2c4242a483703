// math_hooks.cu -- the device math of repro_math.cuh exposed on its own, so that tests can hold every form of the
// reproducible exp against the host restatement (oracle/repro_math.h) bit for bit, and the Cholesky pivot step against a
// high-precision reference, without going through a fit:
//   variant 0   exp_repro_tp             early returns, immediates (models_large.cuh, user models)
//   variant 1   exp_repro                the __noinline__ copy (exp_sel<false>: lane-group, CTA and covariance kernels)
//   variant 2   exp_repro_inl            exp_repro_many<1> inlined (exp_sel<true>)
//   variant 3   exp_repro_many<4>        each thread takes 4 consecutive inputs
//   variant 4   exp_repro_many<16>       each thread takes 16 consecutive inputs (lm_tpp.cuh's widest interleave)
//   variant 5   exp_repro_many_conv<4>   each warp takes 32*4 consecutive inputs, lane l the 4 from 4*l on, so the caller
//   variant 6   exp_repro_many_conv<16>  decides which warps see only |x| < 700 (< 80 in float) and take the fast path
//   variant 7   mux_sqrt_rcp             l = sqrt(a) to y, r = 1/sqrt(a) to y2 (lm_mux.cuh's pivot step)
// Inputs past the end of x are read as 0 and their results dropped; the conv variants always run whole warps.
// Diagnostics, not a hot path: host pointers, synchronous.
#include "repro_math.cuh"
#include "runtime.cuh"

namespace mirb200 {

constexpr int MATH_HOOK_THREADS = 256;

template <class T, int V>
__global__ void __launch_bounds__(MATH_HOOK_THREADS) math_scalar_kernel(size_t n, const T* __restrict__ x, T* __restrict__ y, T* __restrict__ y2)
{
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const T a = x[i];
        if constexpr (V == 0) y[i] = exp_repro_tp(a);
        else if constexpr (V == 1) y[i] = exp_repro(a);
        else if constexpr (V == 2) y[i] = exp_repro_inl(a);
        else { T l, r; mux_sqrt_rcp(a, l, r); y[i] = l; y2[i] = r; }
    }
}

// CONV = false: thread t owns x[K*t, K*t + K).  CONV = true: warp w owns x[32*K*w, 32*K*(w + 1)), lane l the K inputs from
// 32*K*w + K*l; the loop bound is uniform across the warp, so all 32 lanes reach the vote together.
template <class T, int K, bool CONV>
__global__ void __launch_bounds__(MATH_HOOK_THREADS) math_many_kernel(size_t n, const T* __restrict__ x, T* __restrict__ y)
{
    const size_t groups = (n + K - 1) / K;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    const size_t end = CONV ? (groups + 31) / 32 * 32 : groups;
    for (size_t g = (size_t)blockIdx.x * blockDim.x + threadIdx.x; g < end; g += stride) {
        T a[K], e[K];
#pragma unroll
        for (int j = 0; j < K; ++j) { const size_t i = g * K + j; a[j] = i < n ? x[i] : (T)0; }
        if constexpr (CONV) exp_repro_many_conv<K>(a, e); else exp_repro_many<K>(a, e);
#pragma unroll
        for (int j = 0; j < K; ++j) { const size_t i = g * K + j; if (i < n) y[i] = e[j]; }
    }
}

template <class T>
static int math_hook(int variant, size_t n, const T* x, T* y, T* y2, int device)
{
    clear_error();
    if (variant < 0 || variant > 7) {
        set_error("mir_optim_b200: math hook: variant must be 0..7 (0-2 scalar exp, 3-4 exp_repro_many<4|16>, "
                  "5-6 exp_repro_many_conv<4|16>, 7 mux_sqrt_rcp)");
        return MIR_B200_EUNSUPPORTED;
    }
    if (n && (!x || !y || (variant == 7 && !y2))) { set_error("mir_optim_b200: null argument (variant 7 needs y2 as well)"); return MIR_B200_EINVAL; }
    int rc = require_device(device);
    if (rc) return rc;
    if (n == 0) return MIR_B200_OK;
    cudaStream_t stream = nullptr;
    MIRB200_CUDA(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
    const size_t bytes = sizeof(T) * n, abytes = (bytes + 255) & ~(size_t)255;
    char* base = nullptr;
    cudaError_t e = cudaMallocAsync((void**)&base, (variant == 7 ? 3 : 2) * abytes, stream);
    if (e != cudaSuccess) { cudaStreamDestroy(stream); return check_cuda(e, "cudaMallocAsync(math hook buffers)"); }
    T* dx = (T*)base; T* dy = (T*)(base + abytes); T* dy2 = variant == 7 ? (T*)(base + 2 * abytes) : nullptr;
    auto CK = [&](cudaError_t err, const char* what) { if (rc == MIR_B200_OK) rc = check_cuda(err, what); };
    CK(cudaMemcpyAsync(dx, x, bytes, cudaMemcpyHostToDevice, stream), "H2D x");
    if (rc == MIR_B200_OK) {
        const int K = (variant == 3 || variant == 5) ? 4 : (variant == 4 || variant == 6) ? 16 : 1;
        const size_t threads = variant >= 5 && variant <= 6 ? ((n + K - 1) / K + 31) / 32 * 32 : (n + K - 1) / K;
        const unsigned grid = (unsigned)std::min<size_t>((threads + MATH_HOOK_THREADS - 1) / MATH_HOOK_THREADS, 148 * 32);
        switch (variant) {
        case 0: math_scalar_kernel<T, 0><<<grid, MATH_HOOK_THREADS, 0, stream>>>(n, dx, dy, dy2); break;
        case 1: math_scalar_kernel<T, 1><<<grid, MATH_HOOK_THREADS, 0, stream>>>(n, dx, dy, dy2); break;
        case 2: math_scalar_kernel<T, 2><<<grid, MATH_HOOK_THREADS, 0, stream>>>(n, dx, dy, dy2); break;
        case 3: math_many_kernel<T, 4, false><<<grid, MATH_HOOK_THREADS, 0, stream>>>(n, dx, dy); break;
        case 4: math_many_kernel<T, 16, false><<<grid, MATH_HOOK_THREADS, 0, stream>>>(n, dx, dy); break;
        case 5: math_many_kernel<T, 4, true><<<grid, MATH_HOOK_THREADS, 0, stream>>>(n, dx, dy); break;
        case 6: math_many_kernel<T, 16, true><<<grid, MATH_HOOK_THREADS, 0, stream>>>(n, dx, dy); break;
        default: math_scalar_kernel<T, 7><<<grid, MATH_HOOK_THREADS, 0, stream>>>(n, dx, dy, dy2); break;
        }
        count_launch();
        CK(cudaGetLastError(), "math hook launch");
    }
    if (rc == MIR_B200_OK) CK(cudaMemcpyAsync(y, dy, bytes, cudaMemcpyDeviceToHost, stream), "D2H y");
    if (rc == MIR_B200_OK && variant == 7) CK(cudaMemcpyAsync(y2, dy2, bytes, cudaMemcpyDeviceToHost, stream), "D2H y2");
    cudaFreeAsync(base, stream);
    cudaError_t se = cudaStreamSynchronize(stream);
    if (rc == MIR_B200_OK) rc = check_cuda(se, "math hook kernel");
    cudaStreamDestroy(stream);
    return rc;
}

}  // namespace mirb200

extern "C" {
int mir_b200_math_hook_d(int variant, size_t n, const double* x, double* y, double* y2, int device)
{ return mirb200::math_hook<double>(variant, n, x, y, y2, device); }
int mir_b200_math_hook_s(int variant, size_t n, const float* x, float* y, float* y2, int device)
{ return mirb200::math_hook<float>(variant, n, x, y, y2, device); }
}
