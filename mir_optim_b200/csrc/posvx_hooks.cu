// posvx_hooks.cu -- the device restatements of LAPACK ?posvx('E','L') (boxcqp.d:194-205, 310-321 call it) exposed on
// their own, so that tests can hold them against the real LAPACK routine without going through BOXCQP or LM:
//   variant 0   posvx_small  (registers, compile-time n <= 8; the batched LM kernels)
//   variant 1   cta_posvx    column loop, 128 threads  (the batched BoxQP kernel)
//   variant 2   cta_posvx    blocked register-tiled LDL^T, 256 threads  (the control kernel of the large-problem path)
//   variant 3   posvx_warp   one warp per system, n <= 64  (the warp-per-QP BoxQP kernel, boxqp_warp.cuh)
//   variant 4   posvx_dist   one 8-lane group per system, four systems per warp, n <= 8  (lm_mux.cuh)
// Outputs per system: x, info (0, or k > 0 = factorisation broke down at pivot k; the condition estimate behind LAPACK's
// info = n + 1 is not computed -- boxcqp.d:212/323 accepts it -- so such systems report 0) and the equilibration
// decision (LAPACK's EQUED = 'Y').  Diagnostics, not a hot path: host pointers, synchronous.
#include "boxqp_cta.cuh"
#include "boxqp_warp.cuh"
#include "lm_mux.cuh"
#include "runtime.cuh"

namespace mirb200 {

template <class T> struct PosvxArgs { const T* A; const T* b; T* x; int32_t* info; int32_t* equed; unsigned batch; int n; };

template <class T, int N>
__global__ void posvx_small_kernel(const PosvxArgs<T> a)
{
    const unsigned p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= a.batch) return;
    constexpr int NP = N * (N + 1) / 2;
    T JJ[NP], b[N], x[N];
    const T* A = a.A + (size_t)p * N * N;
#pragma unroll
    for (int i = 0; i < N; ++i) {
        b[i] = a.b[(size_t)p * N + i];
        x[i] = (T)0;
#pragma unroll
        for (int j = 0; j <= i; ++j) JJ[tri(i, j)] = A[i * N + j];
    }
    bool eq = false;
    const int info = posvx_small<T, N>(JJ, (T)0, FullMask<N>::value, b, x, &eq);
#pragma unroll
    for (int i = 0; i < N; ++i) a.x[(size_t)p * N + i] = x[i];
    a.info[p] = info; a.equed[p] = eq ? 1 : 0;
}

template <class T, int NT, bool BLK>
__global__ void __launch_bounds__(NT) posvx_cta_kernel(const PosvxArgs<T> a)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int n = a.n, tid = threadIdx.x;
    CtaQPScratch<T> w;
    w.carve(smem_raw, n);
    T* sx = reinterpret_cast<T*>(smem_raw + ((CtaQPScratch<T>::bytes(n) + 15) & ~(size_t)15));
    __shared__ int s_eq;
    for (unsigned p = blockIdx.x; p < a.batch; p += gridDim.x) {
        const T* Ag = a.A + (size_t)p * n * n;
        __syncthreads();
        for (int i = tid; i < n; i += NT) { w.b[i] = a.b[(size_t)p * n + i]; sx[i] = (T)0; }
        if (tid == 0) s_eq = 0;
        __syncthreads();
        auto A = [&](int i, int j) -> T { return Ag[(size_t)i * n + j]; };
        const int info = cta_posvx<T, NT, BLK>(n, A, w, w.b, sx, &s_eq);
        __syncthreads();
        for (int i = tid; i < n; i += NT) a.x[(size_t)p * n + i] = sx[i];
        if (tid == 0) { a.info[p] = info; a.equed[p] = s_eq; }
    }
}

// variant 3: one warp per system
template <class T>
__global__ void __launch_bounds__(32) posvx_warp_kernel(const PosvxArgs<T> a)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    WarpQPSmem<T>& sm = *reinterpret_cast<WarpQPSmem<T>*>(smem_raw);
    __shared__ int s_eq;
    const int n = a.n, lane = threadIdx.x;
    for (unsigned p = blockIdx.x; p < a.batch; p += gridDim.x) {
        const T* Ag = a.A + (size_t)p * n * n;
        __syncwarp();
        for (int i = lane; i < n; i += 32) sm.b[i] = a.b[(size_t)p * n + i];
        if (lane == 0) s_eq = 0;
        __syncwarp();
        auto A = [&](int i, int j) -> T { return Ag[(size_t)i * n + j]; };
        const int info = posvx_warp<T>(n, A, sm, lane, &s_eq);
        __syncwarp();
        for (int i = lane; i < n; i += 32) a.x[(size_t)p * n + i] = info ? (T)0 : sm.sx[i];
        if (lane == 0) { a.info[p] = info; a.equed[p] = s_eq; }
    }
}

// variant 4: four systems per warp, lane gl of a group owns row gl
template <class T>
__global__ void __launch_bounds__(32) posvx_dist_kernel(const PosvxArgs<T> a)
{
    const int n = a.n, lane = threadIdx.x, grp = lane >> 3, gl = lane & 7;
    const unsigned p = blockIdx.x * 4 + grp;
    const bool have = p < a.batch;
    T Prow[MUX_G];
    T Pdiag = (T)1, b = (T)0;
#pragma unroll
    for (int j = 0; j < MUX_G; ++j) {
        // symmetric read through the lower triangle (what BOXCQP hands to ?posvx, boxcqp.d:186-188)
        const bool in = have && gl < n && j < n;
        const T v = in ? (gl >= j ? a.A[(size_t)p * n * n + gl * n + j] : a.A[(size_t)p * n * n + j * n + gl]) : (T)0;
        Prow[j] = v;
        if (j == gl) Pdiag = in ? v : (T)1;
    }
    if (have && gl < n) b = a.b[(size_t)p * n + gl];
    T x = (T)0;
    const unsigned free = (1u << n) - 1u;
    const int info = posvx_dist<T>(have, gl, Prow, Pdiag, free, b, x);
    if (have && gl < n) a.x[(size_t)p * n + gl] = info ? (T)0 : x;
    // the ?laqsy decision is not an output of posvx_dist: recompute it the way posvx_small does, for the comparison
    T smin = gmin8((have && gl < n) ? Pdiag : Num<T>::inf()), amax = gmax8((have && gl < n) ? Pdiag : -Num<T>::inf());
    bool equil = false;
    if (smin > (T)0) equil = !(div_ni(sqrt_ni(smin), sqrt_ni(amax)) >= (T)0.1 && amax >= Num<T>::small_() && amax <= Num<T>::large_());
    if (have && gl == 0) { a.info[p] = info; a.equed[p] = equil ? 1 : 0; }
}

template <class T, int N> static void launch_small_n(int n, const PosvxArgs<T>& a, cudaStream_t s)
{
    if constexpr (N >= 1) {
        if (n == N) { posvx_small_kernel<T, N><<<(a.batch + 63) / 64, 64, 0, s>>>(a); count_launch(); }
        else launch_small_n<T, N - 1>(n, a, s);
    }
}

template <class T>
static int posvx_batched(int variant, size_t batch, size_t n, const T* A, const T* b, T* x, int32_t* info, int32_t* equed, int device)
{
    clear_error();
    if (batch && (!A || !b || !x || !info || !equed)) { set_error("mir_optim_b200: null argument"); return MIR_B200_EINVAL; }
    if (n == 0 || n > 128 || ((variant == 0 || variant == 4) && n > 8) || (variant == 3 && n > (size_t)WQP_NMAX) || variant < 0 || variant > 4) {
        set_error("mir_optim_b200: posvx hook: variants 0 and 4 take 1 <= n <= 8, variant 3 takes n <= 64, variants 1 and 2 take 1 <= n <= 128");
        return MIR_B200_EUNSUPPORTED;
    }
    int rc = require_device(device);
    if (rc) return rc;
    if (batch == 0) return MIR_B200_OK;
    cudaStream_t stream = nullptr;
    MIRB200_CUDA(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
    auto align = [](size_t v) { return (v + 255) & ~(size_t)255; };
    const size_t aB = sizeof(T) * batch * n * n, vB = sizeof(T) * batch * n, iB = 4 * batch;
    char* base = nullptr;
    cudaError_t e = cudaMallocAsync((void**)&base, align(aB) + 2 * align(vB) + 2 * align(iB), stream);
    if (e != cudaSuccess) { cudaStreamDestroy(stream); return check_cuda(e, "cudaMallocAsync(posvx buffers)"); }
    char* p = base;
    PosvxArgs<T> a;
    T* dA = (T*)p; p += align(aB); T* db = (T*)p; p += align(vB); T* dx = (T*)p; p += align(vB);
    int32_t* di = (int32_t*)p; p += align(iB); int32_t* de = (int32_t*)p;
    a.A = dA; a.b = db; a.x = dx; a.info = di; a.equed = de; a.batch = (unsigned)batch; a.n = (int)n;
    auto CK = [&](cudaError_t err, const char* what) { if (rc == MIR_B200_OK) rc = check_cuda(err, what); };
    CK(cudaMemcpyAsync(dA, A, aB, cudaMemcpyHostToDevice, stream), "H2D A");
    CK(cudaMemcpyAsync(db, b, vB, cudaMemcpyHostToDevice, stream), "H2D b");
    if (rc == MIR_B200_OK) {
        const size_t smem = ((CtaQPScratch<T>::bytes((int)n) + 15) & ~(size_t)15) + sizeof(T) * n;
        const unsigned grid = (unsigned)(batch < 4096 ? batch : 4096);
        if (variant == 0) launch_small_n<T, 8>((int)n, a, stream);
        else if (variant == 1) {
            CK(cudaFuncSetAttribute(posvx_cta_kernel<T, 128, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem), "smem attribute");
            posvx_cta_kernel<T, 128, false><<<grid, 128, smem, stream>>>(a); count_launch();
        } else if (variant == 3) {
            CK(cudaFuncSetAttribute(posvx_warp_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(WarpQPSmem<T>)), "smem attribute");
            posvx_warp_kernel<T><<<grid, 32, sizeof(WarpQPSmem<T>), stream>>>(a); count_launch();
        } else if (variant == 4) {
            posvx_dist_kernel<T><<<(unsigned)((batch + 3) / 4), 32, 0, stream>>>(a); count_launch();
        } else {
            CK(cudaFuncSetAttribute(posvx_cta_kernel<T, 256, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem), "smem attribute");
            posvx_cta_kernel<T, 256, true><<<grid, 256, smem, stream>>>(a); count_launch();
        }
        CK(cudaGetLastError(), "posvx hook launch");
    }
    if (rc == MIR_B200_OK) {
        CK(cudaMemcpyAsync(x, dx, vB, cudaMemcpyDeviceToHost, stream), "D2H x");
        CK(cudaMemcpyAsync(info, di, iB, cudaMemcpyDeviceToHost, stream), "D2H info");
        CK(cudaMemcpyAsync(equed, de, iB, cudaMemcpyDeviceToHost, stream), "D2H equed");
    }
    cudaFreeAsync(base, stream);
    cudaError_t se = cudaStreamSynchronize(stream);
    if (rc == MIR_B200_OK) rc = check_cuda(se, "posvx hook kernel");
    cudaStreamDestroy(stream);
    return rc;
}

}  // namespace mirb200

extern "C" {
int mir_b200_posvx_batched_d(int variant, size_t batch, size_t n, const double* A, const double* b, double* x, int32_t* info, int32_t* equed, int device)
{ return mirb200::posvx_batched<double>(variant, batch, n, A, b, x, info, equed, device); }
int mir_b200_posvx_batched_s(int variant, size_t batch, size_t n, const float* A, const float* b, float* x, int32_t* info, int32_t* equed, int device)
{ return mirb200::posvx_batched<float>(variant, batch, n, A, b, x, info, equed, device); }
}
