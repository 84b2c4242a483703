// boxqp_batched.cu -- batched BOXCQP (BASELINE configs[4]a).  n <= 64: one WARP per QP (boxqp_warp.cuh: no barriers, packed
// factor in shared memory, P read in place); 64 < n <= 128: one CTA per QP, P's lower triangle, the factor and all vectors in
// shared memory.  Persistent warps / CTAs pull QP indices from an atomic counter.
// C ABI: mir_solve_box_qp_{d,s}, mir_solve_box_qp_batched[_dev]_{d,s}  (solveBoxQP, boxcqp.d:85-102 / 122-379).
#include "boxqp_cta.cuh"
#include "boxqp_warp.cuh"
#include "runtime.cuh"

namespace mirb200 {

template <class T> struct QPBatchArgs {
    const T* P; const T* q; const T* l; const T* u; T* x;
    int32_t* status; uint32_t* iterations;
    unsigned int* counter;
    unsigned int batch; int n;
    typename Num<T>::QPSettings st;
};

// A_SMEM: stage the lower triangle of P in shared memory (n <= ~88 in double); otherwise read P through L1/L2.
template <class T, int NT, bool A_SMEM>
__global__ void __launch_bounds__(NT) boxqp_cta_kernel(const QPBatchArgs<T> a)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int n = a.n, tid = threadIdx.x;
    CtaQPScratch<T> w;
    w.carve(smem_raw, n);
    T* vec = reinterpret_cast<T*>(smem_raw + ((CtaQPScratch<T>::bytes(n) + 15) & ~(size_t)15));
    T* sq = vec; T* sl = vec + n; T* su = vec + 2 * n; T* sx = vec + 3 * n;
    T* sA = vec + 4 * n;                       // n x lda, only used when A_SMEM
    const int lda = n + 8;
    __shared__ unsigned int s_prob;

    for (;;) {
        __syncthreads();
        if (tid == 0) s_prob = atomicAdd(a.counter, 1u);
        __syncthreads();
        const unsigned int prob = s_prob;
        if (prob >= a.batch) break;
        const T* Pg = a.P + (size_t)prob * n * n;
        for (int i = tid; i < n; i += NT) {
            sq[i] = a.q[(size_t)prob * n + i]; sl[i] = a.l[(size_t)prob * n + i]; su[i] = a.u[(size_t)prob * n + i];
            sx[i] = (T)0;
        }
        if (A_SMEM) {
            // coalesced row-major sweep; the strict upper triangle is never read (boxcqp.d:288-302, 335) but is
            // copied along because rows are contiguous
            for (int e = tid; e < n * n; e += NT) { const int r = e / n, c = e - r * n; sA[r * lda + c] = Pg[e]; }
        }
        __syncthreads();
        unsigned iters = 0, solves = 0;
        int st;
        if (A_SMEM) {
            auto P = [&](int i, int j) -> T { return sA[i * lda + j]; };
            st = cta_boxqp<T, NT, false>(a.st, n, P, sq, sl, su, sx, w, iters, solves);
        } else {
            auto P = [&](int i, int j) -> T { return __ldg(Pg + (size_t)i * n + j); };
            st = cta_boxqp<T, NT, false>(a.st, n, P, sq, sl, su, sx, w, iters, solves);
        }
        __syncthreads();
        for (int i = tid; i < n; i += NT) a.x[(size_t)prob * n + i] = sx[i];
        if (tid == 0) { a.status[prob] = st; if (a.iterations) a.iterations[prob] = iters; }
    }
}

// One warp (= one CTA) per QP, n <= 64.
template <class T>
__global__ void __launch_bounds__(32) boxqp_warp_kernel(const QPBatchArgs<T> a)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    WarpQPSmem<T>& sm = *reinterpret_cast<WarpQPSmem<T>*>(smem_raw);
    const int n = a.n, lane = threadIdx.x;
    for (;;) {
        unsigned int prob = 0;
        if (lane == 0) prob = atomicAdd(a.counter, 1u);
        prob = __shfl_sync(0xffffffffu, prob, 0);
        if (prob >= a.batch) break;
        const T* Pg = a.P + (size_t)prob * n * n;
        __syncwarp();
        for (int i = lane; i < n; i += 32) {
            sm.q[i] = a.q[(size_t)prob * n + i]; sm.l[i] = a.l[(size_t)prob * n + i]; sm.u[i] = a.u[(size_t)prob * n + i];
            sm.x[i] = (T)0;
        }
        __syncwarp();
        unsigned iters = 0, solves = 0;
        const int st = boxqp_warp<T>(a.st, n, Pg, sm, lane, iters, solves);
        __syncwarp();
        for (int i = lane; i < n; i += 32) a.x[(size_t)prob * n + i] = sm.x[i];
        if (lane == 0) { a.status[prob] = st; if (a.iterations) a.iterations[prob] = iters; }
    }
}

template <class T> static size_t qp_smem_bytes(int n, bool a_smem)
{
    size_t b = ((CtaQPScratch<T>::bytes(n) + 15) & ~(size_t)15) + sizeof(T) * 4 * (size_t)n;
    if (a_smem) b += sizeof(T) * (size_t)n * (n + 8);
    return b;
}

template <class T>
static int qp_batched_dev(const typename Num<T>::QPSettings* settings, size_t batch, size_t n, const T* P, const T* q, const T* l,
                          const T* u, T* x, int32_t* status, uint32_t* iterations, cudaStream_t stream)
{
    clear_error();
    if (batch && (!P || !q || !l || !u || !x || !status)) { set_error("mir_optim_b200: null argument"); return MIR_B200_EINVAL; }
    if (batch == 0) return MIR_B200_OK;
    if (n == 0 || n > 128) { set_error("mir_optim_b200: batched BoxQP supports 1 <= n <= 128"); return n == 0 ? MIR_B200_EINVAL : MIR_B200_EUNSUPPORTED; }
    if (batch >= 0xffffffffull) { set_error("mir_optim_b200: at most 2^32 - 2 problems per launch"); return MIR_B200_EINVAL; }
    int rc = require_device(-1);
    if (rc) return rc;
    constexpr int NT = 128;
    typename Num<T>::QPSettings def;
    def.relTolerance = def.absTolerance = (T)16 * (std::is_same<T, double>::value ? (T)2.220446049250313e-16 : (T)1.1920929e-7f);
    def.maxIterations = 0;

    QPBatchArgs<T> a;
    a.P = P; a.q = q; a.l = l; a.u = u; a.x = x; a.status = status; a.iterations = iterations;
    a.batch = (unsigned)batch; a.n = (int)n; a.st = settings ? *settings : def;
    MIRB200_CUDA(cudaMallocAsync((void**)&a.counter, sizeof(unsigned int), stream));
    MIRB200_CUDA(cudaMemsetAsync(a.counter, 0, sizeof(unsigned int), stream));

    if (n <= (size_t)WQP_NMAX) {
        auto wk = boxqp_warp_kernel<T>;
        const size_t wsmem = sizeof(WarpQPSmem<T>);
        MIRB200_CUDA(cudaFuncSetAttribute(wk, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)wsmem));
        MIRB200_CUDA(cudaFuncSetAttribute(wk, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
        int perSM = 0;
        MIRB200_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&perSM, wk, 32, wsmem));
        if (perSM < 1) perSM = 1;
        size_t grid = (size_t)sm_count() * perSM;
        if (batch < grid) grid = batch;
        wk<<<(unsigned)grid, 32, wsmem, stream>>>(a);
        count_launch();
        rc = check_cuda(cudaGetLastError(), "boxqp_warp_kernel launch");
        cudaFreeAsync(a.counter, stream);
        return rc;
    }
    const bool a_smem = qp_smem_bytes<T>((int)n, true) <= 100 * 1024;       // >= 2 CTAs per SM
    const size_t smem = qp_smem_bytes<T>((int)n, a_smem);
    auto kern = a_smem ? boxqp_cta_kernel<T, NT, true> : boxqp_cta_kernel<T, NT, false>;
    MIRB200_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int perSM = 0;
    MIRB200_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&perSM, kern, NT, smem));
    if (perSM < 1) perSM = 1;
    size_t grid = (size_t)sm_count() * perSM;
    if (batch < grid) grid = batch;
    kern<<<(unsigned)grid, NT, smem, stream>>>(a);
    count_launch();
    rc = check_cuda(cudaGetLastError(), "boxqp_cta_kernel launch");
    cudaFreeAsync(a.counter, stream);
    return rc;
}

template <class T>
static int qp_batched_host(const typename Num<T>::QPSettings* settings, size_t batch, size_t n, const T* P, const T* q, const T* l,
                           const T* u, T* x, int32_t* status, uint32_t* iterations, int device)
{
    clear_error();
    if (batch && (!P || !q || !l || !u || !x || !status)) { set_error("mir_optim_b200: null argument"); return MIR_B200_EINVAL; }
    int rc = require_device(device);
    if (rc) return rc;
    if (batch == 0) return MIR_B200_OK;
    cudaStream_t stream = nullptr;
    MIRB200_CUDA(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
    auto align = [](size_t v) { return (v + 255) & ~(size_t)255; };
    const size_t pB = sizeof(T) * batch * n * n, vB = sizeof(T) * batch * n, sB = 4 * batch;
    char* base = nullptr;
    cudaError_t e = cudaMallocAsync((void**)&base, align(pB) + 4 * align(vB) + 2 * align(sB), stream);
    if (e != cudaSuccess) { cudaStreamDestroy(stream); return check_cuda(e, "cudaMallocAsync(qp buffers)"); }
    char* p = base;
    T* dP = (T*)p; p += align(pB);
    T* dq = (T*)p; p += align(vB); T* dl = (T*)p; p += align(vB); T* du = (T*)p; p += align(vB); T* dx = (T*)p; p += align(vB);
    int32_t* ds = (int32_t*)p; p += align(sB); uint32_t* di = (uint32_t*)p;
    auto CK = [&](cudaError_t err, const char* what) { if (rc == MIR_B200_OK) rc = check_cuda(err, what); };
    CK(cudaMemcpyAsync(dP, P, pB, cudaMemcpyHostToDevice, stream), "H2D P");
    CK(cudaMemcpyAsync(dq, q, vB, cudaMemcpyHostToDevice, stream), "H2D q");
    CK(cudaMemcpyAsync(dl, l, vB, cudaMemcpyHostToDevice, stream), "H2D l");
    CK(cudaMemcpyAsync(du, u, vB, cudaMemcpyHostToDevice, stream), "H2D u");
    if (rc == MIR_B200_OK) rc = qp_batched_dev<T>(settings, batch, n, dP, dq, dl, du, dx, ds, di, stream);
    if (rc == MIR_B200_OK) {
        CK(cudaMemcpyAsync(x, dx, vB, cudaMemcpyDeviceToHost, stream), "D2H x");
        CK(cudaMemcpyAsync(status, ds, sB, cudaMemcpyDeviceToHost, stream), "D2H status");
        if (iterations) CK(cudaMemcpyAsync(iterations, di, sB, cudaMemcpyDeviceToHost, stream), "D2H iterations");
    }
    cudaFreeAsync(base, stream);
    cudaError_t se = cudaStreamSynchronize(stream);
    if (rc == MIR_B200_OK) rc = check_cuda(se, "batched BoxQP kernel");
    cudaStreamDestroy(stream);
    return rc;
}

}  // namespace mirb200

using namespace mirb200;

extern "C" {

int mir_solve_box_qp_batched_d(const mir_box_qp_settings_d* s, size_t batch, size_t n, const double* P, const double* q, const double* l,
                               const double* u, double* x, int32_t* status, uint32_t* it, int device)
{ return qp_batched_host<double>(s, batch, n, P, q, l, u, x, status, it, device); }
int mir_solve_box_qp_batched_s(const mir_box_qp_settings_s* s, size_t batch, size_t n, const float* P, const float* q, const float* l,
                               const float* u, float* x, int32_t* status, uint32_t* it, int device)
{ return qp_batched_host<float>(s, batch, n, P, q, l, u, x, status, it, device); }
int mir_solve_box_qp_batched_dev_d(const mir_box_qp_settings_d* s, size_t batch, size_t n, const double* P, const double* q, const double* l,
                                   const double* u, double* x, int32_t* status, uint32_t* it, void* stream)
{ return qp_batched_dev<double>(s, batch, n, P, q, l, u, x, status, it, (cudaStream_t)stream); }
int mir_solve_box_qp_batched_dev_s(const mir_box_qp_settings_s* s, size_t batch, size_t n, const float* P, const float* q, const float* l,
                                   const float* u, float* x, int32_t* status, uint32_t* it, void* stream)
{ return qp_batched_dev<float>(s, batch, n, P, q, l, u, x, status, it, (cudaStream_t)stream); }

/* solveBoxQP simple overload, boxcqp.d:85-102.  Returns BoxQPStatus, or -mir_b200_error when the device is unusable. */
int mir_solve_box_qp_d(const mir_box_qp_settings_d* s, size_t n, const double* P, const double* q, const double* l, const double* u, double* x)
{
    if (n == 0) return mir_qp_solved;          /* boxcqp.d:162-163 */
    int32_t st = mir_qp_numericError;
    const int rc = qp_batched_host<double>(s, 1, n, P, q, l, u, x, &st, nullptr, -1);
    return rc ? -rc : st;
}
int mir_solve_box_qp_s(const mir_box_qp_settings_s* s, size_t n, const float* P, const float* q, const float* l, const float* u, float* x)
{
    if (n == 0) return mir_qp_solved;
    int32_t st = mir_qp_numericError;
    const int rc = qp_batched_host<float>(s, 1, n, P, q, l, u, x, &st, nullptr, -1);
    return rc ? -rc : st;
}

}  // extern "C"
