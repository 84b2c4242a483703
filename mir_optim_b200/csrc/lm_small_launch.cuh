// lm_small_launch.cuh -- host-side launcher for lm_small_kernel: picks the rows-per-lane
// instantiation from m, sizes a persistent grid (a multiple of the SM count) and enqueues.
#pragma once
#include <cstdlib>
#include <cstring>
#include "lm_small.cuh"
#include "lm_tpp.cuh"
#include "lm_mux.cuh"
#include "runtime.cuh"

namespace mirb200 {

template <class Model, class T, int LANES, int R, bool FD>
int launch_small_fd(const typename Num<T>::Settings& st, const SmallBatchArgs& args, cudaStream_t stream)
{
    auto kern = lm_small_kernel<Model, T, LANES, R, FD>;
    int blocksPerSM = 0;
    MIRB200_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&blocksPerSM, kern, 128, 0));
    if (blocksPerSM < 1) blocksPerSM = 1;
    const unsigned long long groupsPerBlock = 128 / LANES;
    unsigned long long blocksWanted = (args.batch + groupsPerBlock - 1) / groupsPerBlock;
    unsigned long long grid = (unsigned long long)sm_count() * blocksPerSM;     // persistent: one resident wave
    if (blocksWanted < grid) grid = blocksWanted ? blocksWanted : 1;
    kern<<<(unsigned)grid, 128, 0, stream>>>(st, args);
    count_launch();
    return check_cuda(cudaGetLastError(), "lm_small_kernel launch");
}

template <class Model, class T, int LANES, int R>
int launch_small_one(const typename Num<T>::Settings& st, const SmallBatchArgs& args, cudaStream_t stream)
{
    return (args.flags & MIR_MODEL_FD_JACOBIAN) ? launch_small_fd<Model, T, LANES, R, true>(st, args, stream)
                                                : launch_small_fd<Model, T, LANES, R, false>(st, args, stream);
}

// Thread-per-problem kernel (lm_tpp.cuh): any m; used for large batches, where one thread per problem fills the GPU.
template <class Model, class T, bool FD, bool YOS, bool VL>
int launch_tpp_cfg(const typename Num<T>::Settings& st, const SmallBatchArgs& args, cudaStream_t stream)
{
    auto kern = lm_tpp_kernel<Model, T, FD, YOS, VL>;
    int blocksPerSM = 0;
    const size_t mPad = ((size_t)args.m + 1) & ~(size_t)1;
    // shared abscissa (+ observations) (+ the accepted steps of the v-list)
    const size_t smem = sizeof(T) * (mPad + (YOS ? (size_t)args.m * TPP_THREADS : 0) + (VL ? (size_t)TPP_VLN * Model::N * TPP_THREADS : 0));
    if (smem > 200 * 1024) { set_error("mir_optim_b200: m too large for the thread-per-problem kernel"); return MIR_B200_EUNSUPPORTED; }
    if (smem > 48 * 1024) MIRB200_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    MIRB200_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&blocksPerSM, kern, TPP_THREADS, smem));
    if (blocksPerSM < 1) blocksPerSM = 1;
    unsigned long long blocksWanted = (args.batch + TPP_THREADS - 1) / TPP_THREADS;
    unsigned long long grid = (unsigned long long)sm_count() * blocksPerSM;
    if (blocksWanted < grid) grid = blocksWanted ? blocksWanted : 1;
    const size_t perThread = (size_t)args.m * TppSlab<Model::N, YOS, VL>::ELEMS;
    T* slab = nullptr;
    MIRB200_CUDA(cudaMallocAsync((void**)&slab, sizeof(T) * (perThread ? perThread : 1) * TPP_THREADS * grid, stream));
    kern<<<(unsigned)grid, TPP_THREADS, smem, stream>>>(st, args, slab);
    count_launch();
    const int rc = check_cuda(cudaGetLastError(), "lm_tpp_kernel launch");
    cudaFreeAsync(slab, stream);
    return rc;
}
template <class Model, class T, bool FD>
int launch_tpp_fd(const typename Num<T>::Settings& st, const SmallBatchArgs& args, cudaStream_t stream)
{
    // observations in shared memory while two CTAs per SM still fit (m * 128 threads * sizeof(T) <= ~100 KB)
    const bool yos = Model::kHasData && sizeof(T) * ((size_t)args.m + TPP_VLN * Model::N) * TPP_THREADS <= 100 * 1024;
    if constexpr (!FD) {
        // analytic Jacobian with the default maxAge (3, LS:945) or a smaller one: the v-list scheme (no stored Jacobian)
        if ((st.maxAge ? st.maxAge : 3u) <= (unsigned)TPP_VLN)
            return yos ? launch_tpp_cfg<Model, T, FD, true, true>(st, args, stream) : launch_tpp_cfg<Model, T, FD, false, true>(st, args, stream);
    }
    return yos ? launch_tpp_cfg<Model, T, FD, true, false>(st, args, stream) : launch_tpp_cfg<Model, T, FD, false, false>(st, args, stream);
}
template <class Model, class T>
int launch_tpp(const typename Num<T>::Settings& st, const SmallBatchArgs& args, cudaStream_t stream)
{
    return (args.flags & MIR_MODEL_FD_JACOBIAN) ? launch_tpp_fd<Model, T, true>(st, args, stream) : launch_tpp_fd<Model, T, false>(st, args, stream);
}

// Four problems per warp (lm_mux.cuh): n <= 8, m <= 128.  One warp per CTA; the warp's four problems live in its shared memory.
template <class Model, class T, bool FD, int MUX_WARPS>
int launch_mux_w(const typename Num<T>::Settings& st, const SmallBatchArgs& args, cudaStream_t stream)
{
    auto kern = lm_mux_kernel<Model, T, FD, MUX_WARPS>;
    const size_t smem = sizeof(MuxCtaSmem<T, MUX_WARPS>);
    static bool attrSet = false;       // (per instantiation)
    if (!attrSet) {
        MIRB200_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        MIRB200_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
        attrSet = true;
    }
    int blocksPerSM = 0;
    MIRB200_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&blocksPerSM, kern, 32 * MUX_WARPS, smem));
    if (blocksPerSM < 1) blocksPerSM = 1;
    const unsigned long long perBlock = (unsigned long long)MUX_SLOTS * MUX_WARPS;
    unsigned long long blocksWanted = (args.batch + perBlock - 1) / perBlock;
    unsigned long long grid = (unsigned long long)sm_count() * blocksPerSM;      // persistent: one resident wave
    if (blocksWanted < grid) grid = blocksWanted ? blocksWanted : 1;
    kern<<<(unsigned)grid, 32 * MUX_WARPS, smem, stream>>>(st, args);
    count_launch();
    return check_cuda(cudaGetLastError(), "lm_mux_kernel launch");
}
// Warps per CTA: as many as the shared memory of one SM holds (5 in double, 10 in float), stepping through the phases
// together (lm_mux.cuh); batches too small to fill those CTAs run in single-warp CTAs.
template <class Model, class T, bool FD>
int launch_mux_fd(const typename Num<T>::Settings& st, const SmallBatchArgs& args, cudaStream_t stream)
{
    constexpr int W = sizeof(T) == 8 ? 5 : 10;          // as many warps as the shared memory of one SM holds, in ONE CTA
    constexpr int WH = sizeof(T) == 8 ? 2 : 5;          // two CTAs per SM (they drift out of phase: one in the n-sized phase, one on rows)
    if (args.batch >= (unsigned long long)MUX_SLOTS * W * 2) {
        // float: two CTAs of 5 warps per SM measured 4.78 M fits/s against 4.50 M for one CTA of 10 (the two drift out of
        // phase and overlap the latency-bound n-sized phase of one with the FP-heavy row phase of the other); double has 5
        // warps per SM, which do not split: 2 x 2 warps measured 0.99 M against 1.10 M for one CTA of 5
        if constexpr (sizeof(T) == 4) return launch_mux_w<Model, T, FD, WH>(st, args, stream);
        else return launch_mux_w<Model, T, FD, W>(st, args, stream);
    }
    return launch_mux_w<Model, T, FD, 1>(st, args, stream);
}
template <class Model, class T>
int launch_mux(const typename Num<T>::Settings& st, const SmallBatchArgs& args, cudaStream_t stream)
{
    return (args.flags & MIR_MODEL_FD_JACOBIAN) ? launch_mux_fd<Model, T, true>(st, args, stream) : launch_mux_fd<Model, T, false>(st, args, stream);
}

// Kernel choice: one thread per problem once the batch can fill the GPU with threads, else one lane group per
// problem (more parallelism inside each problem).
inline bool use_thread_per_problem(unsigned long long batch)
{
    return batch >= 16384ull;
}

// Rs...: the rows-per-lane instantiations compiled for this model, ascending.
template <class Model, class T, int LANES, int... Rs>
int launch_small(const typename Num<T>::Settings& st, const SmallBatchArgs& args, cudaStream_t stream)
{
    int rc = MIR_B200_EUNSUPPORTED;
    bool done = false;
    // pick the first R with R*LANES >= m
    (void)std::initializer_list<int>{
        ((!done && (unsigned)(Rs * LANES) >= args.m) ? (done = true, rc = launch_small_one<Model, T, LANES, Rs>(st, args, stream), 0) : 0)...};
    if (!done) set_error("mir_optim_b200: m is larger than the batched small-problem kernels support for this model");
    return rc;
}

// Entry used by the C ABI (lm_batched.cu); one explicit instantiation per precision lives in
// lm_small_inst_{d,s}.cu so the two precisions compile in parallel.
template <class T>
int launch_small_model(unsigned model, size_t n, const typename Num<T>::Settings& st, const SmallBatchArgs& args, cudaStream_t stream);

}  // namespace mirb200
