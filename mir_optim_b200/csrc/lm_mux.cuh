// lm_mux.cuh -- batched Levenberg-Marquardt for problems with up to 8 parameters and up to 128 residuals
// (BASELINE configs[2]: 8-parameter sums of exponentials, finite-difference Jacobian), four problems per warp.
// Follows optimizeLeastSquaresImplGeneric!T, least_squares.d:877-1176, and solveBoxQP, boxcqp.d:122-379 (cites inline).
//
// At n = 8 the n-sized part of a pass (8 x 8 ?posvx + BOXCQP + lambda control) is as long as the m-sized part, one
// thread cannot hold an 8 x 8 system plus an 8-column Jacobian, and a warp per problem runs the n-sized part 32 times
// redundantly.  Each phase therefore gets the lane layout that suits it, and ONE WARP (= one CTA) carries four problems
// ("slots") whose whole state lives in its 44 KB of shared memory:
//
//   * ROW phases (residual evaluation, finite-difference / analytic Jacobian, Broyden update LS:999-1006, J^T y and
//     J^T J, LS:1052, 1065) are WARP-cooperative: all 32 lanes work on ONE slot at a time, lane L owning rows L, L+32,
//     L+64, L+96.  The slots of a CTA post their row requests into a shared-memory queue and the CTA's warps pull
//     them one by one, whichever slot they belong to: the row work of a pass is spread evenly over the warps.  Jacobian, current and trial residuals live
//     in shared memory ([parameter][row], pitch 132: conflict-free for the row accesses, the column writes of the finite
//     differences and the tensor-core fragment loads); the observations are re-read from global memory (L2) per evaluation.
//     J^T J runs on the FP64 TENSOR pipe: mma.sync.m8n8k4.f64 (DMMA) takes J^T (8 x 4 rows) as A and the same values as B,
//     32 MMAs per 128 rows, the 8 x 8 result arrives distributed over the warp -- no cross-lane reduction of 36 sums.
//     J^T y rides along on the same fragment loads (one FMA per MMA, two shuffles at the end).
//   * N-SIZED phases run in four 8-lane GROUPS at once, group g on slot g, lane i owning parameter i: row i of the
//     system matrix, x_i, its bounds, its multipliers.  The ?posvx restatement is a right-looking Cholesky with one
//     broadcast per pivot / column element; BOXCQP's per-variable logic (flags, multipliers, KBN right-hand side,
//     BQ:239-347) is lane-parallel, its any / all tests are ballots.  Control flow in these phases is WARP-UNIFORM:
//     every shuffle / ballot uses the full mask (width 8) and groups that do not take part are predicated off, so the
//     compiler emits plain SHFL / VOTE instructions instead of a convergence loop per collective.
//   * All exponentials of the kernel go through ONE inlined exp_repro_many block inside ONE loop ("evaluation items":
//     initial / trial residuals and the 2n evaluations of a finite-difference Jacobian), and the two row phases of a
//     pass share one copy of the code (the pass loop is folded in two halves): the kernel is a few thousand
//     instructions instead of 11,000 (round-2 ncu of the first version: stall_no_instruction 6.7 of 12 cycles per issue).
//   * Models whose finite-difference evaluations share sub-expressions say so (Model::kFDShared): for a sum of
//     exponentials, perturbing one parameter changes one term, so the other terms' exps are computed once per Jacobian
//     instead of 2n times -- the same operations on the same operands, hence the same bits, 12 exps per row instead of 64.
//
// Equivalences (bit-exact w.r.t. this file's own arithmetic, as in lm_small.cuh): J^T J is rebuilt only when J changed;
// a trial point equal to x skips the evaluation (fCalls still counts it); the provably inert lambda-overflow tail is
// replayed as a scalar recurrence (tail_is_inert, lm_small.cuh -- restated here for the distributed layout).
#pragma once
#include <type_traits>
#include "lm_small.cuh"

namespace mirb200 {

constexpr int MUX_SLOTS = 4;            // problems per warp
constexpr int MUX_G = 8;                // lanes per problem in the n-sized phases: n <= 8
constexpr int MUX_R = 4;                // rows per lane in the row phases (row = lane + 32 k): m <= 128
constexpr int MUX_MMAX = 32 * MUX_R;
constexpr int MUX_JP = MUX_MMAX + 4;    // pitch of one Jacobian column in shared memory
constexpr unsigned MUX_FULL = 0xffffffffu;
// Warps per CTA.  1: every warp is its own CTA and runs free.  > 1: the warps of a CTA (one CTA per SM, as many warps
// as shared memory holds) step through the phases of the pass loop TOGETHER (a CTA barrier after every phase): they
// share nothing but the instruction cache, which then holds one phase's code for all of them instead of thrashing
// between five warps in five different phases.
// (template parameter MUX_WARPS of the kernel)
enum { MUX_EVAL_INIT = 1, MUX_EVAL_TRIAL = 2, MUX_JAC_FRESH = 4, MUX_JAC_BROYDEN = 8 };

// Everything a problem ("slot") keeps between phases, in shared memory of its CTA.
template <class T> struct MuxSlot {
    T J[MUX_G][MUX_JP];                 // Jacobian, [parameter][row]; parameters >= n and rows >= m stay zero
    T vec[2][MUX_MMAX];                 // y (current residuals) and mBuffer (trial / previous residuals); `ysel` says which is which
    T JJ[MUX_G * MUX_G];                // J^T J, full symmetric storage, undamped
    T Jy[MUX_G];                        // J^T y
    // row-task mailbox: written by the slot's group before a row phase, read by whichever warp takes the task
    T p[MUX_G];                         // the point to evaluate at (trial point or x)
    T dX[MUX_G];                        // accepted step (Broyden)
    T fxp[MUX_G], fxm[MUX_G], frt[MUX_G];   // finite differences: x + h, x - h, 1 / (2h) per parameter
    T ddot, result;                     // |dX|^2; ||r||^2 of the evaluation (written by the row phase)
    unsigned long long prob;
    int flags, ysel;
};
struct MuxQueue {
    int qn[2], qhead[2];                // row-task queues of the two halves of the pass loop: length, next task
    int retired;                        // warps of the CTA that have run out of problems (exit consensus)
    unsigned char qtask[2][MUX_SLOTS * 16];
};
template <class T, int W> struct MuxCtaSmem {
    MuxSlot<T> slot[MUX_SLOTS * W];
    MuxQueue q;
};

// ---- group (8-lane) collectives, executed by the whole warp; every lane of a group receives the same bits -----------
template <class T> __device__ __forceinline__ T gshfl(T v, int src) { return __shfl_sync(MUX_FULL, v, src, MUX_G); }
template <class T> __device__ __forceinline__ T gmax8(T v)
{
#pragma unroll
    for (int off = MUX_G / 2; off > 0; off >>= 1) v = t_max(v, __shfl_xor_sync(MUX_FULL, v, off, MUX_G));
    return v;
}
template <class T> __device__ __forceinline__ T gmin8(T v)
{
#pragma unroll
    for (int off = MUX_G / 2; off > 0; off >>= 1) v = t_min(v, __shfl_xor_sync(MUX_FULL, v, off, MUX_G));
    return v;
}
template <class T> __device__ __forceinline__ T gsum8(T v)
{
#pragma unroll
    for (int off = MUX_G / 2; off > 0; off >>= 1) v += __shfl_xor_sync(MUX_FULL, v, off, MUX_G);
    return v;
}
__device__ __forceinline__ bool gall8(bool p, int gshift) { return ((__ballot_sync(MUX_FULL, p) >> gshift) & 0xffu) == 0xffu; }
__device__ __forceinline__ bool gany8(bool p, int gshift) { return ((__ballot_sync(MUX_FULL, p) >> gshift) & 0xffu) != 0u; }

__device__ __forceinline__ void mux_dmma884(double (&c)[2], double a, double b)
{
    asm("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};" : "+d"(c[0]), "+d"(c[1]) : "d"(a), "d"(b));
}

// ---------------------------------------------------------------------------------------------------------------------
// LAPACK ?posvx(FACT='E', UPLO='L') as called at boxcqp.d:194-205 / 310-321, distributed over the 8 lanes of a group:
// lane gl owns row gl of the system.  Steps as in posvx_small (boxqp_small.cuh): ?poequ / ?laqsy over the free rows,
// Cholesky, ?potrs, ?porfs refinement (<= 5 sweeps on the componentwise backward error), un-scaling.  Rows / columns
// whose bit is clear in `free` (fixed variables of the active set, and lanes >= n) are pinned to the identity, so the
// free entries see exactly the operands of the compacted system plus exact zeros.
//   Prow   row gl of P = J^T J + lambda I (all 8 columns, unmasked), Pdiag = Prow[gl]
//   part   this group takes part (the others run along on whatever they hold; their results are ignored)
// Executed by all 32 lanes in lock step.  Returns LAPACK info (0, or k > 0: factorisation broke down at pivot k),
// uniform over the group.
// ---------------------------------------------------------------------------------------------------------------------
template <class T>
__device__ __forceinline__ int posvx_dist(bool part, int gl, const T (&Prow)[MUX_G], T Pdiag, unsigned free, T b_in, T& x_out)
{
    constexpr int G = MUX_G;
    const bool fi = (free >> gl) & 1u;
    T a[G], a0[G];
#pragma unroll
    for (int j = 0; j < G; ++j) {
        const bool fj = (free >> j) & 1u;
        a[j] = (fi && fj) ? Prow[j] : ((j == gl) ? (T)1 : (T)0);
    }
    T b = fi ? b_in : (T)0;
    const T d = fi ? Pdiag : (T)1;
    // ?poequ over the free rows, ?laqsy decision: equilibrate iff scond = sqrt(smin) / sqrt(amax) < 0.1 or amax is out of
    // range.  Single precision settles it unless the ratio is within 10 % of the threshold (or the diagonal leaves the
    // float range); only then the exact minimum / maximum and the two square roots are computed.
    bool equil = false;
    {
        const float df = (float)d;
        float fmin_ = fi ? df : __builtin_huge_valf(), fmax_ = fi ? df : 0.0f;
#pragma unroll
        for (int off = MUX_G / 2; off > 0; off >>= 1) {
            fmin_ = fminf(fmin_, __shfl_xor_sync(MUX_FULL, fmin_, off, MUX_G));
            fmax_ = fmaxf(fmax_, __shfl_xor_sync(MUX_FULL, fmax_, off, MUX_G));
        }
        const bool clearlyFine = fmin_ >= 0.011f * fmax_ && fmin_ > 0x1p-100f && fmax_ < 0x1p100f;
        if (__any_sync(MUX_FULL, part && !clearlyFine)) {
            const T smin = gmin8(fi ? d : Num<T>::inf());
            const T amax = gmax8(fi ? d : -Num<T>::inf());
            if (part && smin > (T)0) {
                bool wellScaled;                       // the roots only near the boundary
                if (smin >= (T)0.0102 * amax) wellScaled = true;
                else if (smin <= (T)0.0098 * amax) wellScaled = false;
                else wellScaled = div_ni(sqrt_ni(smin), sqrt_ni(amax)) >= (T)0.1;
                equil = !(wellScaled && amax >= Num<T>::small_() && amax <= Num<T>::large_());
            }
        }
    }
    T s = (T)1;
    if (__any_sync(MUX_FULL, equil)) {         // rare; groups that do not equilibrate scale by exactly 1
        if (equil && fi) s = rcp_ni(sqrt_ni(d));
#pragma unroll
        for (int j = 0; j < G; ++j) { const T sj = gshfl(s, j); a[j] = (sj * s) * a[j]; }          // dlaqsy: cj * s(i) * A(i,j)
        b = s * b;                                                                                 // dposvx: B := diag(S) B
    }
#pragma unroll
    for (int j = 0; j < G; ++j) a0[j] = a[j];

    // ?potrf, lower, right-looking: a[] becomes row gl of L (columns <= gl), ft[k] = L(k, gl) (row gl of L^T)
    T ft[G];
    T rinv = (T)0;
    int info = 0;
#pragma unroll
    for (int j = 0; j < G; ++j) ft[j] = (T)0;
#pragma unroll
    for (int j = 0; j < G; ++j) {
        const T ajj = gshfl(a[j], j);
        if (info == 0 && ajj <= (T)0) info = j + 1;     // breakdown (a NaN pivot passes through, as in OpenBLAS' potf2: `ajj <= 0`)
        T ljj, r;
        mux_sqrt_rcp(ajj, ljj, r);
        const T fij = a[j] * r;                // L(gl, j) for gl > j
        if (gl == j) { a[j] = ljj; rinv = r; } else a[j] = fij;
#pragma unroll
        for (int k = j + 1; k < G; ++k) {
            const T fk = gshfl(fij, k);        // L(k, j)
            a[k] = fma(-fij, fk, a[k]);        // a(gl, k) -= L(gl, j) L(k, j): the part k <= gl is the matrix, the rest is never read
            if (gl == j) ft[k] = fk;
        }
    }

    auto solve = [&](T v) -> T {               // L L^T z = v, lane gl in: v_gl, out: z_gl
        T acc = v;
#pragma unroll
        for (int k = 0; k < G; ++k) {
            const T cand = acc * rinv;
            const T vk = gshfl(cand, k);
            if (gl == k) acc = cand; else if (gl > k) acc = fma(-a[k], vk, acc);
        }
#pragma unroll
        for (int k = G - 1; k >= 0; --k) {
            const T cand = acc * rinv;
            const T xk = gshfl(cand, k);
            if (gl == k) acc = cand; else if (gl < k) acc = fma(-ft[k], xk, acc);
        }
        return acc;
    };

    // ?potrs, then ?porfs: pass 0 solves for b, later passes solve for the residual and correct x
    const int nfree = __popc(free & 0xffu);
    const T eps = Num<T>::lapack_eps();
    const T safe1 = (T)(nfree + 1) * Num<T>::safmin();
    const T safe2 = safe1 * ((T)1 / Num<T>::lapack_eps());
    T lstres = (T)3, x = (T)0, v = b;
    bool live = part && info == 0;
#pragma unroll 1
    for (int count = 0;; ++count) {
        const T z = solve(v);
        if (live) x += z;
        T r = b, w = t_abs(b);
#pragma unroll
        for (int j = 0; j < G; ++j) {
            const T xj = gshfl(x, j);
            r = fma(-a0[j], xj, r);
            w = fma(t_abs(a0[j]), t_abs(xj), w);
        }
        T qv = (T)0;                           // dporfs: berr = max_i |r_i| / (|b| + |A||x|)_i with the safe1 / safe2 guard
        if (fi) {
            const bool big = w > safe2;
            qv = div_ni(big ? t_abs(r) : t_abs(r) + safe1, big ? w : w + safe1);
        }
        const T berr = gmax8(qv);
        v = r;
        live = live && (berr > eps && (T)2 * berr <= lstres && count < 5);      // at most ITMAX = 5 corrections
        lstres = berr;
        if (!__any_sync(MUX_FULL, live)) break;
    }
    x_out = equil ? x * s : x;
    return info;
}

// solveBoxQP, boxcqp.d:122-379 (unconstrainedSolution = false) with P = J^T J + lambda I, lane gl owning variable gl.
// JJrow: row gl of the undamped J^T J.  q, l, u, x: this lane's entries (lanes >= n: q = 0, l = -inf, u = +inf).
// Executed by all 32 lanes in lock step; groups with act == false run along and return mir_qp_solved.
// Returns mir_box_qp_status, uniform over the group.
template <class T, int N>
__device__ __forceinline__ int boxqp_dist(bool act, int gl, int gshift, const typename Num<T>::QPSettings& st,
                                          const T (&JJrow)[MUX_G], T lambda, T q, T l, T u, T& x, QPCounters& cnt)
{
    constexpr int G = MUX_G;
    constexpr unsigned FULL = (1u << N) - 1u;
    const bool valid = gl < N;
    T Prow[G];
    T Pdiag = (T)0;
#pragma unroll
    for (int j = 0; j < G; ++j) {                                                        // LS:1078-1079: lambda on the diagonal
        Prow[j] = (j == gl) ? JJrow[j] + lambda : JJrow[j];
        Pdiag = (j == gl) ? Prow[j] : Pdiag;
    }
    const unsigned maxIterations = st.maxIterations ? st.maxIterations : (unsigned)N * 10u + 100u;   // BQ:224-226
    T b = -q, la = (T)0, mu = (T)0;                                                      // BQ:191, 231-232
    unsigned free = FULL, lo = 0, up = 0;
    bool first = true;
    unsigned step = 0;
    int res = act ? -1 : (int)mir_qp_solved;                                             // -1: still running
    x = (T)0;
#pragma unroll 1
    for (;;) {
        const bool doSolve = res < 0 && free != 0u;
        {
            T sx;
            const int info = posvx_dist<T>(doSolve, gl, Prow, Pdiag, free, b, sx);
            if (doSolve) {
                ++cnt.solves;
                if (info != 0) res = mir_qp_numericError;                                // BQ:212, 323
                else if ((free >> gl) & 1u) x = sx;                                      // BQ:327-329
            }
        }
        const bool wasFirst = first;
        const bool inAll = gall8(!valid || (l <= x && x <= u), gshift);
        if (res < 0 && first) {
            first = false;                                                               // BQ:216-219
            if (inAll) res = mir_qp_solved;
        }
        if (!__any_sync(MUX_FULL, res < 0)) break;
        if (__any_sync(MUX_FULL, res < 0 && !wasFirst)) {
            T d1 = (T)0, d2 = (T)0;                                                      // multipliers, BQ:333-337
#pragma unroll
            for (int j = 0; j < G; ++j) {
                const T xj = gshfl(x, j);
                if (j < gl) d1 = fma(Prow[j], xj, d1); else d2 = fma(Prow[j], xj, d2);
            }
            const T val = d1 + d2 + q;
            const bool mine = res < 0 && !wasFirst;
            bool bad = false;
            if (mine) {
                if ((lo >> gl) & 1u)      { la = val;  bad = !(val >= (T)0); }           // BQ:343
                else if ((up >> gl) & 1u) { mu = -val; bad = !(-val >= (T)0); }          // BQ:344
                else bad = valid && !(x >= l && x <= u);                                 // BQ:345
            }
            const bool anyBad = gany8(bad, gshift);
            if (mine) {
                if (!anyBad) { x = t_max(t_min(x, u), l); res = mir_qp_solved; }         // applyBounds, BQ:349
                else ++step;
            }
            if (!__any_sync(MUX_FULL, res < 0)) break;
        }
        if (res < 0 && step >= maxIterations) res = mir_qp_maxIterations;                // BQ:378
        const bool run = res < 0;
        if (run) ++cnt.iterations;
        int cls = 0;                                                                     // BQ:239-263
        if (run && valid) {
            const T xl = x - l, ux = u - x;
            if (xl < (T)0 || (xl < st.relTolerance + st.absTolerance * t_abs(l) && la >= (T)0)) { cls = 1; x = l; mu = (T)0; }
            else if (ux < (T)0 || (ux < st.relTolerance + st.absTolerance * t_abs(u) && mu >= (T)0)) { cls = 2; x = u; la = (T)0; }
            else { mu = (T)0; la = (T)0; }
        }
        const unsigned lon = (__ballot_sync(MUX_FULL, cls == 1) >> gshift) & FULL;
        const unsigned upn = (__ballot_sync(MUX_FULL, cls == 2) >> gshift) & FULL;
        if (run) {
            lo = lon; up = upn;
            free = FULL & ~(lo | up);
            if (free == FULL) res = mir_qp_maxIterations;                                // BQ:265-266: `break` falls out to :378
        }
        const unsigned fixed = lo | up;
        const T bound = (cls == 1) ? l : u;                                              // reduced right-hand side, BQ:282-305
        KBN<T> sum(q);
#pragma unroll
        for (int j = 0; j < G; ++j) {
            const T bj = gshfl(bound, j);
            if ((fixed >> j) & 1u) sum.put(mul_rn(Prow[j], bj));
        }
        if (res < 0) b = -sum.sum();
        if (!__any_sync(MUX_FULL, res < 0)) break;
    }
    return res;
}

template <class Model, class T, bool ON> struct SharedFD { struct State {}; static constexpr int CPI = 1; };
template <class Model, class T> struct SharedFD<Model, T, true> { using State = typename Model::template FDState<MUX_R>; static constexpr int CPI = Model::CPI; };

// MUX_WARPS warps per CTA walk the phases of the pass loop together (a CTA barrier after every phase) and pool their row
// work in one queue.
template <class Model, class T, bool FD, int MUX_WARPS>
__global__ void __launch_bounds__(32 * MUX_WARPS)
lm_mux_kernel(const typename Num<T>::Settings st, const SmallBatchArgs args)
{
    constexpr int N = Model::N, G = MUX_G, S = MUX_SLOTS, R = MUX_R, NE = Model::NE;
    static_assert(N <= G, "lm_mux_kernel: at most 8 parameters");
    static_assert(NE >= 1 && NE <= 4, "lm_mux_kernel: models with 1..4 exponentials per row");
    constexpr int KB = NE * R;                // exponentials per evaluation of my four rows (<= 16), interleaved in one exp block
    constexpr bool kShared = FD && Model::kFDShared;
    using Result = typename Num<T>::Result;
    extern __shared__ __align__(16) unsigned char mux_smem_raw[];
    using Cta = MuxCtaSmem<T, MUX_WARPS>;
    Cta& cta = *reinterpret_cast<Cta*>(mux_smem_raw);
    const int lane = threadIdx.x & 31;
    const int grp = lane >> 3, gl = lane & 7, gshift = grp * 8;
    const bool valid = gl < N;
    const int m = (int)args.m;
    const bool gridPerProblem = (args.flags & MIR_MODEL_GRID_PER_PROBLEM) != 0;
    const bool tailShortcut = (args.flags & MIR_MODEL_NO_TAIL_SHORTCUT) == 0;
    const T* __restrict__ tptr = static_cast<const T*>(args.t);
    const T* __restrict__ yptr = static_cast<const T*>(args.y);

    const int myslot = (threadIdx.x >> 5) * S + grp;
    MuxSlot<T>& my = cta.slot[myslot];                                       // the slot of this lane's group
    for (int e = threadIdx.x; e < (int)(sizeof(Cta) / 4); e += 32 * MUX_WARPS) reinterpret_cast<unsigned*>(&cta)[e] = 0u;
    if constexpr (MUX_WARPS > 1) __syncthreads(); else __syncwarp();
    const int warpId = threadIdx.x >> 5;
    MuxQueue& tq = cta.q;
    auto cta_sync = [&]() {
        if constexpr (MUX_WARPS == 1) __syncwarp();
        else __syncthreads();
    };

    // ---- warp-role state: the shared abscissa of my rows (lane + 32 k)
    T tts[R];
#pragma unroll
    for (int k = 0; k < R; ++k) { const int row = lane + 32 * k; tts[k] = (Model::kHasData && !gridPerProblem && row < m) ? tptr[row] : (T)0; }

    // ---- group-role state: problem `grp` of this warp, parameter gl.  Scalars are bit-identical in the 8 lanes.
    bool active = false, retired = false, init = false, finished = false, passOpen = false, skipRest = false;
    unsigned long long prob = 0;
    int ysel = 0, jacMode = 0;
    T x = (T)0, xt = (T)0, dX = (T)0, Jy = (T)0, lo = -Num<T>::inf(), up = Num<T>::inf();
    T lambda = (T)0, mu = (T)1, residual = Num<T>::inf(), deltaX_dot = (T)0, nd = (T)0, trial = (T)0;
    T fd_xp = (T)0, fd_xm = (T)0, fd_rt = (T)0;
    unsigned age = 0, maxAge = 1, iterations = 0, fCalls = 0, gCalls = 0;
    int status = mir_ls_numericError;
    bool needJacobian = false, fConverged = false, countedRetired = false;
    unsigned sPasses = 0, sAccepted = 0, sFresh = 0, sBroyden = 0, sEvals = 0, sSolves = 0, sQPIt = 0, sProblems = 0;

    for (;;) {
#pragma unroll 1
        for (int half = 0; half < 2; ++half) {
            int rf = 0;                        // row work this group's slot asks for (MUX_EVAL_* / MUX_JAC_*)
            if (half == 0) {
                // ======================================================= close the open pass: accept / reject, LS:1117-1175
                const bool closing = active && !finished && passOpen;
                bool accepted = false;
                T improvement = (T)0;
                if (closing && !skipRest) {
                    if (!(trial <= Num<T>::inf())) { status = mir_ls_numericError; finished = true; }        // LS:1117-1122
                    else {
                        improvement = residual - trial;                                                      // LS:1124
                        if (!(improvement > (T)0)) { lambda *= st.lambdaIncrease * mu; mu *= (T)2; }         // LS:1125-1130
                        else accepted = true;
                    }
                }
                if (__any_sync(MUX_FULL, accepted)) {
                    T acc = (T)0;                                                                            // symv(Lower, 1, JJ, deltaX, 2, Jy), LS:1141
#pragma unroll
                    for (int j = 0; j < G; ++j) acc = fma(my.JJ[gl * G + j], gshfl(dX, j), acc);
                    const T Jy2 = acc + (T)2 * Jy;
                    const T pred = -gsum8(Jy2 * dX);                                                         // LS:1142
                    T xss = gsum8(valid ? xt * xt : (T)0);                                                   // LS:1164: nrm2(x)
                    T xsc = (T)1;
                    if (__any_sync(MUX_FULL, accepted && !(xss >= Num<T>::small_() && xss <= Num<T>::large_()))) {   // BLAS scales: so do we when it matters
                        const T xmax = gmax8(valid ? t_abs(xt) : (T)0);
                        xsc = (xmax > (T)0 && xmax < Num<T>::inf()) ? xmax : (T)1;
                        const T vx = valid ? xt * rcp_ni(xsc) : (T)0;
                        xss = gsum8(vx * vx);
                    }
                    const T xn = xsc * sqrt_ni(xss);
                    if (accepted) {
                        needJacobian = true; mu = (T)1; ++iterations; ++sAccepted;                           // LS:1132-1139
                        x = xt; ysel ^= 1;                     // the reference swaps the slices y / mBuffer, LS:1136
                        residual = trial;
                        fConverged = residual <= st.maxGoodResidual;
                        deltaX_dot = nd;
                        Jy = Jy2;                              // (scratch from here, as in the reference)
                        if (!(pred > (T)0)) { status = mir_ls_furtherImprovement; finished = true; }         // LS:1144-1148
                        else {
                            const T rho = div_ni(pred, improvement);                                         // LS:1150
                            if (rho < st.minStepQuality) { lambda *= st.lambdaIncrease * mu; mu *= (T)2; }   // LS:1152-1156
                            else if (rho >= st.goodStepQuality) lambda = t_max(st.lambdaDecrease * lambda * mu, st.minLambda);   // LS:1158-1161
                            const T sd = sqrt_ni(deltaX_dot);
                            if (!(sd > st.absTolerance && xn > sd * st.relTolerance)) {                      // LS:1164-1173
                                if (age == 0) { status = mir_ls_xConverged; finished = true; }
                                else age = maxAge;
                            }
                        }
                    }
                }
                if (closing && !finished && !(iterations < st.maxIterations)) { status = mir_ls_maxIterations; finished = true; }   // LS:1175
                passOpen = false;

                // ======================================================= next pass: guards LS:974-995, Jacobian decision LS:996-1015
                bool open = false;
                if (active && !finished && !init) {
                    ++sPasses;
                    if (fConverged) { status = mir_ls_fConverged; finished = true; }                             // LS:974-978
                    else if (!(lambda <= st.maxLambda)) { status = mir_ls_furtherImprovement; finished = true; } // LS:979-983
                    else {
                        if (mu > (T)16 && age) { needJacobian = true; age = maxAge; mu = (T)1; }                 // LS:984-989
                        open = true;
                    }
                }
                if (gany8(valid && !(x <= x), gshift) && open) { status = mir_ls_numericError; finished = true; open = false; }   // LS:990-995
                const bool wantTail = open && !needJacobian && age == 0 && tailShortcut;
                if (__any_sync(MUX_FULL, wantTail)) {
                    // tail_is_inert (lm_small.cuh), distributed: lane gl holds x_gl, (J^T y)_gl and row gl of J^T J
                    const T q2 = gsum8(Jy * Jy);
                    const T xmin = gmin8(valid ? t_abs(x) : Num<T>::inf());
                    const bool small = xmin > (T)0 && st.maxStep > (T)0 && sqrt_ni(q2) < lambda * (xmin * (Num<T>::lapack_eps() * (T)0.125));
                    const bool strict = gall8(!valid || ((lo < x) && (x < up)), gshift);
                    const bool inside = gall8(!valid || ((lo <= x) && (x <= up)), gshift);
                    bool inert = wantTail && small && strict;
                    if (__any_sync(MUX_FULL, wantTail && small && !strict && inside)) {                          // tail_bounds_certificate
                        T row = (T)0;
#pragma unroll
                        for (int j = 0; j < G; ++j) row += t_abs(my.JJ[gl * G + j]);
                        const T nu = gmax8(row), qinf = gmax8(t_abs(Jy));
                        const T thr = ((T)8 * nu) * (qinf / lambda), dmax = xmin * (Num<T>::lapack_eps() * (T)0.25);
                        const T ql = lo - x, qu = up - x;
                        const bool onL = ql == (T)0, onU = qu == (T)0;
                        const bool farL = (-ql - dmax) >= (T)2 * (st.qpSettings.relTolerance + st.qpSettings.absTolerance * t_abs(ql));
                        const bool farU = (qu - dmax) >= (T)2 * (st.qpSettings.relTolerance + st.qpSettings.absTolerance * t_abs(qu));
                        bool ok;
                        if (onL && onU) ok = false;
                        else if (onL || onU) ok = (onL ? farU : farL) && (t_abs(Jy) >= thr);
                        else ok = farL && farU;
                        const bool allOk = gall8(!valid || ok, gshift);
                        if (wantTail && small && !strict && inside) inert = (lambda >= (T)4 * nu) && allOk;
                    }
                    if (inert) {
                        for (;;) {                             // replay LS:1112, 1125-1130 and the next pass's LS:979-983
                            ++fCalls;
                            lambda *= st.lambdaIncrease * mu; mu *= (T)2;
                            ++sPasses;
                            if (!(lambda <= st.maxLambda)) break;
                        }
                        status = mir_ls_furtherImprovement; finished = true; open = false;
                    }
                }
                jacMode = 0;
                if (open) {
                    passOpen = true; skipRest = false;
                    if (needJacobian) {                                                                          // LS:996-998
                        needJacobian = false;
                        if (age < maxAge) { ++age; jacMode = MUX_JAC_BROYDEN; ++sBroyden; }                      // LS:999-1007
                        else {
                            age = 0; jacMode = MUX_JAC_FRESH; ++sFresh;                                          // LS:1010
                            if (FD) fCalls += N; else gCalls += 1;                                               // LS:1049 (counts tasks) / LS:1014
                            if constexpr (FD) {                                                                  // LS:1026-1033, parameter gl
                                fd_xm = t_max(x - st.jacobianEpsilon, lo);
                                fd_xp = t_min(x + st.jacobianEpsilon, up);
                                const T twh = fd_xp - fd_xm;
                                fd_rt = (twh != (T)0) ? rcp_ni(twh) : (T)0;      // 0 marks "column = 0" (LS:1045-1047); 1 / twh is never 0
                            }
                        }
                    }
                    rf = jacMode;
                }

                // ======================================================= retire finished problems, refill the slot
                if (active && finished) {
                    if (valid) static_cast<T*>(args.x)[prob * N + gl] = x;
                    if (gl == 0) {
                        Result ret;
                        ret.status = status; ret.iterations = iterations; ret.fCalls = fCalls; ret.gCalls = gCalls;
                        ret.residual = residual; ret.lambda = lambda;
                        static_cast<Result*>(args.results)[prob] = ret;
                    }
                    active = false;
                }
                if (__any_sync(MUX_FULL, !active && !retired)) {
                    const bool want = !active && !retired;
                    unsigned int idx = 0, staged = 1;
                    if (want && gl == 0) {
                        idx = atomicAdd(args.counter, 1u);
                        if (idx < args.batch) staged = wait_staged(args.ready, idx, args.spin_limit) ? 1u : 0u;
                    }
                    idx = gshfl(idx, 0); staged = gshfl(staged, 0);
                    const bool take = want && idx < args.batch && staged;
                    T nx = (T)0, nlo = -Num<T>::inf(), nup = Num<T>::inf();
                    if (take && valid) {
                        nx = static_cast<const T*>(args.x)[(unsigned long long)idx * N + gl];
                        nlo = static_cast<const T*>(args.l)[(unsigned long long)idx * args.bound_stride + gl];
                        nup = static_cast<const T*>(args.u)[(unsigned long long)idx * args.bound_stride + gl];
                    }
                    // validation, LS:930-943 (first failure wins)
                    const bool finite = gall8(!valid || (-Num<T>::inf() < nx && nx < Num<T>::inf()), gshift);
                    const bool inb = gall8(!valid || ((nlo <= nx) && (nx <= nup)), gshift);
                    if (want) {
                        if (idx >= args.batch) retired = true;
                        else {
                            ++sProblems;
                            int vs = 0;
                            if (!staged) vs = mir_ls_numericError;     // inputs never arrived: the host discards this launch (flag ready[1])
                            else if (m == 0 || !finite) vs = mir_ls_badGuess;
                            else if (!inb) vs = mir_ls_badBounds;
                            else if (!((T)0 <= st.minStepQuality && st.minStepQuality < (T)1)) vs = mir_ls_badMinStepQuality;
                            else if (!((T)0 <= st.goodStepQuality && st.goodStepQuality <= (T)1)) vs = mir_ls_badGoodStepQuality;
                            else if (!(st.minStepQuality < st.goodStepQuality)) vs = mir_ls_badStepQuality;
                            else if (!((T)1 <= st.lambdaIncrease && st.lambdaIncrease <= Num<T>::sqrt_max())) vs = mir_ls_badLambdaParams;
                            else if (!(Num<T>::sqrt_min_normal() <= st.lambdaDecrease && st.lambdaDecrease <= (T)1)) vs = mir_ls_badLambdaParams;
                            if (vs) {
                                if (gl == 0) {                     // x is left untouched
                                    Result ret;
                                    ret.status = vs; ret.iterations = 0; ret.fCalls = 0; ret.gCalls = 0; ret.residual = Num<T>::inf(); ret.lambda = (T)0;
                                    static_cast<Result*>(args.results)[idx] = ret;
                                }
                            } else {
                                active = true; init = true; finished = false; passOpen = false; skipRest = false;
                                prob = idx; x = nx; lo = nlo; up = nup;
                                xt = x; dX = (T)0; Jy = (T)0; ysel = 0;
                                maxAge = st.maxAge ? st.maxAge : (FD ? 2u * N : 3u);                                 // LS:945
                                iterations = 0; fCalls = 0; gCalls = 0; status = mir_ls_maxIterations;               // LS:959-971
                                residual = Num<T>::inf(); lambda = warm_lambda<T>(args, prob); mu = (T)1; deltaX_dot = (T)0;
                                age = maxAge; needJacobian = false; fConverged = false; jacMode = 0;
                                rf = MUX_EVAL_INIT;                                                                  // initial residual, LS:953-956
                            }
                        }
                    }
                }
            } else {
                // ======================================================= the initial residual has arrived, LS:953-971
                bool go = active && !finished && passOpen;
                if (active && init) {
                    init = false; go = false;
                    residual = trial; fCalls = 1;
                    fConverged = residual <= st.maxGoodResidual;
                    needJacobian = true; age = maxAge;
                }
                // ======================================================= g-test LS:1053-1062
                const bool jacd = go && jacMode != 0;
                if (__any_sync(MUX_FULL, jacd)) {
                    const T jyn = valid ? my.Jy[gl] : (T)0;
                    T gsel = gmax8(t_abs(jyn));                    // iamax picks the first max |.|: its magnitude is the max
                    const T j0 = gshfl(jyn, 0);
                    if (!(j0 == j0)) gsel = j0;                    // BLAS: a NaN wins iamax only as the first element
                    if (jacd) {
                        Jy = jyn;
                        if (!(gsel > st.gradTolerance)) {
                            go = false;
                            if (age == 0) { status = mir_ls_gConverged; finished = true; }
                            else { age = maxAge; skipRest = true; }
                        }
                    }
                }
                // ======================================================= lambda LS:1067-1072, BOXCQP LS:1074-1085, trial point LS:1087-1112
                if (__any_sync(MUX_FULL, go)) {
                    T JJrow[G];
                    T JJdiag = (T)0;
#pragma unroll
                    for (int j = 0; j < G; ++j) { JJrow[j] = my.JJ[gl * G + j]; JJdiag = (j == gl) ? JJrow[j] : JJdiag; }
                    const T dmax = gmax8(valid ? JJdiag : (T)0);          // diag[iamax]; the diagonal of J^T J is >= 0
                    if (go && !(lambda >= st.minLambda)) {                                                       // LS:1067-1072
                        lambda = (T)(0.001 * (double)dmax);
                        if (!(lambda >= st.minLambda)) lambda = (T)1;
                    }
                    QPCounters qc{0, 0};
                    T dXn;
                    const int qps = boxqp_dist<T, N>(go, gl, gshift, st.qpSettings, JJrow, lambda, Jy, lo - x, up - x, dXn, qc);   // LS:1074-1080
                    sSolves += qc.solves; sQPIt += qc.iterations;
                    const bool nan = gany8(valid && !(dXn <= dXn), gshift);                                      // LS:1087-1092
                    const T dXr = valid ? add_rn(add_rn(dXn, x), -x) : (T)0;                                     // LS:1096-1097
                    const T ndn = gsum8(dXr * dXr);                                                              // LS:1099
                    const T xtn = valid ? t_max(t_min(add_rn(dXr, x), up), lo) : (T)0;                           // LS:1108-1110
                    const bool same = gall8(!valid || ((xtn == x) && (signbit(xtn) == signbit(x))), gshift);
                    const T sdn = sqrt_ni(ndn);
                    if (go) {
                        if (qps != mir_qp_solved || nan) { status = mir_ls_numericError; finished = true; }      // LS:1080-1092
                        else {
                            dX = dXr; nd = ndn;
                            if (!(sdn < st.maxStep)) { lambda *= st.lambdaIncrease * mu; mu *= (T)2; skipRest = true; }   // LS:1101-1106
                            else {
                                xt = xtn;
                                ++fCalls;                                                                        // LS:1112
                                if (same) trial = residual;       // f(xt) == y bit for bit: evaluation skipped, a rejection follows
                                else rf = MUX_EVAL_TRIAL;
                            }
                        }
                    }
                }
            }

            // =========================================================== row phase: post this slot's request, then pull tasks
            // (Tried: pulling as soon as a warp has posted, the queue growing while it is served, with fences and a posted-
            //  warps counter instead of the barrier below -- +3 % at 262,144 fits, but the n-sized phases of the warps end
            //  together anyway, and compute-sanitizer's racecheck cannot see through flag-based hand-offs.  Not kept.)
            bool evalPending = false;
            if (rf != 0) {
                my.p[gl] = (rf & MUX_EVAL_TRIAL) ? xt : x;
                if (rf & MUX_JAC_BROYDEN) my.dX[gl] = dX;
                if (FD && (rf & MUX_JAC_FRESH)) { my.fxp[gl] = fd_xp; my.fxm[gl] = fd_xm; my.frt[gl] = fd_rt; }
                if (gl == 0) {
                    my.ddot = deltaX_dot; my.prob = prob; my.flags = rf; my.ysel = ysel;
                    tq.qtask[half][atomicAdd(&tq.qn[half], 1)] = (unsigned char)myslot;
                }
                evalPending = (rf & (MUX_EVAL_INIT | MUX_EVAL_TRIAL)) != 0;
            }
            // exit consensus of the CTA: every warp that has run out of problems is counted once
            const bool warpRetired = __all_sync(MUX_FULL, retired);
            if (half == 0 && warpRetired && lane == 0 && !countedRetired) atomicAdd(&tq.retired, 1);
            if (half == 0 && warpRetired) countedRetired = true;
            cta_sync();
            if (half == 0 && *(volatile int*)&tq.retired == MUX_WARPS) goto done;
            if (lane == 0 && warpId == 0) { tq.qn[half ^ 1] = 0; tq.qhead[half ^ 1] = 0; }     // the other half's queue is idle now
            const int nTasks = tq.qn[half];
#pragma unroll 1
            for (;;) {
                int task = 0;
                if (lane == 0) task = atomicAdd(&tq.qhead[half], 1);
                task = __shfl_sync(MUX_FULL, task, 0);
                if (task >= nTasks) break;
                const int s = tq.qtask[half][task];
                MuxSlot<T>& sl = cta.slot[s];
                const int f = sl.flags;
                const unsigned long long sprob = sl.prob;
                T* const yv = sl.vec[sl.ysel];
                T* const mv = sl.vec[sl.ysel ^ 1];
                const bool evalOnly = (f & (MUX_EVAL_INIT | MUX_EVAL_TRIAL)) != 0;
                T p[N];
#pragma unroll
                for (int j = 0; j < N; ++j) p[j] = sl.p[j];
                T tk[R];
#pragma unroll
                for (int k = 0; k < R; ++k) {
                    const int row = lane + 32 * k;
                    tk[k] = gridPerProblem ? ((Model::kHasData && row < m) ? tptr[sprob * (unsigned long long)m + row] : (T)0) : tts[k];
                }

                if (evalOnly || (f & MUX_JAC_FRESH)) {
                    T yo[R];
#pragma unroll
                    for (int k = 0; k < R; ++k) {
                        const int row = lane + 32 * k;
                        yo[k] = (Model::kHasData && row < m && (evalOnly || FD)) ? yptr[sprob * (unsigned long long)m + row] : (T)0;
                    }
                    T* const dst = (f & MUX_EVAL_INIT) ? yv : mv;
                    T part = (T)0;
                    // evaluation items.  evalOnly: one evaluation at p.  Fresh analytic Jacobian: one item that delivers
                    // Jacobian rows.  Fresh finite-difference Jacobian: 2 N evaluations, (column j, +h) then (column j, -h),
                    // LS:1018-1049 -- or, for models that share sub-expressions between those evaluations
                    // (Model::kFDShared, models.cuh), 1 + NE / CPI items.
                    const bool shared = kShared && !evalOnly;
                    int nItems = (evalOnly || !FD) ? 1 : 2 * N;
                    if constexpr (kShared) { if (shared) nItems = 1 + NE / Model::CPI; }
                    [[maybe_unused]] typename SharedFD<Model, T, kShared>::State fds = {};
                    if (lane == 0 && !evalOnly && FD) sEvals += 2u * N;
#pragma unroll 1
                    for (int it = 0; it < nItems; ++it) {
                        const int j = it >> 1, sgn = it & 1;
                        T pp[N], ea[KB], ee[KB];
                        T rt = (T)0;
                        constexpr int CPI = SharedFD<Model, T, kShared>::CPI;
                        [[maybe_unused]] T xpr[CPI], xmr[CPI], rtr[CPI], xpa[CPI], xma[CPI], rta[CPI];
                        if constexpr (kShared) {
                            if (shared) {
#pragma unroll
                                for (int c = 0; c < CPI; ++c) {
                                    const int kc = (it >= 1) ? (it - 1) * CPI + c : 0;
                                    xpr[c] = sl.fxp[2 * kc + 1]; xmr[c] = sl.fxm[2 * kc + 1];
                                    rtr[c] = sl.frt[2 * kc + 1];
                                    xpa[c] = sl.fxp[2 * kc]; xma[c] = sl.fxm[2 * kc];
                                    rta[c] = sl.frt[2 * kc];
                                }
                            }
                        }
                        if (FD && !evalOnly && !kShared) {
                            const T xpm = sgn ? sl.fxm[j] : sl.fxp[j];
                            rt = sl.frt[j];
#pragma unroll
                            for (int i = 0; i < N; ++i) pp[i] = (i == j) ? xpm : p[i];
                        } else {
#pragma unroll
                            for (int i = 0; i < N; ++i) pp[i] = p[i];
                        }
                        const typename Model::Pre pre = Model::prepare(pp);
                        bool generic = true;
                        if constexpr (kShared) {
                            if (shared) { generic = false; Model::template fds_args<R>(it, p, tk, xpr, xmr, ea); }
                        }
                        if (generic) {
#pragma unroll
                            for (int r = 0; r < R; ++r) Model::exp_args(pre, pp, tk[r], ea + r * NE);
                        }
                        exp_repro_many_conv<KB>(ea, ee);
                        if constexpr (kShared) {
                            if (shared)
                                Model::template fds_deliver<R>(it, p, yo, ee, fds, xpr, xmr, rtr, xpa, xma, rta,
                                    [&](int col, int k, T v) { const int row = lane + 32 * k; sl.J[col][row] = (row < m) ? v : (T)0; });
                        }
                        if (generic) {
#pragma unroll
                            for (int r = 0; r < R; ++r) {
                                const int row = lane + 32 * r;
                                if (!FD && !evalOnly) {                                                          // LS:1011-1015
                                    T Jr[N];
                                    Model::finish_j(pre, pp, tk[r], ee + r * NE, Jr);
#pragma unroll
                                    for (int i = 0; i < N; ++i) sl.J[i][row] = (row < m) ? Jr[i] : (T)0;
                                } else {
                                    T v;
                                    Model::finish_r(pre, pp, tk[r], yo[r], ee + r * NE, v);
                                    v = (row < m) ? v : (T)0;
                                    if (evalOnly) { dst[row] = v; part += v * v; }
                                    else if (sgn == 0) sl.J[j][row] = v;                                      // f(x + h e_j), parked in its column
                                    else sl.J[j][row] = (rt != (T)0) ? (sl.J[j][row] - v) * rt : (T)0;     // LS:1040-1047
                                }
                            }
                        }
                    }
                    if (lane == 0 && evalOnly) ++sEvals;
                    if (evalOnly) {
#pragma unroll
                        for (int off = 16; off > 0; off >>= 1) part += __shfl_xor_sync(MUX_FULL, part, off);
                        if (lane == 0) sl.result = part;
                    }
                }

                if (f & MUX_JAC_BROYDEN) {                                                                       // LS:999-1007
                    T dxs[N];
#pragma unroll
                    for (int j = 0; j < N; ++j) dxs[j] = sl.dX[j];
                    const T negd = -rcp_ni(sl.ddot);                                                             // LS:1001
#pragma unroll
                    for (int k = 0; k < R; ++k) {
                        const int row = lane + 32 * k;
                        T Jr[N];
#pragma unroll
                        for (int i = 0; i < N; ++i) Jr[i] = sl.J[i][row];
                        T acc = (T)0;                                            // here y = f_new, mBuffer = f_old (after the swap, LS:1136)
#pragma unroll
                        for (int i = 0; i < N; ++i) acc = fma(Jr[i], dxs[i], acc);                               // gemv(1, J, deltaX, 1, mBuffer)
                        const T v = ((mv[row] - yv[row]) + acc) * negd;                                          // axpy(-1, y, mBuffer); scal(-d, mBuffer)
                        if (row < m) {
#pragma unroll
                            for (int i = 0; i < N; ++i) sl.J[i][row] = fma(v, dxs[i], Jr[i]);                 // ger(1, mBuffer, deltaX, J)
                        }
                    }
                }

                if (f & (MUX_JAC_FRESH | MUX_JAC_BROYDEN)) {
                    // J^T y (LS:1052) and J^T J (syrk, LS:1065) on the FP64 tensor pipe.  m8n8k4: A = J^T (8 parameters x 4 rows),
                    // lane holds A[lane / 4][lane % 4]; B = J (4 rows x 8 parameters), lane holds B[lane % 4][lane / 4] -- the same
                    // value.  Four independent accumulator sets (rows 4q..4q+3 go to set q % 4), summed in a fixed order.
                    __syncwarp();
                    const int pi = lane >> 2, kk = lane & 3;
                    const T* const Ji = sl.J[pi];
                    double c[4][2], jy4[4];
#pragma unroll
                    for (int a = 0; a < 4; ++a) { c[a][0] = 0.0; c[a][1] = 0.0; jy4[a] = 0.0; }
                    const int nq = (m + 15) >> 4;
#pragma unroll 1
                    for (int q = 0; q < nq; ++q) {
#pragma unroll
                        for (int a = 0; a < 4; ++a) {
                            const double av = (double)Ji[16 * q + 4 * a + kk];
                            const double yy = (double)yv[16 * q + 4 * a + kk];
                            mux_dmma884(c[a], av, av);
                            jy4[a] = fma(av, yy, jy4[a]);
                        }
                    }
                    const double c0 = (c[0][0] + c[1][0]) + (c[2][0] + c[3][0]);
                    const double c1 = (c[0][1] + c[1][1]) + (c[2][1] + c[3][1]);
                    double jy = (jy4[0] + jy4[1]) + (jy4[2] + jy4[3]);
                    jy += __shfl_xor_sync(MUX_FULL, jy, 1);
                    jy += __shfl_xor_sync(MUX_FULL, jy, 2);
                    // lane holds (J^T J)[pi][2 kk], [pi][2 kk + 1]; the lower triangle is mirrored so the matrix is exactly symmetric
                    const int j0 = 2 * kk, j1 = 2 * kk + 1;
                    if (j0 <= pi) { sl.JJ[pi * G + j0] = (T)c0; sl.JJ[j0 * G + pi] = (T)c0; }
                    if (j1 <= pi) { sl.JJ[pi * G + j1] = (T)c1; sl.JJ[j1 * G + pi] = (T)c1; }
                    if (kk == 0) sl.Jy[pi] = (T)jy;
                }
                __syncwarp();
            }
            cta_sync();
            if (evalPending) trial = my.result;
        }
    }
done:
    if (args.stats && gl == 0 && sProblems) {
        atomicAdd((unsigned long long*)&args.stats->problems, (unsigned long long)sProblems);
        atomicAdd((unsigned long long*)&args.stats->passes, (unsigned long long)sPasses);
        atomicAdd((unsigned long long*)&args.stats->accepted, (unsigned long long)sAccepted);
        atomicAdd((unsigned long long*)&args.stats->fresh_jacobians, (unsigned long long)sFresh);
        atomicAdd((unsigned long long*)&args.stats->broyden_updates, (unsigned long long)sBroyden);
        atomicAdd((unsigned long long*)&args.stats->model_evals, (unsigned long long)sEvals);
        atomicAdd((unsigned long long*)&args.stats->qp_solves, (unsigned long long)sSolves);
        atomicAdd((unsigned long long*)&args.stats->qp_iterations, (unsigned long long)sQPIt);
    }
}

}  // namespace mirb200
