// lm_small.cuh -- one group (LANES lanes of a warp; LANES = 32 is "one warp per problem") per
// Levenberg-Marquardt problem.  Persistent groups pull problem indices from an atomic counter.
//
// Follows optimizeLeastSquaresImplGeneric!T, least_squares.d:877-1176 (line cites inline).
//
// Data layout.  Residual rows are dealt round-robin to the lanes (row = k*LANES + lane, k < R):
// each lane keeps its rows of y (current residuals), mBuffer (trial / previous residuals), the
// abscissa/observations and its rows of J in registers, so J (needed in place by the Broyden
// update, LS:1003-1006) never leaves the register file.  The n-sized state (x, bounds, J^T r,
// packed lower J^T J, lambda, mu, age, counters) is replicated bit-identically in every lane:
// all cross-row reductions are xor-butterflies, which hand every lane the same bits, so the
// "serial" part (BoxQP / Cholesky / lambda control) needs no communication and no divergence.
//
// Equivalences used (all bit-exact with respect to this file's own arithmetic):
//   * J^T J is rebuilt only when J changed, together with J^T r (the reference re-runs syrk every
//     pass, LS:1065; with unchanged J it returns the same matrix).
//   * If the trial point equals x bit for bit, f(trial) == y and trial residual == residual, so
//     the pass is a rejection (LS:1124-1130); the model evaluation is skipped, fCalls still counts it.
//   * The lambda-overflow tail (the reference's normal exit on noisy data, LS:979-983 + 1125-1130) is
//     fast-forwarded once it is provably inert -- see tail_is_inert() below.
#pragma once
#include "boxqp_small.cuh"
#include "models.cuh"

namespace mirb200 {

struct SmallBatchArgs {
    const void* t;          // abscissa: T[m] or T[batch*m]
    const void* y;          // observations T[batch*m]
    void*       x;          // T[batch*n] in/out
    const void* l;          // T[n] or T[batch*bound_stride]
    const void* u;
    void*       results;    // Result[batch]
    unsigned int* counter;         // work queue head (zeroed by the launcher); batch < 2^32 per launch
    const unsigned int* ready;     // null, or {watermark, time-out flag}: problems [0, ready[0]) have been staged into device
                                   // memory.  The host-pointer entry copies the inputs in chunks, bumping the watermark after
                                   // each chunk, and runs the kernel beside the copies, so the transfer overlaps the solve.
    unsigned int spin_limit;       // wait_staged gives up after this many ~1 us polls of one problem
    mir_batch_stats* stats; // may be null
    unsigned long long batch;
    unsigned m;
    unsigned bound_stride;
    unsigned flags;         // MIR_MODEL_* flags
};

// Blocks until problem `idx` has been staged (see SmallBatchArgs::ready).  ready[0] is the watermark, written by the
// copy engine (stream-ordered after the chunk's data) and read here with acquire semantics at gpu scope; ready[1] is a
// time-out flag owned by the kernel.  Chunks are multiples of 65536 problems, so no cache line of any input array
// straddles staged and unstaged data.  The host enqueues every copy BEFORE the launch and orders the launch after the
// first chunk (lm_batched.cu), so a launch that blocks the host (CUDA_LAUNCH_BLOCKING, profilers) cannot starve the
// copies; the wait is still bounded (`spin_limit` polls of ~1 us) in case the copy engine cannot run beside the kernel
// at all.  On time-out the flag is raised, every later waiter fails at once, and the host -- which always reads the
// flag back -- discards the launch and re-runs it unstaged: a time-out never surfaces as per-problem results.
__device__ __forceinline__ bool wait_staged(const unsigned int* ready, unsigned int idx, unsigned int spin_limit)
{
    if (!ready) return true;
    unsigned spins = 0;
    for (;;) {
        unsigned int v, bad;
        asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(ready) : "memory");
        if (v > idx) return true;
        asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(bad) : "l"(ready + 1) : "memory");
        if (bad || ++spins > spin_limit) {
            if (!bad) atomicExch(const_cast<unsigned int*>(ready) + 1, 1u);
            return false;
        }
        __nanosleep(1000);
    }
}


// Warm start (MIR_MODEL_WARM_START; the reference documents Result.lambda as the "(inverse of) initial trust region
// radius", LS:141-142, but always restarts from 0, LS:966 -- SURVEY 8f-4): the caller's Result.lambda, if it is a usable
// damping value, replaces the 0.  A value >= minLambda also skips the 0.001 max diag(J^T J) initialisation, LS:1067-1072.
template <class T> __device__ __forceinline__ T warm_lambda(const SmallBatchArgs& args, unsigned long long prob)
{
    if (!(args.flags & MIR_MODEL_WARM_START)) return (T)0;
    const T v = static_cast<const typename Num<T>::Result*>(args.results)[prob].lambda;
    return (v > (T)0 && v < Num<T>::inf()) ? v : (T)0;
}

// Lambda-overflow tail.  State: J is current (needJacobian == false), age == 0, the last pass was a rejection.
// The step solves min 1/2 d'Pd + q'd over a box that contains d = 0, with P = J'J + lambda I >= lambda I and
// q = J'r.  The minimiser has objective <= 0, hence lambda/2 |d|^2 <= -q'd <= |q| |d| and |d|_2 <= 2 |q|_2 / lambda.
// Once 2 |q|_2 / lambda < 1/4 min_i ulp(x_i) (all x_i != 0; ulp(x) >= |x| eps/2, and the factor 4 covers the
// O(eps) relative error of the computed solution of this perfectly conditioned system and the half-width binade
// just below a power of two), every component of (d + x) - x (LS:1096-1097) is exactly 0, so the trial point is x,
// the trial residual equals the residual bit for bit and the pass is a rejection: lambda *= lambdaIncrease * mu,
// mu *= 2 (LS:1125-1130).  Nothing else changes (age == 0, so `mu > 16` cannot force a new Jacobian, LS:984-989),
// |q| / lambda only shrinks, and the same holds for every later pass until !(lambda <= maxLambda) ends the run with
// furtherImprovement (LS:979-983).  The caller therefore replays only the scalar recurrence (fCalls, lambda, mu).
// Two more conditions make the replay exact in the corners: maxStep must be positive (otherwise LS:1101-1106 rejects BEFORE
// the evaluation is counted and fCalls would differ), and the step must provably come back from BOXCQP as `solved`:
//  * No x_i on a bound: x_i - l_i >= ulp(x_i)/2 > |d_i|, the unconstrained solution passes the first test (BQ:216-219,
//    no tolerance involved) and is returned.
//  * Some x_i ON a bound (qpl_i == 0 or qpu_i == 0; ~10 % of BASELINE configs[1] end like this): the active-set loop may
//    run, and the certificate below (tail_bounds_certificate) shows it returns `solved` with a step that still vanishes.
//    Let nu = ||JJ||_inf and lambda >= 4 nu.  For ANY free set f the sub-solution is d_f = -(lambda I + JJ_ff)^-1 q_f =
//    -(q_f + e)/lambda with |e|_inf <= (4 nu / 3 lambda) |q|_inf, so |d|_inf <= 1.34 |q|_inf / lambda (tiny: the bound used
//    above) and, for every on-bound i with |q_i| >= 8 nu |q|_inf / lambda, sign(d_i) = -sign(q_i) and the multiplier
//    (P d + q)_i = q_i + sum_f JJ_if d_f has the sign of q_i.  Variables off their bounds keep a margin of more than the
//    QP tolerance plus |d| on both sides, so BQ:239-263 never flags them.  Trace of BQ:234-375: the first test fails only if
//    some on-bound variable points outward; iteration 1 flags those (xl < 0) and possibly inward ones (xl < tol with a zero
//    multiplier); outward ones get multipliers of the right sign and stay flagged (xl = 0 < tol, la >= 0), inward ones get
//    a negative multiplier, are released in iteration 2 (mu = la = 0, d_i > 0 inside) and the tests at BQ:339-347 pass:
//    `solved` after at most two iterations, never the all-free exit (BQ:265-266: an outward variable stays flagged).
//    Every condition only gets easier as lambda grows, so it holds for all later passes of the tail.
template <class T, int N> struct TailCase {
    T x[N], q[N], lo[N], up[N], JJ[N * (N + 1) / 2];
    T lambda, dmax, relTol, absTol;
};
template <class T, int N>
__device__ __noinline__ bool tail_bounds_certificate(const TailCase<T, N> c)
{
    bool any = false;
    for (int i = 0; i < N; ++i) any = any || (c.lo[i] == c.x[i]) || (c.up[i] == c.x[i]);
    if (!any) return true;                                 // (the caller has checked lo < x < up otherwise)
    T nu = (T)0, qinf = (T)0;
    for (int i = 0; i < N; ++i) {
        T row = (T)0;
        for (int j = 0; j < N; ++j) row += t_abs(c.JJ[trisym(i, j)]);
        nu = t_max(nu, row); qinf = t_max(qinf, t_abs(c.q[i]));
    }
    if (!(c.lambda >= (T)4 * nu)) return false;
    const T thr = ((T)8 * nu) * (qinf / c.lambda);
    for (int i = 0; i < N; ++i) {
        const T ql = c.lo[i] - c.x[i], qu = c.up[i] - c.x[i];                       // LS:1074-1077
        const bool onL = ql == (T)0, onU = qu == (T)0;
        const bool farL = (-ql - c.dmax) >= (T)2 * (c.relTol + c.absTol * t_abs(ql));   // an infinite bound is far (inf >= inf)
        const bool farU = (qu - c.dmax) >= (T)2 * (c.relTol + c.absTol * t_abs(qu));
        if (onL && onU) return false;
        if (onL || onU) {
            if (!(onL ? farU : farL)) return false;
            if (!(t_abs(c.q[i]) >= thr)) return false;
        } else if (!(farL && farU)) return false;
    }
    return true;
}

template <class T, int N, class BL, class BU>
__device__ __forceinline__ bool tail_is_inert(const T (&x)[N], const T (&Jy)[N], const T (&JJ)[N * (N + 1) / 2], T lambda, const BL& lo, const BU& up,
                                              const typename Num<T>::Settings& st)
{
    T q2 = (T)0, xmin = Num<T>::inf();
#pragma unroll
    for (int i = 0; i < N; ++i) { q2 += Jy[i] * Jy[i]; xmin = t_min(xmin, t_abs(x[i])); }
    if (!(xmin > (T)0 && st.maxStep > (T)0 && sqrt_ni(q2) < lambda * (xmin * (Num<T>::lapack_eps() * (T)0.125)))) return false;
    bool inside = true, strict = true;
#pragma unroll
    for (int i = 0; i < N; ++i) { inside = inside && (lo[i] <= x[i]) && (x[i] <= up[i]); strict = strict && (lo[i] < x[i]) && (x[i] < up[i]); }
    if (strict) return true;
    if (!inside) return false;
    TailCase<T, N> c;                                      // rare path, out of line: the caller's registers stay untouched
#pragma unroll
    for (int i = 0; i < N; ++i) { c.x[i] = x[i]; c.q[i] = Jy[i]; c.lo[i] = lo[i]; c.up[i] = up[i]; }
#pragma unroll
    for (int i = 0; i < N * (N + 1) / 2; ++i) c.JJ[i] = JJ[i];
    c.lambda = lambda; c.dmax = xmin * (Num<T>::lapack_eps() * (T)0.25);
    c.relTol = st.qpSettings.relTolerance; c.absTol = st.qpSettings.absTolerance;
    return tail_bounds_certificate<T, N>(c);
}

template <class Model, class T, int LANES, int R, bool FD>
__global__ void __launch_bounds__(128, 1)
lm_small_kernel(const typename Num<T>::Settings st, const SmallBatchArgs args)
{
    constexpr int N = Model::N;
    constexpr int NP = N * (N + 1) / 2;
    using Result = typename Num<T>::Result;

    const unsigned gmask = group_mask<LANES>();
    const int glane = threadIdx.x & (LANES - 1);
    // Cross-lane reduction scratch of this group: K = NP + N running sums, one padded row per value.
    constexpr int K = NP + N;
    __shared__ T s_red[128 / LANES][K * (LANES + 1) + K];
    T* const red = s_red[threadIdx.x / LANES];
    const int m = (int)args.m;
    constexpr bool useFD = FD;        // g == null semantics (finite differences), compile-time to keep the code small
    const bool gridPerProblem = (args.flags & MIR_MODEL_GRID_PER_PROBLEM) != 0;
    const bool tailShortcut = (args.flags & MIR_MODEL_NO_TAIL_SHORTCUT) == 0;
    const T* __restrict__ tptr = static_cast<const T*>(args.t);
    const T* __restrict__ yptr = static_cast<const T*>(args.y);

    // local work counters, flushed once per group at the end
    unsigned long long sPasses = 0, sAccepted = 0, sFresh = 0, sBroyden = 0, sEvals = 0, sSolves = 0, sQPIt = 0, sProblems = 0;

    // abscissa shared by every problem: load once
    T tt[R];
    if (Model::kHasData && !gridPerProblem) {
#pragma unroll
        for (int k = 0; k < R; ++k) { const int row = k * LANES + glane; tt[k] = row < m ? tptr[row] : (T)0; }
    }

    for (;;) {
        unsigned int prob32 = 0;
        unsigned int staged = 1;
        if (glane == 0) {
            prob32 = atomicAdd(args.counter, 1u);
            if (prob32 < args.batch) staged = wait_staged(args.ready, prob32, args.spin_limit) ? 1u : 0u;
        }
        prob32 = __shfl_sync(gmask, prob32, 0, LANES);
        staged = __shfl_sync(gmask, staged, 0, LANES);
        if (prob32 >= args.batch) break;
        const unsigned long long prob = prob32;
        ++sProblems;
        if (!staged) {                                  // inputs never arrived: the host discards this launch (flag ready[1]); do not touch x
            if (glane == 0) {
                Result bad;
                bad.status = mir_ls_numericError; bad.iterations = 0; bad.fCalls = 0; bad.gCalls = 0; bad.residual = Num<T>::inf(); bad.lambda = (T)0;
                static_cast<Result*>(args.results)[prob] = bad;
            }
            continue;
        }

        // ---- load the problem ----
        T x[N], lo[N], up[N];
        {
            const T* xp = static_cast<const T*>(args.x) + prob * N;
            const T* lp = static_cast<const T*>(args.l) + prob * args.bound_stride;
            const T* upp = static_cast<const T*>(args.u) + prob * args.bound_stride;
#pragma unroll
            for (int i = 0; i < N; ++i) { x[i] = xp[i]; lo[i] = lp[i]; up[i] = upp[i]; }
        }
        T yo[R];
        if (Model::kHasData) {
#pragma unroll
            for (int k = 0; k < R; ++k) {
                const int row = k * LANES + glane;
                yo[k] = row < m ? yptr[prob * (unsigned long long)m + row] : (T)0;
                if (gridPerProblem) tt[k] = row < m ? tptr[prob * (unsigned long long)m + row] : (T)0;
            }
        } else {
#pragma unroll
            for (int k = 0; k < R; ++k) { yo[k] = (T)0; tt[k] = (T)0; }
        }

        Result ret;                                                   // LeastSquaresResult.init, LS:131-142
        ret.status = mir_ls_numericError; ret.iterations = 0; ret.fCalls = 0; ret.gCalls = 0;
        ret.residual = Num<T>::inf(); ret.lambda = (T)0;

        // residual vector evaluation: out[k] = r_row(p) for this lane's rows, returns ||r||^2
        auto eval = [&](const T (&p)[N], T (&out)[R]) -> T {
            const typename Model::Pre pre = Model::prepare(p);
            T part = (T)0;
#pragma unroll
            for (int k = 0; k < R; ++k) {
                const int row = k * LANES + glane;
                T r = (T)0;
                if (row < m) r = Model::residual(pre, p, row, tt[k], yo[k]);
                out[k] = r;
                part += r * r;
            }
            ++sEvals;
            return group_sum<LANES>(gmask, part);
        };

        // ---- validation, LS:930-943 (first failure wins) ----
        bool valid = false;
        {
            bool finite = true, inb = true;
#pragma unroll
            for (int i = 0; i < N; ++i) {
                finite = finite && (-Num<T>::inf() < x[i] && x[i] < Num<T>::inf());
                inb = inb && (lo[i] <= x[i]) && (x[i] <= up[i]);
            }
            if (m == 0 || !finite) ret.status = mir_ls_badGuess;
            else if (!inb) ret.status = mir_ls_badBounds;
            else if (!((T)0 <= st.minStepQuality && st.minStepQuality < (T)1)) ret.status = mir_ls_badMinStepQuality;
            else if (!((T)0 <= st.goodStepQuality && st.goodStepQuality <= (T)1)) ret.status = mir_ls_badGoodStepQuality;
            else if (!(st.minStepQuality < st.goodStepQuality)) ret.status = mir_ls_badStepQuality;
            else if (!((T)1 <= st.lambdaIncrease && st.lambdaIncrease <= Num<T>::sqrt_max())) ret.status = mir_ls_badLambdaParams;
            else if (!(Num<T>::sqrt_min_normal() <= st.lambdaDecrease && st.lambdaDecrease <= (T)1)) ret.status = mir_ls_badLambdaParams;
            else valid = true;
        }

        if (valid) {
            const unsigned maxAge = st.maxAge ? st.maxAge : (useFD ? 2u * N : 3u);          // LS:945

            T yv[R], mb[R];          // y and mBuffer (this lane's rows)
            T J[R][N];
            T JJ[NP], Jy[N], dX[N];
#pragma unroll
            for (int i = 0; i < N; ++i) { Jy[i] = (T)0; dX[i] = (T)0; }
#pragma unroll
            for (int i = 0; i < NP; ++i) JJ[i] = (T)0;
#pragma unroll
            for (int k = 0; k < R; ++k) {
                mb[k] = (T)0;
#pragma unroll
                for (int i = 0; i < N; ++i) J[k][i] = (T)0;
            }

            ret.residual = eval(x, yv);                                                      // LS:953-955
            ret.fCalls = 1;
            bool fConverged = ret.residual <= st.maxGoodResidual;                            // LS:956
            bool needJacobian = true;                                                        // LS:959-971
            unsigned age = maxAge;
            T lambda = warm_lambda<T>(args, prob), mu = (T)1, deltaX_dot = (T)0;
            int status = mir_ls_maxIterations;
            unsigned iterations = 0;

            do {                                                                             // LS:972
                ++sPasses;
                if (fConverged) { status = mir_ls_fConverged; break; }                       // LS:974-978
                if (!(lambda <= st.maxLambda)) { status = mir_ls_furtherImprovement; break; } // LS:979-983
                if (mu > (T)16 && age) { needJacobian = true; age = maxAge; mu = (T)1; }     // LS:984-989
                {
                    bool nan = false;                                                        // LS:990-995
#pragma unroll
                    for (int i = 0; i < N; ++i) nan = nan || !(x[i] <= x[i]);
                    if (nan) { status = mir_ls_numericError; break; }
                }
                if (needJacobian) {                                                          // LS:996
                    needJacobian = false;
                    if (age < maxAge) {                                                      // Broyden, LS:999-1007
                        ++age; ++sBroyden;
                        const T d = rcp_ni(deltaX_dot);
#pragma unroll
                        for (int k = 0; k < R; ++k) {
                            T v = mb[k] - yv[k];                                             // axpy(-1, y, mBuffer)
                            T acc = (T)0;
#pragma unroll
                            for (int i = 0; i < N; ++i) acc += J[k][i] * dX[i];              // gemv(1, J, deltaX, 1, mBuffer)
                            v = (v + acc) * -d;                                              // scal(-d, mBuffer)
                            mb[k] = v;
#pragma unroll
                            for (int i = 0; i < N; ++i) J[k][i] += v * dX[i];                // ger(1, mBuffer, deltaX, J)
                        }
                    } else {
                        age = 0; ++sFresh;                                                   // LS:1010
                        if constexpr (!useFD) {                                              // LS:1011-1015
                            const typename Model::Pre pre = Model::prepare(x);
#pragma unroll
                            for (int k = 0; k < R; ++k) {
                                const int row = k * LANES + glane;
                                if (row < m) Model::jacobian(pre, x, row, tt[k], J[k]);
                            }
                            ret.gCalls += 1;
                        } else {                                                             // LS:1018-1049
#pragma unroll 1
                            for (int j = 0; j < N; ++j) {          // rolled: parameter j is selected by predication
                                T save = (T)0, lj = (T)0, uj = (T)0;
#pragma unroll
                                for (int i = 0; i < N; ++i) if (i == j) { save = x[i]; lj = lo[i]; uj = up[i]; }
                                T xmh = save - st.jacobianEpsilon;
                                T xph = save + st.jacobianEpsilon;
                                xmh = t_max(xmh, lj);
                                xph = t_min(xph, uj);
                                const T twh = xph - xmh;
                                T col[R];
#pragma unroll
                                for (int k = 0; k < R; ++k) col[k] = (T)0;
                                if (twh != (T)0) {
                                    T p[N], fp[R], fm[R];
#pragma unroll
                                    for (int i = 0; i < N; ++i) p[i] = (i == j) ? xph : x[i];
                                    eval(p, fp);
#pragma unroll
                                    for (int i = 0; i < N; ++i) p[i] = (i == j) ? xmh : x[i];
                                    eval(p, fm);
                                    const T rt = rcp_ni(twh);
#pragma unroll
                                    for (int k = 0; k < R; ++k) col[k] = (fp[k] - fm[k]) * rt;
                                    // (the reference evaluates through mBuffer, LS:1036-1039; nothing reads it
                                    //  before the next trial evaluation overwrites it, so it is not mirrored)
                                }
#pragma unroll
                                for (int k = 0; k < R; ++k)
#pragma unroll
                                    for (int i = 0; i < N; ++i) if (i == j) J[k][i] = col[k];
                            }
                            ret.fCalls += N;                                                 // LS:1049 (counts tasks)
                        }
                    }
                    {   // Jy = J^T y (LS:1052) and JJ = J^T J (syrk, LS:1065) in one cross-lane reduction.
                        // (The reference rebuilds JJ on every pass; J only changes here, so this is the one
                        //  place it has to be formed.)  Each lane sums its rows, the partials go through shared
                        //  memory, lane k adds the LANES partials of value k in a fixed order, and every lane
                        //  reads back the same K totals -- bit-identical replicas, and a rolled loop instead of
                        //  5*K unrolled shuffles keeps the kernel inside the instruction cache.
                        T part[K];
#pragma unroll
                        for (int i = 0; i < K; ++i) part[i] = (T)0;
#pragma unroll
                        for (int k = 0; k < R; ++k)
#pragma unroll
                            for (int i = 0; i < N; ++i) {
                                part[NP + i] += J[k][i] * yv[k];
#pragma unroll
                                for (int j = 0; j <= i; ++j) part[tri(i, j)] += J[k][i] * J[k][j];
                            }
                        __syncwarp(gmask);
#pragma unroll
                        for (int i = 0; i < K; ++i) red[i * (LANES + 1) + glane] = part[i];
                        __syncwarp(gmask);
#pragma unroll 1
                        for (int v = glane; v < K; v += LANES) {
                            const T* row = red + v * (LANES + 1);
                            T s0 = (T)0, s1 = (T)0, s2 = (T)0, s3 = (T)0;
#pragma unroll 2
                            for (int i = 0; i < LANES; i += 4) { s0 += row[i]; s1 += row[i + 1]; s2 += row[i + 2]; s3 += row[i + 3]; }
                            red[K * (LANES + 1) + v] = (s0 + s1) + (s2 + s3);
                        }
                        __syncwarp(gmask);
#pragma unroll
                        for (int i = 0; i < NP; ++i) JJ[i] = red[K * (LANES + 1) + i];
#pragma unroll
                        for (int i = 0; i < N; ++i) Jy[i] = red[K * (LANES + 1) + NP + i];
                    }
                    T gmax = (T)0; bool gnan = false;                                        // LS:1053
#pragma unroll
                    for (int i = 0; i < N; ++i) { gmax = t_max(gmax, t_abs(Jy[i])); gnan = gnan || !(Jy[i] == Jy[i]); }
                    // iamax picks an index by |.|; a NaN entry makes the reference's comparison false as well
                    // only when it is the selected entry -- treat any NaN as "not above tolerance" is NOT safe,
                    // so mirror BLAS: NaN never wins iamax unless it is the first element.
                    if (gnan && !(Jy[0] == Jy[0])) gmax = Jy[0];
                    if (!(gmax > st.gradTolerance)) {                                        // LS:1053-1062
                        if (age == 0) { status = mir_ls_gConverged; break; }
                        age = maxAge;
                        continue;
                    }
                }

                if (age == 0 && tailShortcut && tail_is_inert<T, N>(x, Jy, JJ, lambda, lo, up, st)) {
                    // (needJacobian is false here.)  Replay the rejections: LS:1112, 1125-1130, then the next pass's LS:979-983.
                    for (;;) {
                        ++ret.fCalls;
                        lambda *= st.lambdaIncrease * mu; mu *= (T)2;
                        ++sPasses;
                        if (!(lambda <= st.maxLambda)) break;
                    }
                    status = mir_ls_furtherImprovement;
                    break;
                }

                if (!(lambda >= st.minLambda)) {                                             // LS:1067-1072
                    T dmax = JJ[0];                                                          // diag[iamax]: first max |.|; diag >= 0
#pragma unroll
                    for (int i = 1; i < N; ++i) if (t_abs(JJ[tri(i, i)]) > t_abs(dmax)) dmax = JJ[tri(i, i)];
                    lambda = (T)(0.001 * (double)dmax);
                    if (!(lambda >= st.minLambda)) lambda = (T)1;
                }

                T qpl[N], qpu[N];                                                            // LS:1074-1077
#pragma unroll
                for (int i = 0; i < N; ++i) { qpl[i] = lo[i] - x[i]; qpu[i] = up[i] - x[i]; }
                QPCounters qc{0, 0};
                const int qps = boxqp_small<T, N>(st.qpSettings, JJ, lambda, Jy, qpl, qpu, dX, qc);   // LS:1078-1080
                sSolves += qc.solves; sQPIt += qc.iterations;
                if (qps != mir_qp_solved) { status = mir_ls_numericError; break; }           // LS:1080-1085
                {
                    bool nan = false;                                                        // LS:1087-1092
#pragma unroll
                    for (int i = 0; i < N; ++i) nan = nan || !(dX[i] <= dX[i]);
                    if (nan) { status = mir_ls_numericError; break; }
                }
                T nd = (T)0;                                                                 // LS:1096-1099
#pragma unroll
                for (int i = 0; i < N; ++i) { dX[i] = add_rn(add_rn(dX[i], x[i]), -x[i]); nd += dX[i] * dX[i]; }

                if (!(sqrt_ni(nd) < st.maxStep)) { lambda *= st.lambdaIncrease * mu; mu *= (T)2; continue; }   // LS:1101-1106

                T xt[N];                                                                     // LS:1108-1110
                bool same = true;
#pragma unroll
                for (int i = 0; i < N; ++i) {
                    xt[i] = t_max(t_min(add_rn(dX[i], x[i]), up[i]), lo[i]);
                    same = same && (xt[i] == x[i]) && (signbit(xt[i]) == signbit(x[i]));
                }
                ++ret.fCalls;                                                                // LS:1112
                T trial;
                if (same) trial = ret.residual;         // f(xt) == y bit for bit: skip the evaluation
                else      trial = eval(xt, mb);                                              // LS:1113-1115
                if (!(trial <= Num<T>::inf())) { status = mir_ls_numericError; break; }      // LS:1117-1122

                const T improvement = ret.residual - trial;                                  // LS:1124-1130
                if (!(improvement > (T)0)) { lambda *= st.lambdaIncrease * mu; mu *= (T)2; continue; }

                needJacobian = true; mu = (T)1; ++iterations; ++sAccepted;                   // LS:1132-1139
#pragma unroll
                for (int i = 0; i < N; ++i) x[i] = xt[i];
#pragma unroll
                for (int k = 0; k < R; ++k) { const T tmp = mb[k]; mb[k] = yv[k]; yv[k] = tmp; }
                ret.residual = trial;
                fConverged = ret.residual <= st.maxGoodResidual;
                deltaX_dot = nd;

                T pred = (T)0;                                                               // LS:1141-1142
#pragma unroll
                for (int i = 0; i < N; ++i) {
                    T acc = (T)0;
#pragma unroll
                    for (int j = 0; j < N; ++j) acc += JJ[trisym(i, j)] * dX[j];
                    Jy[i] = acc + (T)2 * Jy[i];          // symv(Lower, 1, JJ, deltaX, 2, Jy): Jy is scratch from here
                    pred += Jy[i] * dX[i];
                }
                pred = -pred;
                if (!(pred > (T)0)) { status = mir_ls_furtherImprovement; break; }           // LS:1144-1148

                const T rho = div_ni(pred, improvement);                                            // LS:1150
                if (rho < st.minStepQuality) { lambda *= st.lambdaIncrease * mu; mu *= (T)2; }   // LS:1152-1156
                else if (rho >= st.goodStepQuality) lambda = t_max(st.lambdaDecrease * lambda * mu, st.minLambda);   // LS:1158-1161

                // LS:1164: !(sqrt(dd) > absTol && nrm2(x) > sqrt(dd) * relTol)
                T xmax = (T)0;
#pragma unroll
                for (int i = 0; i < N; ++i) xmax = t_max(xmax, t_abs(x[i]));
                T xn = (T)0;
                if (xmax > (T)0) {
                    const T inv = rcp_ni(xmax);
                    T ss = (T)0;
#pragma unroll
                    for (int i = 0; i < N; ++i) { const T v = x[i] * inv; ss += v * v; }
                    xn = xmax * sqrt_ni(ss);
                }
                const T sd = sqrt_ni(deltaX_dot);
                if (!(sd > st.absTolerance && xn > sd * st.relTolerance)) {                  // LS:1164-1173
                    if (age == 0) { status = mir_ls_xConverged; break; }
                    age = maxAge;
                    continue;
                }
            } while (iterations < st.maxIterations);                                         // LS:1175

            ret.status = status;
            ret.iterations = iterations;
            ret.lambda = lambda;
        }

        if (glane == 0) {
            T* xp = static_cast<T*>(args.x) + prob * N;
#pragma unroll
            for (int i = 0; i < N; ++i) xp[i] = x[i];
            static_cast<Result*>(args.results)[prob] = ret;
        }
    }

    if (args.stats && glane == 0 && sProblems) {
        atomicAdd((unsigned long long*)&args.stats->problems, sProblems);
        atomicAdd((unsigned long long*)&args.stats->passes, sPasses);
        atomicAdd((unsigned long long*)&args.stats->accepted, sAccepted);
        atomicAdd((unsigned long long*)&args.stats->fresh_jacobians, sFresh);
        atomicAdd((unsigned long long*)&args.stats->broyden_updates, sBroyden);
        atomicAdd((unsigned long long*)&args.stats->model_evals, sEvals);
        atomicAdd((unsigned long long*)&args.stats->qp_solves, sSolves);
        atomicAdd((unsigned long long*)&args.stats->qp_iterations, sQPIt);
    }
}

}  // namespace mirb200
