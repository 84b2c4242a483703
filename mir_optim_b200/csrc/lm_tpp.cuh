// lm_tpp.cuh -- batched Levenberg-Marquardt, one THREAD per problem, for large batches of small problems
// (BASELINE configs[1], [2], [4]b).  Follows optimizeLeastSquaresImplGeneric!T, least_squares.d:877-1176.
//
// Why not a warp (or sub-warp group) per problem, as lm_small.cuh does: the n-sized part of a pass (BOXCQP /
// posvx / lambda control, ~55 % of the instructions at n = 4) is serial, so a group of L lanes executes it L
// times redundantly, and different problems in one warp diverge (measured on B200: 18 of 32 lanes active,
// FP64 pipe 20 % busy, 5.9 M fits/s).  With one thread per problem nothing is replicated and no shuffle or
// barrier is needed; the price is that the m-sized per-problem state no longer fits in registers.
//
// Data layout.  Per thread: x, bounds, trial point, step, J^T r, packed lower J^T J, lambda/mu/age and the
// counters live in registers.  The m-sized vectors -- observations, y (current residuals), mBuffer (trial /
// previous residuals), the Broyden vector v and the m x n Jacobian that the Broyden update needs in place
// (LS:1003-1006) -- live in a per-CTA slab in global memory laid out [element][thread], so the 32 problems of
// a warp read and write 32 consecutive values: every access is a fully coalesced 256-byte (double) transaction.
//
// Lock-step state machine.  All threads of a warp walk the same phase sequence once per warp pass
//     fetch -> guards -> [FD Jacobian] -> g-test -> step (BOXCQP) -> row phase -> accept/reject
// and a phase a problem does not need is predicated off, so the warp reconverges after every phase; a thread
// that finishes its problem pulls the next index from an atomic counter at the next pass boundary.
//
// ONE row loop per pass.  A separate Jacobian phase would run with a third of the lanes (only problems whose last
// step was accepted need it; ncu, round 1: 50 % of the warp instructions at 8.7 of 32 lanes, every row iteration
// exposing a full memory round trip).  Instead the trial evaluation f(x + delta) (LS:1113) also does, row by row
// and SPECULATIVELY, what the next pass's Jacobian step would do if the trial is accepted:
//   * Broyden (age < maxAge):  v = ((y_old - f_new) + J delta) * (-1/|delta|^2),  J_new = J + v delta'  (LS:999-1006)
//   * fresh analytic Jacobian at the trial point (age == maxAge; g(x, J), LS:1011-1015) -- it shares exp() with f
//   * J_new' f_new and J_new' J_new (LS:1052, 1065) in registers.
// If the trial is rejected the speculative results are dropped; if it is accepted they ARE the next pass's
// Jacobian step, operation for operation (same operands, same order), so results are bit-identical to doing it
// afterwards.  The Jacobian in memory is updated lazily: a speculative pass stores only v; J_mem + v_p delta_p'
// (the pending term of the last accepted step) is materialised in place by the next row pass that reads J --
// in place is safe because the pending term belongs to an already accepted step.  A speculative FRESH Jacobian is
// stored in place directly: with age == maxAge the old J is dead (the next Jacobian operation is a fresh one on
// every path).  The few cases speculation cannot cover -- a forced fresh Jacobian at the current point (LS:984-989,
// 1059-1061, 1171) -- run the same row loop in INSTALL mode (recompute f(x), bit-identical to y, and build J at x),
// and that problem solves its QP one warp pass later.  Finite-difference fresh Jacobians (2n evaluations,
// LS:1018-1049) keep their own phase.
//
// Equivalences (bit-exact w.r.t. this file's arithmetic; same as lm_small.cuh): J^T J rebuilt only when J
// changed; trial == x skips the model evaluation; the inert lambda-overflow tail is fast-forwarded.
#pragma once
#include "lm_small.cuh"

namespace mirb200 {

constexpr int TPP_THREADS = 128;
enum { JAC_NONE_ = 0, JAC_BROYDEN_ = 1, JAC_FRESH_ = 2 };
enum { ROW_NONE_ = 0, ROW_EVAL_ = 1, ROW_INSTALL_ = 2 };

// number of slab vectors of length m per thread besides the m x N Jacobian
// (stored-J scheme: [yobs] buf0 buf1 v + m x N Jacobian;  v-list scheme: [yobs] buf0 buf1 v0 v1 v2, no Jacobian)
constexpr int TPP_VLN = 3;          // Broyden terms the v-list scheme can hold = largest maxAge it serves
template <int N, bool YOS, bool VL> struct TppSlab { static constexpr int ELEMS = (YOS ? 2 : 3) + (VL ? TPP_VLN : 1 + N); };

// YOS: the observations of the thread's current problem live in shared memory ([row][thread], conflict-free)
// instead of the slab -- they are read by every model evaluation, the most frequent phase.
// VL ("v-list", analytic Jacobians with maxAge <= TPP_VLN only): the Jacobian is never stored.  Between two fresh
// Jacobians at most maxAge Broyden terms exist, so the current J row is rebuilt on the fly as
//     ((g_row(x_anchor) + v_1 d_1') + v_2 d_2') + v_3 d_3'
// -- the same operations in the same order as the in-place updates (LS:1006), hence the same bits -- from the anchor
// point (registers), the accepted steps d_k (shared memory) and the vectors v_k (slab).  One extra exp per row buys
// a 3x smaller memory stream (ncu, round 1: the stored-J row loop moved 233 KB per fit and ran at 44 % of HBM
// bandwidth with 12 % occupancy) and a slab that fits the L2.
template <class Model, class T, bool FD, bool YOS, bool VL>
__global__ void __launch_bounds__(TPP_THREADS, 1)
lm_tpp_kernel(const typename Num<T>::Settings st, const SmallBatchArgs args, T* __restrict__ slabBase)
{
    constexpr int N = Model::N;
    constexpr int NP = N * (N + 1) / 2;
    constexpr int NT = TPP_THREADS;
    using Result = typename Num<T>::Result;
    const int m = (int)args.m;
    const int tid = threadIdx.x;
    const bool gridPerProblem = (args.flags & MIR_MODEL_GRID_PER_PROBLEM) != 0;
    const bool tailShortcut = (args.flags & MIR_MODEL_NO_TAIL_SHORTCUT) == 0;
    const T* __restrict__ tptr = static_cast<const T*>(args.t);
    const T* __restrict__ yptr = static_cast<const T*>(args.y);

    // abscissa shared by every problem: one copy in shared memory, then (YOS) the observations
    extern __shared__ __align__(16) unsigned char tpp_smem[];
    T* const st_ = reinterpret_cast<T*>(tpp_smem);

    static_assert(!(VL && FD), "the v-list scheme needs an analytic Jacobian");
    // slab of this CTA: [yobs m (only !YOS)][buf0 m][buf1 m][v m (x TPP_VLN if VL)][J m*N (not VL)], each element strided by NT
    T* const slab = slabBase + (size_t)blockIdx.x * ((size_t)m * TppSlab<N, YOS, VL>::ELEMS) * NT + tid;
    const int mPad = (m + 1) & ~1;
    T* const pYO = YOS ? st_ + mPad + tid : slab;
    T* const pB0 = slab + (size_t)(YOS ? 0 : 1) * m * NT;
    T* const pB1 = pB0 + (size_t)m * NT;
    T* const pV = pB1 + (size_t)m * NT;
    T* const pJ = pV + (size_t)m * NT;                                         // (stored-J scheme only)
    // accepted steps d_k of the v-list, [k][i][thread] in shared memory
    T* const pDL = st_ + mPad + (YOS ? (size_t)m * NT : 0) + tid;
    auto DL = [&](int k, int i) -> T& { return pDL[(k * N + i) * NT]; };
    auto YO = [&](int row) -> T& { return pYO[row * NT]; };
    auto JE = [&](int row, int i) -> T& { return pJ[(row * N + i) * NT]; };

    if (Model::kHasData && !gridPerProblem) {
        for (int row = tid; row < m; row += NT) st_[row] = tptr[row];
        __syncthreads();
    }

    // per-thread work counters (32 bits: a thread sees far fewer than 2^32 passes per launch)
    unsigned sPasses = 0, sAccepted = 0, sFresh = 0, sBroyden = 0, sEvals = 0, sSolves = 0, sQPIt = 0, sProblems = 0;

    // per-problem state
    bool active = false, retired = false, init = false;
    bool resume = false;        // the Jacobian of this pass was just built by an INSTALL row pass: continue at the g-test
    bool specOK = false;        // J / JJ / Jy already hold what the next Jacobian step (of kind specKind) produces
    bool pend = false;          // stored-J: current J = J_mem + v dXp' (pending rank-1 term of the last accepted step)
    int nterm = 0;              // v-list: Broyden terms accepted since the anchor
    int specKind = JAC_NONE_;
    unsigned long long prob = 0;
    const T* tp = st_;
    T x[N], xt[N], dX[N], Jy[N], JJ[NP];      // (bounds are re-read from global memory where needed)
    T dXp[N];                   // stored-J: step of the pending term;  v-list: the anchor point of the last fresh Jacobian
    const T* lp = static_cast<const T*>(args.l);
    const T* upp = static_cast<const T*>(args.u);
    T lambda = (T)0, mu = (T)1, residual = Num<T>::inf(), deltaX_dot = (T)0, nd = (T)0;
    unsigned age = 0, maxAge = 1, iterations = 0, fCalls = 0, gCalls = 0;
    int status = mir_ls_numericError, ysel = 0;
    bool needJacobian = false, fConverged = false;
#pragma unroll
    for (int i = 0; i < N; ++i) { x[i] = xt[i] = dX[i] = dXp[i] = Jy[i] = (T)0; }
#pragma unroll
    for (int i = 0; i < NP; ++i) JJ[i] = (T)0;

    for (;;) {
        // ------------------------------------------------------------------ fetch
        if (!active && !retired) {
            const unsigned int idx = atomicAdd(args.counter, 1u);
            if (idx >= args.batch) retired = true;
            else if (!wait_staged(args.ready, idx, args.spin_limit)) {
                // inputs never arrived: the host discards this launch (flag ready[1]); do not touch x
                Result ret;
                ret.status = mir_ls_numericError; ret.iterations = 0; ret.fCalls = 0; ret.gCalls = 0; ret.residual = Num<T>::inf(); ret.lambda = (T)0;
                static_cast<Result*>(args.results)[idx] = ret;
                ++sProblems;
            } else {
                prob = idx; ++sProblems;
                const T* xp = static_cast<const T*>(args.x) + prob * N;
                lp = static_cast<const T*>(args.l) + prob * args.bound_stride;
                upp = static_cast<const T*>(args.u) + prob * args.bound_stride;
#pragma unroll
                for (int i = 0; i < N; ++i) x[i] = xp[i];
                // validation, LS:930-943 (first failure wins)
                bool finite = true, inb = true;
#pragma unroll
                for (int i = 0; i < N; ++i) {
                    finite = finite && (-Num<T>::inf() < x[i] && x[i] < Num<T>::inf());
                    inb = inb && (lp[i] <= x[i]) && (x[i] <= upp[i]);
                }
                int vs = 0;
                if (m == 0 || !finite) vs = mir_ls_badGuess;
                else if (!inb) vs = mir_ls_badBounds;
                else if (!((T)0 <= st.minStepQuality && st.minStepQuality < (T)1)) vs = mir_ls_badMinStepQuality;
                else if (!((T)0 <= st.goodStepQuality && st.goodStepQuality <= (T)1)) vs = mir_ls_badGoodStepQuality;
                else if (!(st.minStepQuality < st.goodStepQuality)) vs = mir_ls_badStepQuality;
                else if (!((T)1 <= st.lambdaIncrease && st.lambdaIncrease <= Num<T>::sqrt_max())) vs = mir_ls_badLambdaParams;
                else if (!(Num<T>::sqrt_min_normal() <= st.lambdaDecrease && st.lambdaDecrease <= (T)1)) vs = mir_ls_badLambdaParams;
                if (vs) {
                    Result ret;
                    ret.status = vs; ret.iterations = 0; ret.fCalls = 0; ret.gCalls = 0; ret.residual = Num<T>::inf(); ret.lambda = (T)0;
                    static_cast<Result*>(args.results)[prob] = ret;          // x is left untouched
                } else {
                    active = true; init = true; resume = false; specOK = false; pend = false; nterm = 0; specKind = JAC_NONE_;
                    tp = gridPerProblem ? tptr + prob * (unsigned long long)m : st_;
                    if (Model::kHasData) {
                        const T* yp = yptr + prob * (unsigned long long)m;
#pragma unroll 8
                        for (int row = 0; row < m; ++row) YO(row) = yp[row];
                    }
#pragma unroll
                    for (int i = 0; i < N; ++i) { xt[i] = x[i]; Jy[i] = (T)0; dX[i] = (T)0; }
                    maxAge = st.maxAge ? st.maxAge : (FD ? 2u * N : 3u);                             // LS:945
                    ysel = 0; iterations = 0; fCalls = 0; gCalls = 0; status = mir_ls_maxIterations;
                    residual = Num<T>::inf(); lambda = (T)0; mu = (T)1; deltaX_dot = (T)0;     // (warm start: the launcher sends those batches to the lane-group / general kernels -- this kernel sits on a register-allocation cliff, the extra load cost 2 %)
                    age = maxAge; needJacobian = false; fConverged = false;
                }
            }
        }
        if (__all_sync(0xffffffffu, retired)) break;

        // ------------------------------------------------------------------ guards of this pass, LS:974-995, and the Jacobian decision, LS:996-1015
        int rowMode = ROW_NONE_, rowKind = JAC_NONE_;
        bool skipRest = false, finished = false, gtest = false, fdFresh = false;
        if (active) {
            if (init) {
                // initial residual, LS:953-956; the first Jacobian step is always a fresh one at x (age == maxAge)
                rowMode = ROW_EVAL_; rowKind = FD ? JAC_NONE_ : JAC_FRESH_;
            } else if (resume) {
                resume = false; gtest = true;                   // Jacobian step of this pass done by the INSTALL row pass
            } else {
                ++sPasses;
                if (fConverged) { status = mir_ls_fConverged; finished = true; }                         // LS:974-978
                else if (!(lambda <= st.maxLambda)) { status = mir_ls_furtherImprovement; finished = true; }   // LS:979-983
                else {
                    if (mu > (T)16 && age) { needJacobian = true; age = maxAge; mu = (T)1; specOK = false; }   // LS:984-989
                    bool nan = false;                                                                    // LS:990-995
#pragma unroll
                    for (int i = 0; i < N; ++i) nan = nan || !(x[i] <= x[i]);
                    if (nan) { status = mir_ls_numericError; finished = true; }
                    else if (!needJacobian && age == 0 && tailShortcut && tail_is_inert<T, N>(x, Jy, JJ, lambda, lp, upp, st)) {
                        for (;;) {                         // replay LS:1112, 1125-1130 and the next pass's LS:979-983
                            ++fCalls;
                            lambda *= st.lambdaIncrease * mu; mu *= (T)2;
                            ++sPasses;
                            if (!(lambda <= st.maxLambda)) break;
                        }
                        status = mir_ls_furtherImprovement; finished = true;
                    } else if (needJacobian) {                                                           // LS:996-998
                        needJacobian = false;
                        int mode;
                        if (age < maxAge) { ++age; mode = JAC_BROYDEN_; ++sBroyden; }                    // LS:999-1007
                        else { age = 0; mode = JAC_FRESH_; ++sFresh; if (FD) fCalls += N; else gCalls += 1; }   // LS:1010-1015, 1049
                        if (specOK && specKind == mode) gtest = true;            // built speculatively by the accepted trial's row pass
                        else if (FD && mode == JAC_FRESH_) { fdFresh = true; gtest = true; }
                        else { rowMode = ROW_INSTALL_; rowKind = mode; }
                        specOK = false;
                    }
                }
            }
        }

        // ------------------------------------------------------------------ finite-difference fresh Jacobian, LS:1018-1049 (+ J^T y, J^T J)
        if constexpr (FD) {
            if (active && !finished && fdFresh) {
#pragma unroll 1
                for (int j = 0; j < N; ++j) {
                    T save = (T)0, lj = (T)0, uj = (T)0;
#pragma unroll
                    for (int i = 0; i < N; ++i) if (i == j) { save = x[i]; lj = lp[i]; uj = upp[i]; }
                    const T xmh = t_max(save - st.jacobianEpsilon, lj);
                    const T xph = t_min(save + st.jacobianEpsilon, uj);
                    const T twh = xph - xmh;
                    if (twh != (T)0) {
                        T pp[N], pm[N];
#pragma unroll
                        for (int i = 0; i < N; ++i) { pp[i] = (i == j) ? xph : x[i]; pm[i] = (i == j) ? xmh : x[i]; }
                        const typename Model::Pre prep = Model::prepare(pp);
                        const typename Model::Pre prem = Model::prepare(pm);
                        const T rt = rcp_ni(twh);
                        constexpr int NE = Model::NE;
#pragma unroll 1
                        for (int row = 0; row < m; row += 2) {
                            const bool two = row + 1 < m;
                            const int rowB = two ? row + 1 : row;
                            const T t0 = Model::kHasData ? tp[row] : (T)0, y0 = Model::kHasData ? YO(row) : (T)0;
                            const T t1 = Model::kHasData ? tp[rowB] : (T)0, y1 = Model::kHasData ? YO(rowB) : (T)0;
                            T ea[4 * NE], ee[4 * NE];                     // the exps of f(x+h), f(x-h) for both rows, interleaved
                            Model::exp_args(prep, pp, t0, ea); Model::exp_args(prem, pm, t0, ea + NE);
                            Model::exp_args(prep, pp, t1, ea + 2 * NE); Model::exp_args(prem, pm, t1, ea + 3 * NE);
                            exp_repro_many<4 * NE>(ea, ee);
                            T fp0, fm0, fp1, fm1;
                            Model::finish_r(prep, pp, t0, y0, ee, fp0); Model::finish_r(prem, pm, t0, y0, ee + NE, fm0);
                            Model::finish_r(prep, pp, t1, y1, ee + 2 * NE, fp1); Model::finish_r(prem, pm, t1, y1, ee + 3 * NE, fm1);
                            JE(row, j) = (fp0 - fm0) * rt;                                               // LS:1040-1042
                            if (two) JE(rowB, j) = (fp1 - fm1) * rt;
                        }
                        sEvals += 2;
                    } else {
#pragma unroll 1
                        for (int row = 0; row < m; ++row) JE(row, j) = (T)0;                             // LS:1045-1047
                    }
                }
                pend = false;
                T pJy[N], pJJ[NP];
#pragma unroll
                for (int i = 0; i < N; ++i) pJy[i] = (T)0;
#pragma unroll
                for (int i = 0; i < NP; ++i) pJJ[i] = (T)0;
                const T* const yv = ysel ? pB1 : pB0;
#pragma unroll 2
                for (int row = 0; row < m; ++row) {                                                      // LS:1052, 1065
                    const T yr = yv[row * NT];
                    T Jr[N];
#pragma unroll
                    for (int i = 0; i < N; ++i) Jr[i] = JE(row, i);
#pragma unroll
                    for (int i = 0; i < N; ++i) {
                        pJy[i] += Jr[i] * yr;
#pragma unroll
                        for (int j = 0; j <= i; ++j) pJJ[tri(i, j)] += Jr[i] * Jr[j];
                    }
                }
#pragma unroll
                for (int i = 0; i < N; ++i) Jy[i] = pJy[i];
#pragma unroll
                for (int i = 0; i < NP; ++i) JJ[i] = pJJ[i];
            }
        }

        // ------------------------------------------------------------------ gradient test, LS:1053-1062
        if (active && !finished && gtest) {
            T gsel = Jy[0]; T gbest = t_abs(Jy[0]);                                                      // iamax: first max |.|
#pragma unroll
            for (int i = 1; i < N; ++i) { const T v = t_abs(Jy[i]); if (v > gbest) { gbest = v; gsel = Jy[i]; } }
            if (!(t_abs(gsel) > st.gradTolerance)) {
                if (age == 0) { status = mir_ls_gConverged; finished = true; }
                else { age = maxAge; skipRest = true; }
            }
        }

        // ------------------------------------------------------------------ step: lambda init, BOXCQP, trial point
        if (active && !finished && !init && !skipRest && rowMode != ROW_INSTALL_) {
            if (!(lambda >= st.minLambda)) {                                                             // LS:1067-1072
                T dmax = JJ[0];
#pragma unroll
                for (int i = 1; i < N; ++i) if (t_abs(JJ[tri(i, i)]) > t_abs(dmax)) dmax = JJ[tri(i, i)];
                lambda = (T)(0.001 * (double)dmax);
                if (!(lambda >= st.minLambda)) lambda = (T)1;
            }
            T qpl[N], qpu[N], lo[N], up[N];                                                              // LS:1074-1077
#pragma unroll
            for (int i = 0; i < N; ++i) { lo[i] = lp[i]; up[i] = upp[i]; qpl[i] = lo[i] - x[i]; qpu[i] = up[i] - x[i]; }
            QPCounters qc{0, 0};
            const int qps = boxqp_small<T, N>(st.qpSettings, JJ, lambda, Jy, qpl, qpu, dX, qc);          // LS:1078-1080
            sSolves += qc.solves; sQPIt += qc.iterations;
            bool nan = false;                                                                            // LS:1087-1092
#pragma unroll
            for (int i = 0; i < N; ++i) nan = nan || !(dX[i] <= dX[i]);
            if (qps != mir_qp_solved || nan) { status = mir_ls_numericError; finished = true; }          // LS:1080-1092
            else {
                nd = (T)0;                                                                               // LS:1096-1099
#pragma unroll
                for (int i = 0; i < N; ++i) { dX[i] = add_rn(add_rn(dX[i], x[i]), -x[i]); nd += dX[i] * dX[i]; }
                if (!(sqrt_ni(nd) < st.maxStep)) { lambda *= st.lambdaIncrease * mu; mu *= (T)2; skipRest = true; }   // LS:1101-1106
                else {
                    bool same = true;                                                                    // LS:1108-1110
#pragma unroll
                    for (int i = 0; i < N; ++i) {
                        xt[i] = t_max(t_min(add_rn(dX[i], x[i]), up[i]), lo[i]);
                        same = same && (xt[i] == x[i]) && (signbit(xt[i]) == signbit(x[i]));
                    }
                    ++fCalls;                                                                            // LS:1112
                    // f(xt) == y bit for bit when xt == x: evaluation skipped, trial = residual (a rejection)
                    if (!same) {
                        rowMode = ROW_EVAL_;
                        // what the next pass's Jacobian step will be if this trial is accepted (mu = 1 after an accept,
                        // so LS:984-989 cannot intervene; LS:1171 can still force a fresh one: checked at the guards)
                        rowKind = (age < maxAge) ? JAC_BROYDEN_ : (FD ? JAC_NONE_ : JAC_FRESH_);
                    }
                }
            }
        }

        // ------------------------------------------------------------------ row phase: f (LS:953, 1113) + Jacobian step of the next pass (LS:999-1015, 1052, 1065)
        T trial = residual;
        T pJy[N], pJJ[NP];
        if (active && !finished && rowMode != ROW_NONE_) {
            const bool isEval = rowMode == ROW_EVAL_;
            const bool kB = rowKind == JAC_BROYDEN_, kF = rowKind == JAC_FRESH_;
            const bool pnd = kB && pend;
            if (!isEval) {                                      // INSTALL evaluates at x (xt is scratch until the next QP)
#pragma unroll
                for (int i = 0; i < N; ++i) xt[i] = x[i];
            }
            const typename Model::Pre pre = Model::prepare(xt);
            // EVAL: f goes to mBuffer (the buffer that is not y), the previous point's residuals are y.
            // INSTALL: f(x) is recomputed (== y, not stored), the previous point's residuals are mBuffer.
            T* const out = ysel ? pB0 : pB1;
            const T* const fold = isEval ? (ysel ? pB1 : pB0) : (ysel ? pB0 : pB1);
            const T negd = kB ? -rcp_ni(isEval ? nd : deltaX_dot) : (T)0;                                // LS:1001
#pragma unroll
            for (int i = 0; i < N; ++i) pJy[i] = (T)0;
#pragma unroll
            for (int i = 0; i < NP; ++i) pJJ[i] = (T)0;
            T acc2 = (T)0;

            constexpr int NE = Model::NE;
            if constexpr (VL) {
                const int k = nterm;                             // terms already in the list; this pass computes term k
                T* const pVk = pV + (size_t)k * m * NT;
                T anchor[N], d0[N], d1[N];
#pragma unroll
                for (int i = 0; i < N; ++i) {
                    anchor[i] = kB ? dXp[i] : xt[i];
                    d0[i] = (kB && k > 0) ? DL(0, i) : (T)0;
                    d1[i] = (kB && k > 1) ? DL(1, i) : (T)0;
                }
                const typename Model::Pre preA = Model::prepare(anchor);
                // slab values are loaded a pair of rows ahead (global-memory latency); abscissa and observation come from
                // shared memory at compute time
                struct RowIn { T fo, v0, v1; };
                auto rowLoad = [&](int row, RowIn& in, bool on) {
                    in.fo = (kB && on) ? fold[row * NT] : (T)0;
                    in.v0 = (kB && k > 0 && on) ? pV[row * NT] : (T)0;
                    in.v1 = (kB && k > 1 && on) ? *(pV + (size_t)m * NT + row * NT) : (T)0;
                };
                // Branch-free: every lane runs the Broyden arithmetic (selects pick the result, loads and stores are
                // predicated).  eT / eA: the exps of this row at the trial point and at the anchor.
                auto rowFinish = [&](int row, const RowIn& in, T tt, T yo, const T* eT, const T* eA, bool on) {
                    T r, Jf[N], Jr[N], Jn[N];
                    Model::finish_rj(pre, xt, tt, yo, eT, r, Jf);                     // f and the fresh-Jacobian candidate
                    Model::finish_j(preA, anchor, tt, eA, Jr);                        // g_row(x_anchor), then the accepted terms
                    // Terms beyond the list length have v = 0 and d = 0 (rowLoad / d0, d1 above), so applying both terms
                    // unconditionally changes nothing but the sign of an exact zero entry (-0 + (+0) = +0).  A zero of J only
                    // ever meets the accumulators below through products that are themselves zeros, and an accumulator that
                    // starts at +0 stays +0 under either sign: x, ||r||^2, lambda and every counter are bit-identical to the
                    // selected form, which cost 16 extra select instructions per row.
#pragma unroll
                    for (int i = 0; i < N; ++i) {
                        Jr[i] = fma(in.v0, d0[i], Jr[i]);
                        Jr[i] = fma(in.v1, d1[i], Jr[i]);
                    }
                    T acc = (T)0;                                                     // LS:1002-1006
#pragma unroll
                    for (int i = 0; i < N; ++i) acc = fma(Jr[i], dX[i], acc);
                    const T v = ((in.fo - r) + acc) * negd;
#pragma unroll
                    for (int i = 0; i < N; ++i) Jn[i] = kB ? fma(v, dX[i], Jr[i]) : Jf[i];
                    if (kB && on) pVk[row * NT] = v;
                    if (isEval && on) out[row * NT] = r;
                    if (on) {
                        acc2 = fma(r, r, acc2);
#pragma unroll
                        for (int i = 0; i < N; ++i) {                                 // LS:1052, 1065
                            pJy[i] = fma(Jn[i], r, pJy[i]);
#pragma unroll
                            for (int j = 0; j <= i; ++j) pJJ[tri(i, j)] = fma(Jn[i], Jn[j], pJJ[tri(i, j)]);
                        }
                    }
                };
                // A pair of rows: four independent exp batches (2 rows x {trial point, anchor}) in one interleaved call.
                auto pairCompute = [&](int row, const RowIn& A, const RowIn& B, bool two) {
                    const int rowB = two ? row + 1 : row;
                    const T ta = Model::kHasData ? tp[row] : (T)0, ya = Model::kHasData ? YO(row) : (T)0;
                    const T tb = Model::kHasData ? tp[rowB] : (T)0, yb = Model::kHasData ? YO(rowB) : (T)0;
                    T ea[4 * NE], ee[4 * NE];
                    Model::exp_args(pre, xt, ta, ea); Model::exp_args(pre, xt, tb, ea + NE);
                    Model::exp_args(preA, anchor, ta, ea + 2 * NE); Model::exp_args(preA, anchor, tb, ea + 3 * NE);
                    exp_repro_many<4 * NE>(ea, ee);
                    rowFinish(row, A, ta, ya, ee, ee + 2 * NE, true);
                    rowFinish(row + 1, B, tb, yb, ee + NE, ee + 3 * NE, two);
                };
                int row = 0;
                RowIn ra, rb;
                rowLoad(0, ra, m >= 2); rowLoad(1, rb, m >= 2);
#pragma unroll 1
                for (; row + 2 <= m; row += 2) {
                    RowIn na, nb;
                    const bool more = row + 4 <= m;
                    rowLoad(row + 2, na, more); rowLoad(row + 3, nb, more);
                    pairCompute(row, ra, rb, true);
                    ra = na; rb = nb;
                }
                if (row < m) { rowLoad(row, ra, true); pairCompute(row, ra, ra, false); }
            } else {
                // Stored-J scheme.  One row = slab/shared loads (issued a pair of rows ahead: their latency hides behind
                // the previous pair's exp chains) + compute.
                struct RowIn { T fo, vp; T Jr[N]; };
                auto rowLoad = [&](int row, RowIn& in, bool on) {
#pragma unroll
                    for (int i = 0; i < N; ++i) in.Jr[i] = (kB && on) ? JE(row, i) : (T)0;
                    in.fo = (kB && on) ? fold[row * NT] : (T)0;
                    in.vp = (pnd && on) ? pV[row * NT] : (T)0;
                };
                auto rowFinish = [&](int row, RowIn& in, T tt, T yo, const T* eT, bool on) {
                    T r, Jn[N];
                    if constexpr (!FD) Model::finish_rj(pre, xt, tt, yo, eT, r, Jn);         // f and the fresh-Jacobian candidate
                    else {
                        Model::finish_r(pre, xt, tt, yo, eT, r);
#pragma unroll
                        for (int i = 0; i < N; ++i) Jn[i] = (T)0;
                    }
                    if (kB && on) {
                        if (pnd) {                                                  // materialise the pending rank-1 term
#pragma unroll
                            for (int i = 0; i < N; ++i) in.Jr[i] = fma(in.vp, dXp[i], in.Jr[i]);
                            if (isEval) {
#pragma unroll
                                for (int i = 0; i < N; ++i) JE(row, i) = in.Jr[i];
                            }
                        }
                        T acc = (T)0;                                               // LS:1002-1006
#pragma unroll
                        for (int i = 0; i < N; ++i) acc = fma(in.Jr[i], dX[i], acc);
                        const T v = ((in.fo - r) + acc) * negd;
#pragma unroll
                        for (int i = 0; i < N; ++i) Jn[i] = fma(v, dX[i], in.Jr[i]);
                        if (isEval) pV[row * NT] = v;
                    }
                    if (on && (kF || (kB && !isEval))) {
#pragma unroll
                        for (int i = 0; i < N; ++i) JE(row, i) = Jn[i];
                    }
                    if (isEval && on) out[row * NT] = r;
                    if (on) {
                        acc2 = fma(r, r, acc2);
#pragma unroll
                        for (int i = 0; i < N; ++i) {                               // LS:1052, 1065
                            pJy[i] = fma(Jn[i], r, pJy[i]);
#pragma unroll
                            for (int j = 0; j <= i; ++j) pJJ[tri(i, j)] = fma(Jn[i], Jn[j], pJJ[tri(i, j)]);
                        }
                    }
                };
                auto pairCompute = [&](int row, RowIn& A, RowIn& B, bool two) {
                    const int rowB = two ? row + 1 : row;
                    const T ta = Model::kHasData ? tp[row] : (T)0, ya = Model::kHasData ? YO(row) : (T)0;
                    const T tb = Model::kHasData ? tp[rowB] : (T)0, yb = Model::kHasData ? YO(rowB) : (T)0;
                    T ea[2 * NE], ee[2 * NE];
                    Model::exp_args(pre, xt, ta, ea); Model::exp_args(pre, xt, tb, ea + NE);
                    exp_repro_many<2 * NE>(ea, ee);
                    rowFinish(row, A, ta, ya, ee, true);
                    rowFinish(row + 1, B, tb, yb, ee + NE, two);
                };
                int row = 0;
                RowIn ra, rb;
                rowLoad(0, ra, m >= 2); rowLoad(1, rb, m >= 2);
#pragma unroll 1
                for (; row + 2 <= m; row += 2) {
                    RowIn na, nb;
                    const bool more = row + 4 <= m;
                    rowLoad(row + 2, na, more); rowLoad(row + 3, nb, more);
                    pairCompute(row, ra, rb, true);
                    ra = na; rb = nb;
                }
                if (row < m) { rowLoad(row, ra, true); rb = ra; pairCompute(row, ra, rb, false); }
            }
            if (isEval) { trial = acc2; ++sEvals; }
        }

        // ------------------------------------------------------------------ accept / reject, LS:1117-1175
        if (active && !finished) {
            const bool wasInit = init;
            bool passEnds = true;
            if (rowMode == ROW_INSTALL_) {
                // the Jacobian step of this pass (LS:996-1052, 1065) is done; g-test and QP follow in the next warp pass
#pragma unroll
                for (int i = 0; i < N; ++i) Jy[i] = pJy[i];
#pragma unroll
                for (int i = 0; i < NP; ++i) JJ[i] = pJJ[i];
                if constexpr (VL) {
                    if (rowKind == JAC_BROYDEN_) {
#pragma unroll
                        for (int i = 0; i < N; ++i) DL(nterm, i) = dX[i];
                        ++nterm;
                    } else {
#pragma unroll
                        for (int i = 0; i < N; ++i) dXp[i] = x[i];
                        nterm = 0;
                    }
                }
                pend = false; resume = true; passEnds = false;
            } else if (init) {                                                                           // LS:953-971
                init = false;
                residual = trial; ysel ^= 1; fCalls = 1;
                fConverged = residual <= st.maxGoodResidual;
                needJacobian = true; age = maxAge;
                if (rowKind == JAC_FRESH_) {
#pragma unroll
                    for (int i = 0; i < N; ++i) Jy[i] = pJy[i];
#pragma unroll
                    for (int i = 0; i < NP; ++i) JJ[i] = pJJ[i];
                    specOK = true; specKind = JAC_FRESH_; pend = false;
                    if constexpr (VL) {
#pragma unroll
                        for (int i = 0; i < N; ++i) dXp[i] = x[i];
                        nterm = 0;
                    }
                }
            } else if (!skipRest) {
                if (!(trial <= Num<T>::inf())) { status = mir_ls_numericError; finished = true; }        // LS:1117-1122
                else {
                    const T improvement = residual - trial;                                              // LS:1124
                    if (!(improvement > (T)0)) {                                                         // LS:1125-1130
                        lambda *= st.lambdaIncrease * mu; mu *= (T)2;
                        // rejected: a materialised pending term stays materialised, a speculative fresh J overwrote a dead J
                        if (rowMode == ROW_EVAL_ && rowKind != JAC_NONE_) pend = false;
                    } else {
                        needJacobian = true; mu = (T)1; ++iterations; ++sAccepted;                       // LS:1132-1139
#pragma unroll
                        for (int i = 0; i < N; ++i) x[i] = xt[i];
                        ysel ^= 1;
                        residual = trial;
                        fConverged = residual <= st.maxGoodResidual;
                        deltaX_dot = nd;
                        T pred = (T)0;                                                                   // LS:1141-1142
#pragma unroll
                        for (int i = 0; i < N; ++i) {
                            T acc = (T)0;
#pragma unroll
                            for (int j = 0; j < N; ++j) acc += JJ[trisym(i, j)] * dX[j];
                            Jy[i] = acc + (T)2 * Jy[i];
                            pred += Jy[i] * dX[i];
                        }
                        pred = -pred;
                        // the speculative Jacobian step becomes the state (used only if the run continues)
                        if (rowKind != JAC_NONE_) {
#pragma unroll
                            for (int i = 0; i < N; ++i) Jy[i] = pJy[i];
#pragma unroll
                            for (int i = 0; i < NP; ++i) JJ[i] = pJJ[i];
                            specOK = true; specKind = rowKind;
                            if constexpr (VL) {
                                if (rowKind == JAC_BROYDEN_) {
#pragma unroll
                                    for (int i = 0; i < N; ++i) DL(nterm, i) = dX[i];
                                    ++nterm;
                                } else {
#pragma unroll
                                    for (int i = 0; i < N; ++i) dXp[i] = x[i];
                                    nterm = 0;
                                }
                            } else {
                                pend = rowKind == JAC_BROYDEN_;
#pragma unroll
                                for (int i = 0; i < N; ++i) dXp[i] = dX[i];
                            }
                        }
                        if (!(pred > (T)0)) { status = mir_ls_furtherImprovement; finished = true; }     // LS:1144-1148
                        else {
                            const T rho = div_ni(pred, improvement);                                     // LS:1150
                            if (rho < st.minStepQuality) { lambda *= st.lambdaIncrease * mu; mu *= (T)2; }   // LS:1152-1156
                            else if (rho >= st.goodStepQuality) lambda = t_max(st.lambdaDecrease * lambda * mu, st.minLambda);   // LS:1158-1161
                            T xmax = (T)0;                                                               // LS:1164 (nrm2, scaled)
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
                                if (age == 0) { status = mir_ls_xConverged; finished = true; }
                                else age = maxAge;
                            }
                        }
                    }
                }
            }
            // LS:1175 (a do-while: the first pass always runs)
            if (passEnds && !wasInit && !finished && !(iterations < st.maxIterations)) { status = mir_ls_maxIterations; finished = true; }
        }

        if (active && finished) {
            T* xp = static_cast<T*>(args.x) + prob * N;
#pragma unroll
            for (int i = 0; i < N; ++i) xp[i] = x[i];
            Result ret;
            ret.status = status; ret.iterations = iterations; ret.fCalls = fCalls; ret.gCalls = gCalls;
            ret.residual = residual; ret.lambda = lambda;
            static_cast<Result*>(args.results)[prob] = ret;
            active = false;
        }
    }

    if (args.stats) {
        auto wsum = [](unsigned v32) {
            unsigned long long v = v32;
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
            return v;
        };
        const unsigned long long wProblems = wsum(sProblems), wPasses = wsum(sPasses), wAccepted = wsum(sAccepted), wFresh = wsum(sFresh);
        const unsigned long long wBroyden = wsum(sBroyden), wEvals = wsum(sEvals), wSolves = wsum(sSolves), wQPIt = wsum(sQPIt);
        if ((tid & 31) == 0 && wProblems) {
            atomicAdd((unsigned long long*)&args.stats->problems, wProblems);
            atomicAdd((unsigned long long*)&args.stats->passes, wPasses);
            atomicAdd((unsigned long long*)&args.stats->accepted, wAccepted);
            atomicAdd((unsigned long long*)&args.stats->fresh_jacobians, wFresh);
            atomicAdd((unsigned long long*)&args.stats->broyden_updates, wBroyden);
            atomicAdd((unsigned long long*)&args.stats->model_evals, wEvals);
            atomicAdd((unsigned long long*)&args.stats->qp_solves, wSolves);
            atomicAdd((unsigned long long*)&args.stats->qp_iterations, wQPIt);
        }
    }
}

}  // namespace mirb200
