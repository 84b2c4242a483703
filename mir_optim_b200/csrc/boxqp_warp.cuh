// boxqp_warp.cuh -- BOXCQP and ?posvx('E','L') restated for ONE WARP per QP, n <= 64 (BASELINE configs[4]a: n = 64).
//
//   posvx_warp  <- LAPACK dposvx/sposvx FACT='E', UPLO='L' as called at boxcqp.d:194-205, 310-321 (?poequ/?laqsy decision,
//                  Cholesky, ?potrs, ?porfs refinement with at most 5 corrections on the componentwise backward error).
//   boxqp_warp  <- solveBoxQP!T full overload, boxcqp.d:122-379 (unconstrainedSolution = false); active-set sub-systems are
//                  compacted through the ascending free-index list exactly like boxcqp.d:269-305.
//
// Why not a CTA per QP (boxqp_cta.cuh, which remains for 64 < n <= 128 and for the LM control kernels): at n = 64 the
// column loop of a 128-thread CTA is three CTA barriers per column with a handful of flops between them -- round-1 ncu:
// stall_barrier 5.5 of 10 cycles per issue, 463 M shared-memory bank conflicts, 216 us per QP and CTA, as slow as one CPU
// core.  A warp needs no barrier at all:
//   * lane L owns rows L and s-1-L of the current s x s system (the pairing evens out the triangular work); the factor
//     lives in shared memory as a packed lower triangle (16.6 KB at n = 64, nine warps per SM), a pivot column is
//     broadcast through a 64-entry buffer, the trailing update walks each lane's own rows;
//   * the triangular solves keep the right-hand side in registers (two entries per lane) and broadcast one solved entry per
//     column with a shuffle;
//   * P itself is never copied: only its lower triangle is read (boxcqp.d:288-302, 335), a lane's own row through L1
//     (sequential), the rest of a symmetric row as column entries, which are coalesced across the lanes.
#pragma once
#include "boxqp_small.cuh"   // KBN
#include "repro_math.cuh"

namespace mirb200 {

constexpr int WQP_NMAX = 64;
constexpr unsigned WQP_FULL = 0xffffffffu;

// Packed lower triangle, row i begins at wtri(i).
__host__ __device__ constexpr int wtri(int i) { return i * (i + 1) / 2; }

template <class T> struct WarpQPSmem {
    T F[WQP_NMAX * (WQP_NMAX + 1) / 2];    // packed lower factor of the current (sub-)system
    T q[WQP_NMAX], l[WQP_NMAX], u[WQP_NMAX], x[WQP_NMAX];   // by variable
    T b[WQP_NMAX], sx[WQP_NMAX];           // right-hand side / solution of the current (sub-)system, by compact index
    T col[WQP_NMAX], rdiag[WQP_NMAX], sc[WQP_NMAX];
    int idx[WQP_NMAX];                     // compact index -> variable, ascending
    signed char flag[WQP_NMAX];            // -1 lower, 0 free, +1 upper (boxcqp.d:153-158)
};

template <class T> __device__ __forceinline__ T warp_max(T v)
{
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) v = t_max(v, __shfl_xor_sync(WQP_FULL, v, off));
    return v;
}
template <class T> __device__ __forceinline__ T warp_min(T v)
{
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) v = t_min(v, __shfl_xor_sync(WQP_FULL, v, off));
    return v;
}

// A(a, c) for a >= c: the (unscaled) lower triangle of the s x s system.  b: sm.b (overwritten by its scaled copy),
// solution in sm.sx.  Returns LAPACK info (0, or k > 0: breakdown at pivot k), uniform over the warp.
template <class T, class AGet>
__device__ int posvx_warp(int s, AGet A, WarpQPSmem<T>& sm, int lane, int* equed_out = nullptr)
{
    const int nh = (s + 1) >> 1;
    const int r0 = lane, r1 = s - 1 - lane;
    const bool v0 = lane < nh, v1 = lane < (s >> 1);
    auto Asym = [&](int i, int c) -> T { return (i >= c) ? A(i, c) : A(c, i); };

    // ---- ?poequ / ?laqsy decision (single precision settles it unless the ratio is within 10 % of the threshold)
    const T d0 = v0 ? A(r0, r0) : (T)1, d1 = v1 ? A(r1, r1) : (T)1;
    bool equil = false;
    {
        const float f0 = (float)d0, f1 = (float)d1;
        float fmn = fminf(v0 ? f0 : __builtin_huge_valf(), v1 ? f1 : __builtin_huge_valf()), fmx = fmaxf(v0 ? f0 : 0.0f, v1 ? f1 : 0.0f);
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) {
            fmn = fminf(fmn, __shfl_xor_sync(WQP_FULL, fmn, off));
            fmx = fmaxf(fmx, __shfl_xor_sync(WQP_FULL, fmx, off));
        }
        const bool clearlyFine = fmn >= 0.011f * fmx && fmn > 0x1p-100f && fmx < 0x1p100f;
        if (!clearlyFine) {                    // (uniform: the reduced values are the same in every lane)
            const T smin = warp_min(t_min(v0 ? d0 : Num<T>::inf(), v1 ? d1 : Num<T>::inf()));
            const T amax = warp_max(t_max(v0 ? d0 : -Num<T>::inf(), v1 ? d1 : -Num<T>::inf()));
            if (smin > (T)0) {
                bool wellScaled;
                if (smin >= (T)0.0102 * amax) wellScaled = true;
                else if (smin <= (T)0.0098 * amax) wellScaled = false;
                else wellScaled = div_ni(sqrt_ni(smin), sqrt_ni(amax)) >= (T)0.1;
                equil = !(wellScaled && amax >= Num<T>::small_() && amax <= Num<T>::large_());
            }
        }
    }
    if (equed_out && lane == 0) *equed_out = equil ? 1 : 0;
    T sc0 = (T)1, sc1 = (T)1;
    if (equil) {
        if (v0) { sc0 = rcp_ni(sqrt_ni(d0)); sm.sc[r0] = sc0; }
        if (v1) { sc1 = rcp_ni(sqrt_ni(d1)); sm.sc[r1] = sc1; }
        __syncwarp();
    }
    // entry (i, c) of the equilibrated matrix (dlaqsy: cj * s(i) * A(i,j))
    auto Asc = [&](int i, T sci, int c) -> T { const T a = Asym(i, c); return equil ? (sm.sc[c] * sci) * a : a; };

    // ---- the lower triangle of the (equilibrated) system, packed, and the scaled right-hand side
    // (four independent loads in flight per row: the loop is latency-bound on L1 / L2 otherwise)
    auto fill_row = [&](int r, T scr) {
        T* Fr = sm.F + wtri(r);
        int c = 0;
        for (; c + 3 <= r; c += 4) {
            const T a0 = A(r, c), a1 = A(r, c + 1), a2 = A(r, c + 2), a3 = A(r, c + 3);
            if (equil) { Fr[c] = (sm.sc[c] * scr) * a0; Fr[c + 1] = (sm.sc[c + 1] * scr) * a1; Fr[c + 2] = (sm.sc[c + 2] * scr) * a2; Fr[c + 3] = (sm.sc[c + 3] * scr) * a3; }
            else { Fr[c] = a0; Fr[c + 1] = a1; Fr[c + 2] = a2; Fr[c + 3] = a3; }
        }
        for (; c <= r; ++c) Fr[c] = Asc(r, scr, c);
    };
    if (v0) fill_row(r0, sc0);
    if (v1) fill_row(r1, sc1);
    T b0 = v0 ? sm.b[r0] * sc0 : (T)0, b1 = v1 ? sm.b[r1] * sc1 : (T)0;         // dposvx: B := diag(S) B
    __syncwarp();

    // ---- ?potrf, right-looking.  The diagonal entry of L is kept as its reciprocal (rdiag), F keeps the pivot.
    for (int j = 0; j < s; ++j) {
        const T d = sm.F[wtri(j) + j];
        if (d <= (T)0) return j + 1;           // breakdown (uniform; a NaN pivot passes, as in OpenBLAS' potf2)
        T ljj, rinv;
        mux_sqrt_rcp(d, ljj, rinv);
        T l0 = (T)0, l1 = (T)0;
        if (v0 && r0 > j) { T* p = sm.F + wtri(r0) + j; l0 = *p * rinv; *p = l0; sm.col[r0] = l0; }
        if (v1 && r1 > j) { T* p = sm.F + wtri(r1) + j; l1 = *p * rinv; *p = l1; sm.col[r1] = l1; }
        if (lane == 0) sm.rdiag[j] = rinv;
        __syncwarp();
        {
            // both rows of the lane in one sweep over k (r0 <= r1: the pivot-column entry is loaded once for the two)
            T* F0 = sm.F + wtri(r0); T* F1 = sm.F + wtri(r1);
            const int e0 = (v0 && r0 > j) ? r0 : j, e1 = (v1 && r1 > j) ? r1 : ((v0 && r0 > j) ? r0 : j);
            int k = j + 1;
            for (; k + 1 <= e0; k += 2) {
                const T c0 = sm.col[k], c1 = sm.col[k + 1];
                const T a0 = F0[k], a1 = F0[k + 1], b0_ = F1[k], b1_ = F1[k + 1];
                F0[k] = fma(-l0, c0, a0); F0[k + 1] = fma(-l0, c1, a1);
                if (v1) { F1[k] = fma(-l1, c0, b0_); F1[k + 1] = fma(-l1, c1, b1_); }
            }
            for (; k <= e0; ++k) { const T c0 = sm.col[k]; F0[k] = fma(-l0, c0, F0[k]); if (v1) F1[k] = fma(-l1, c0, F1[k]); }
            if (v1 && r1 > j) {
                for (; k + 1 <= e1; k += 2) { const T c0 = sm.col[k], c1 = sm.col[k + 1]; const T b0_ = F1[k], b1_ = F1[k + 1]; F1[k] = fma(-l1, c0, b0_); F1[k + 1] = fma(-l1, c1, b1_); }
                for (; k <= e1; ++k) F1[k] = fma(-l1, sm.col[k], F1[k]);
            }
        }
        __syncwarp();
    }

    // L L^T z = v for the entries of my rows (in / out: z0, z1)
    auto solve = [&](T& z0, T& z1) {
        for (int j = 0; j < s; ++j) {                                  // forward, column j of L
            const bool lowHalf = j < nh;
            const T zj = __shfl_sync(WQP_FULL, lowHalf ? z0 : z1, lowHalf ? j : s - 1 - j) * sm.rdiag[j];
            if (lowHalf) { if (lane == j) z0 = zj; } else { if (lane == s - 1 - j) z1 = zj; }
            if (v0 && r0 > j) z0 = fma(-sm.F[wtri(r0) + j], zj, z0);
            if (v1 && r1 > j) z1 = fma(-sm.F[wtri(r1) + j], zj, z1);
        }
        for (int j = s - 1; j >= 0; --j) {                             // backward, row j of L (= column j of L^T)
            const bool lowHalf = j < nh;
            const T xj = __shfl_sync(WQP_FULL, lowHalf ? z0 : z1, lowHalf ? j : s - 1 - j) * sm.rdiag[j];
            if (lowHalf) { if (lane == j) z0 = xj; } else { if (lane == s - 1 - j) z1 = xj; }
            const T* Fj = sm.F + wtri(j);
            if (v0 && r0 < j) z0 = fma(-Fj[r0], xj, z0);
            if (v1 && r1 < j) z1 = fma(-Fj[r1], xj, z1);
        }
    };

    // ---- ?potrs, then ?porfs: pass 0 solves for b, later passes solve for the residual and correct x
    const T eps = Num<T>::lapack_eps();
    const T safe1 = (T)(s + 1) * Num<T>::safmin();
    const T safe2 = safe1 * ((T)1 / Num<T>::lapack_eps());
    T x0 = (T)0, x1 = (T)0, z0 = b0, z1 = b1, lstres = (T)3;
    for (int count = 0;; ++count) {
        solve(z0, z1);
        x0 += z0; x1 += z1;
        __syncwarp();
        if (v0) sm.sx[r0] = x0;
        if (v1) sm.sx[r1] = x1;
        __syncwarp();
        T rr0 = b0, rr1 = b1, w0 = t_abs(b0), w1 = t_abs(b1);
        {
            int c = 0;
            for (; c + 3 < s; c += 4) {                // eight independent loads in flight
                T a[4], g[4];
#pragma unroll
                for (int e = 0; e < 4; ++e) { a[e] = v0 ? Asc(r0, sc0, c + e) : (T)0; g[e] = v1 ? Asc(r1, sc1, c + e) : (T)0; }
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const T xc = sm.sx[c + e];
                    rr0 = fma(-a[e], xc, rr0); w0 = fma(t_abs(a[e]), t_abs(xc), w0);
                    rr1 = fma(-g[e], xc, rr1); w1 = fma(t_abs(g[e]), t_abs(xc), w1);
                }
            }
            for (; c < s; ++c) {
                const T xc = sm.sx[c];
                if (v0) { const T a = Asc(r0, sc0, c); rr0 = fma(-a, xc, rr0); w0 = fma(t_abs(a), t_abs(xc), w0); }
                if (v1) { const T a = Asc(r1, sc1, c); rr1 = fma(-a, xc, rr1); w1 = fma(t_abs(a), t_abs(xc), w1); }
            }
        }
        T qv = (T)0;                           // dporfs: berr = max_i |r_i| / (|b| + |A||x|)_i with the safe1 / safe2 guard
        if (v0) { const bool big = w0 > safe2; qv = div_ni(big ? t_abs(rr0) : t_abs(rr0) + safe1, big ? w0 : w0 + safe1); }
        if (v1) { const bool big = w1 > safe2; qv = t_max(qv, div_ni(big ? t_abs(rr1) : t_abs(rr1) + safe1, big ? w1 : w1 + safe1)); }
        const T berr = warp_max(qv);
        z0 = rr0; z1 = rr1;
        if (!(berr > eps && (T)2 * berr <= lstres && count < 5)) break;         // at most ITMAX = 5 corrections
        lstres = berr;
    }
    __syncwarp();
    if (v0) sm.sx[r0] = equil ? x0 * sc0 : x0;
    if (v1) sm.sx[r1] = equil ? x1 * sc1 : x1;
    __syncwarp();
    return 0;
}

// solveBoxQP for one QP by one warp.  P: n x n row-major in global memory (lower triangle read); sm.q / l / u hold the
// problem vectors; the solution is left in sm.x.  Returns mir_box_qp_status (uniform).
template <class T>
__device__ int boxqp_warp(const typename Num<T>::QPSettings& st, int n, const T* __restrict__ P, WarpQPSmem<T>& sm, int lane,
                          unsigned& iterations, unsigned& solves)
{
    iterations = 0; solves = 0;
    if (n == 0) return mir_qp_solved;                                          // boxcqp.d:162-163
    const int nh = (n + 1) >> 1;
    const int i0 = lane, i1 = n - 1 - lane;                                    // my variables
    const bool v0 = lane < nh, v1 = lane < (n >> 1);
    auto Pl = [&](int i, int j) -> T { return P[(size_t)i * n + j]; };         // i >= j
    auto Psym = [&](int i, int j) -> T { return (i >= j) ? Pl(i, j) : Pl(j, i); };

    if (v0) sm.b[i0] = -sm.q[i0];                                              // boxcqp.d:191
    if (v1) sm.b[i1] = -sm.q[i1];
    __syncwarp();
    ++solves;
    if (posvx_warp<T>(n, Pl, sm, lane) != 0) return mir_qp_numericError;   // boxcqp.d:194-213
    T x0 = v0 ? sm.sx[i0] : (T)0, x1 = v1 ? sm.sx[i1] : (T)0;
    const T l0 = v0 ? sm.l[i0] : (T)0, u0 = v0 ? sm.u[i0] : (T)0, l1 = v1 ? sm.l[i1] : (T)0, u1 = v1 ? sm.u[i1] : (T)0;
    const T q0 = v0 ? sm.q[i0] : (T)0, q1 = v1 ? sm.q[i1] : (T)0;
    {
        const bool out = (v0 && !(l0 <= x0 && x0 <= u0)) || (v1 && !(l1 <= x1 && x1 <= u1));      // boxcqp.d:216-219
        if (!__any_sync(WQP_FULL, out)) {
            if (v0) sm.x[i0] = x0;
            if (v1) sm.x[i1] = x1;
            __syncwarp();
            return mir_qp_solved;
        }
    }
    const unsigned maxIterations = st.maxIterations ? st.maxIterations : (unsigned)n * 10u + 100u;   // boxcqp.d:224-226
    T la0 = (T)0, mu0 = (T)0, la1 = (T)0, mu1 = (T)0;
    for (unsigned step = 0; step < maxIterations; ++step) {                    // boxcqp.d:234
        ++iterations;
        int f0 = 0, f1 = 0;                                                    // boxcqp.d:239-263
        auto classify = [&](T& x, T l, T u, T& la, T& mu) -> int {
            const T xl = x - l, ux = u - x;
            if (xl < (T)0 || (xl < st.relTolerance + st.absTolerance * t_abs(l) && la >= (T)0)) { x = l; mu = (T)0; return -1; }
            if (ux < (T)0 || (ux < st.relTolerance + st.absTolerance * t_abs(u) && mu >= (T)0)) { x = u; la = (T)0; return 1; }
            mu = (T)0; la = (T)0; return 0;
        };
        if (v0) f0 = classify(x0, l0, u0, la0, mu0);
        if (v1) f1 = classify(x1, l1, u1, la1, mu1);
        // ascending free list: variables 0 .. nh-1 sit in slot 0 of lanes 0 .. nh-1, variables n-1 .. nh in slot 1 of lanes 0 .. n/2-1
        const unsigned m0 = __ballot_sync(WQP_FULL, v0 && f0 == 0), m1 = __ballot_sync(WQP_FULL, v1 && f1 == 0);
        const int s = __popc(m0) + __popc(m1);
        __syncwarp();
        if (v0) { sm.flag[i0] = (signed char)f0; sm.x[i0] = x0; if (f0 == 0) sm.idx[__popc(m0 & ((1u << lane) - 1u))] = i0; }
        if (v1) { sm.flag[i1] = (signed char)f1; sm.x[i1] = x1; if (f1 == 0) sm.idx[__popc(m0) + __popc(m1 & ~((2u << lane) - 1u))] = i1; }
        __syncwarp();
        if (s == n) break;                                                     // boxcqp.d:265-266 -> maxIterations

        if (s > 0) {
            // reduced right-hand side, boxcqp.d:282-305: b_a = -KBN(q_i + sum over fixed j (ascending) of P(i,j) bound_j), i = idx[a]
            const int sh = (s + 1) >> 1;
            const int a0 = lane, a1 = s - 1 - lane;
            const bool w0 = lane < sh, w1 = lane < (s >> 1);
            const int c0 = w0 ? sm.idx[a0] : 0, c1 = w1 ? sm.idx[a1] : 0;
            KBN<T> s0(w0 ? sm.q[c0] : (T)0), s1(w1 ? sm.q[c1] : (T)0);
            for (int j = 0; j < n; ++j) {
                const int f = sm.flag[j];
                if (f) {                                                       // (uniform)
                    const T bound = f < 0 ? sm.l[j] : sm.u[j];
                    if (w0) s0.put(mul_rn(Psym(c0, j), bound));
                    if (w1) s1.put(mul_rn(Psym(c1, j), bound));
                }
            }
            if (w0) sm.b[a0] = -s0.sum();
            if (w1) sm.b[a1] = -s1.sum();
            __syncwarp();
            ++solves;
            const int* idx = sm.idx;
            auto Asub = [&](int a, int c) -> T { return Pl(idx[a], idx[c]); };   // idx ascending: a >= c => idx[a] >= idx[c]
            if (posvx_warp<T>(s, Asub, sm, lane) != 0) return mir_qp_numericError;   // boxcqp.d:310-324
            if (w0) sm.x[c0] = sm.sx[a0];                                      // boxcqp.d:327-329
            if (w1) sm.x[c1] = sm.sx[a1];
            __syncwarp();
            if (v0) x0 = sm.x[i0];
            if (v1) x1 = sm.x[i1];
        }

        // multipliers of the fixed variables, boxcqp.d:333-337: (P x + q)_i, lower part then upper part
        auto multiplier = [&](int i, T qi) -> T {
            T d1 = (T)0, d2 = (T)0;
            for (int j = 0; j < i; ++j) d1 = fma(Pl(i, j), sm.x[j], d1);
            for (int j = i; j < n; ++j) d2 = fma(Pl(j, i), sm.x[j], d2);
            return d1 + d2 + qi;
        };
        bool again = false;                                                    // boxcqp.d:339-347
        if (v0) {
            if (f0) { const T val = multiplier(i0, q0); if (f0 < 0) { la0 = val; again = !(la0 >= (T)0); } else { mu0 = -val; again = !(mu0 >= (T)0); } }
            else again = !(x0 >= l0 && x0 <= u0);
        }
        if (v1) {
            if (f1) { const T val = multiplier(i1, q1); if (f1 < 0) { la1 = val; again = again || !(la1 >= (T)0); } else { mu1 = -val; again = again || !(mu1 >= (T)0); } }
            else again = again || !(x1 >= l1 && x1 <= u1);
        }
        if (__any_sync(WQP_FULL, again)) continue;
        __syncwarp();
        if (v0) sm.x[i0] = t_max(t_min(x0, u0), l0);                           // applyBounds, boxcqp.d:349
        if (v1) sm.x[i1] = t_max(t_min(x1, u1), l1);
        __syncwarp();
        return mir_qp_solved;
    }
    return mir_qp_maxIterations;                                               // boxcqp.d:378
}

}  // namespace mirb200
