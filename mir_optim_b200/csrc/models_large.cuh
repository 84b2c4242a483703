// models_large.cuh -- runtime-n device residual functors for the single-large-problem path
// (one problem, rows spread over the whole GPU / several GPUs; BASELINE configs[0] and configs[3]).
//
// Same role as models.cuh (the GPU counterparts of LeastSquaresFunction / LeastSquaresJacobian,
// least_squares.d:73-80), same explicitly rounded operation sequences -- a row evaluated here
// returns the same bits as the batched functor and as the oracle's host callback
// (oracle/models_oracle.cpp).  Differences: n is a run-time value (GAUSSMIX has n = 3K+2 up to
// 128) and parameters are read through a ParamView, which lets the finite-difference Jacobian
// (least_squares.d:1018-1049) override one parameter without copying the vector.
//
// Per-parameter auxiliaries (reciprocals of widths) are computed once per kernel by
// `aux_of` -- the same correctly rounded division the oracle performs per row.
//
// jac_items(n) / jac_item(...) split one Jacobian row into independent column groups so a CTA
// can spread a 32-row tile over all its threads.
#pragma once
#include "common.cuh"
#include "repro_math.cuh"

namespace mirb200 {

template <class T> struct ParamView {
    const T* p;      // parameters (shared memory)
    const T* aux;    // per-parameter auxiliaries (shared memory)
    int j;           // overridden index, -1 for none
    T vj, auxj;
    __device__ __forceinline__ T operator()(int k) const { return k == j ? vj : p[k]; }
    __device__ __forceinline__ T a(int k) const { return k == j ? auxj : aux[k]; }
};

// r_i = sum_k p[3k] exp(-(t_i - p[3k+1])^2 / (2 p[3k+2]^2)) + p[n-2] + p[n-1] t_i - y_i     BASELINE configs[3]
template <class T> struct LModelGaussMix {
    __host__ __device__ static bool valid_n(int n) { return n >= 2 && (n - 2) % 3 == 0; }
    __device__ static T aux_of(int k, int n, T v) { return (k < n - 2 && k % 3 == 2) ? rcp_ni(v) : (T)0; }
    __device__ static T residual(const ParamView<T>& p, int n, T t, T y) {
        T acc = add_rn(p(n - 2), mul_rn(p(n - 1), t));
        for (int k = 0; k + 3 <= n - 2; k += 3) {
            const T z = mul_rn(sub_rn(t, p(k + 1)), p.a(k + 2));
            acc = add_rn(acc, mul_rn(p(k), exp_repro_tp(mul_rn((T)-0.5, mul_rn(z, z)))));
        }
        return sub_rn(acc, y);
    }
    __host__ __device__ static int jac_items(int n) { return (n - 2) / 3 + 1; }
    __device__ static void jac_item(const ParamView<T>& p, int n, int item, T t, T* row) {
        const int k = 3 * item;
        if (k + 3 <= n - 2) {
            const T is = p.a(k + 2);
            const T z = mul_rn(sub_rn(t, p(k + 1)), is);
            const T zz = mul_rn(z, z);
            const T e = exp_repro_tp(mul_rn((T)-0.5, zz));
            const T ae = mul_rn(p(k), e);
            row[k] = e; row[k + 1] = mul_rn(mul_rn(ae, z), is); row[k + 2] = mul_rn(mul_rn(ae, zz), is);
        } else {
            row[n - 2] = (T)1; row[n - 1] = t;
        }
    }
};

// r_i = sum_k p[2k] exp(-p[2k+1] t_i) - y_i                                                 BASELINE configs[2]
template <class T> struct LModelSumExp {
    __host__ __device__ static bool valid_n(int n) { return n >= 2 && n % 2 == 0; }
    __device__ static T aux_of(int, int, T) { return (T)0; }
    __device__ static T residual(const ParamView<T>& p, int n, T t, T y) {
        T acc = (T)0;
        for (int k = 0; k + 1 < n; k += 2) acc = add_rn(acc, mul_rn(p(k), exp_repro_tp(mul_rn(-p(k + 1), t))));
        return sub_rn(acc, y);
    }
    __host__ __device__ static int jac_items(int n) { return n / 2; }
    __device__ static void jac_item(const ParamView<T>& p, int, int item, T t, T* row) {
        const int k = 2 * item;
        const T e = exp_repro_tp(mul_rn(-p(k + 1), t));
        row[k] = e; row[k + 1] = mul_rn(-mul_rn(p(k), t), e);
    }
};

// r_i = p0 exp(-p1 t_i) + p2 - y_i                                                          BASELINE configs[0]
template <class T> struct LModelExpDecay3 {
    __host__ __device__ static bool valid_n(int n) { return n == 3; }
    __device__ static T aux_of(int, int, T) { return (T)0; }
    __device__ static T residual(const ParamView<T>& p, int, T t, T y) {
        return sub_rn(add_rn(mul_rn(p(0), exp_repro_tp(mul_rn(-p(1), t))), p(2)), y);
    }
    __host__ __device__ static int jac_items(int) { return 1; }
    __device__ static void jac_item(const ParamView<T>& p, int, int, T t, T* row) {
        const T e = exp_repro_tp(mul_rn(-p(1), t));
        row[0] = e; row[1] = mul_rn(-mul_rn(p(0), t), e); row[2] = (T)1;
    }
};

// r_i = p0 exp(-t_i p1) - y_i                                                               least_squares.d:347, 360
template <class T> struct LModelExpDecay2 {
    __host__ __device__ static bool valid_n(int n) { return n == 2; }
    __device__ static T aux_of(int, int, T) { return (T)0; }
    __device__ static T residual(const ParamView<T>& p, int, T t, T y) { return sub_rn(mul_rn(p(0), exp_repro_tp(mul_rn(-t, p(1)))), y); }
    __host__ __device__ static int jac_items(int) { return 1; }
    __device__ static void jac_item(const ParamView<T>& p, int, int, T t, T* row) {
        const T e = exp_repro_tp(mul_rn(-t, p(1)));
        row[0] = e; row[1] = mul_rn(-mul_rn(p(0), t), e);
    }
};

// r_i = p0 exp(-t_i / p1) + p2 - y_i                                                        least_squares.d:378, 390
template <class T> struct LModelExpTau3 {
    __host__ __device__ static bool valid_n(int n) { return n == 3; }
    __device__ static T aux_of(int, int, T) { return (T)0; }
    __device__ static T residual(const ParamView<T>& p, int, T t, T y) {
        return sub_rn(add_rn(mul_rn(p(0), exp_repro_tp(div_ni(-t, p(1)))), p(2)), y);
    }
    __host__ __device__ static int jac_items(int) { return 1; }
    __device__ static void jac_item(const ParamView<T>& p, int, int, T t, T* row) {
        const T e = exp_repro_tp(div_ni(-t, p(1)));
        row[0] = e; row[1] = div_ni(mul_rn(mul_rn(p(0), e), t), mul_rn(p(1), p(1))); row[2] = (T)1;
    }
};

// r_i = A exp(-(t_i - mu)^2 / (2 sigma^2)) + c - y_i                                        BASELINE configs[1]
template <class T> struct LModelGauss4 {
    __host__ __device__ static bool valid_n(int n) { return n == 4; }
    __device__ static T aux_of(int k, int, T v) { return k == 2 ? rcp_ni(v) : (T)0; }
    __device__ static T residual(const ParamView<T>& p, int, T t, T y) {
        const T z = mul_rn(sub_rn(t, p(1)), p.a(2));
        return sub_rn(add_rn(mul_rn(p(0), exp_repro_tp(mul_rn((T)-0.5, mul_rn(z, z)))), p(3)), y);
    }
    __host__ __device__ static int jac_items(int) { return 1; }
    __device__ static void jac_item(const ParamView<T>& p, int, int, T t, T* row) {
        const T is = p.a(2);
        const T z = mul_rn(sub_rn(t, p(1)), is);
        const T zz = mul_rn(z, z);
        const T e = exp_repro_tp(mul_rn((T)-0.5, zz));
        const T ae = mul_rn(p(0), e);
        row[0] = e; row[1] = mul_rn(mul_rn(ae, z), is); row[2] = mul_rn(mul_rn(ae, zz), is); row[3] = (T)1;
    }
};

#ifndef __CUDACC_RTC__
template <class M> struct ModelTag { using type = M; };

// The functor of a model id: f(ModelTag<L>{}) for the ids above, otherwise() for every other id.
template <class T, class F, class G> auto visit_large_model(unsigned id, F&& f, G&& otherwise)
{
    switch (id) {
    case MIR_MODEL_EXPDECAY2: return f(ModelTag<LModelExpDecay2<T>>{});
    case MIR_MODEL_EXPTAU3:   return f(ModelTag<LModelExpTau3<T>>{});
    case MIR_MODEL_EXPDECAY3: return f(ModelTag<LModelExpDecay3<T>>{});
    case MIR_MODEL_GAUSS4:    return f(ModelTag<LModelGauss4<T>>{});
    case MIR_MODEL_SUMEXP:    return f(ModelTag<LModelSumExp<T>>{});
    case MIR_MODEL_GAUSSMIX:  return f(ModelTag<LModelGaussMix<T>>{});
    default:                  return otherwise();
    }
}
#endif

}  // namespace mirb200
