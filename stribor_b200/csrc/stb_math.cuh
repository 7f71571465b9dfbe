// Element-wise device math shared by every kernel: activations, the rational-quadratic
// spline (reference: stribor/util/rational_quadratic_spline.py) and the cubic spline
// (reference: stribor/util/cubic_spline.py).  Generic over the scalar type T (float or double);
// IEEE division and sqrt (the library is built WITHOUT --use_fast_math) and no approximate
// intrinsics, so results track the reference's ATen CPU kernels to a few ulp of T.
//
// Parameter access is abstracted by an indexable "P" object (p[i] -> T&): the generic
// kernel keeps one element's parameters in a shared-memory column, the tensor-core kernel
// in registers.
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <type_traits>
#include <utility>
#include "../../include/stribor_b200.h"

namespace stb {

// ---------------------------------------------------------------------------------------
// scalar type plumbing
// ---------------------------------------------------------------------------------------
// A non-integer literal in the scalar type T of the enclosing code: the float literal the fp32
// kernels have always folded in, or the double one.
#define STB_LIT(v) (std::is_same<T, float>::value ? T(v##f) : T(v))

// the float functions the fp32 kernels call, and their double counterparts
#define STB_MATH1(NAME, F32, F64)                                                   \
    __device__ __forceinline__ float NAME(float v) { return F32(v); }                \
    __device__ __forceinline__ double NAME(double v) { return F64(v); }
#define STB_MATH2(NAME, F32, F64)                                                   \
    __device__ __forceinline__ float NAME(float a, float b) { return F32(a, b); }    \
    __device__ __forceinline__ double NAME(double a, double b) { return F64(a, b); }
STB_MATH1(exp_, expf, exp)
STB_MATH1(expm1_, expm1f, expm1)
STB_MATH1(log_, logf, log)
STB_MATH1(log1p_, log1pf, log1p)
STB_MATH1(tanh_, tanhf, tanh)
STB_MATH1(erf_, erff, erf)
STB_MATH1(sqrt_, sqrtf, sqrt)
STB_MATH1(cos_, cosf, cos)
STB_MATH1(sin_, sinf, sin)
STB_MATH1(fabs_, fabsf, fabs)
STB_MATH2(atan2_, atan2f, atan2)
STB_MATH2(fmax_, fmaxf, fmax)
STB_MATH2(fmin_, fminf, fmin)
#undef STB_MATH1
#undef STB_MATH2

// element type of an indexable parameter object
template <class P>
using elem_t = std::remove_cv_t<std::remove_reference_t<decltype(std::declval<P>()[0])>>;

// ---------------------------------------------------------------------------------------
// activations (torch.nn defaults)
// ---------------------------------------------------------------------------------------
template <class T>
__device__ __forceinline__ T softplus_f(T v) {                   // F.softplus: beta 1, threshold 20
    return v > T(20) ? v : log1p_(exp_(v));
}
template <class T>
__device__ __forceinline__ T sigmoid_f(T v) { return T(1) / (T(1) + exp_(-v)); }

template <class T>
__device__ __forceinline__ T activate(int act, T v) {
    switch (act) {
        case STB_ACT_TANH: return tanh_(v);
        case STB_ACT_RELU: return v > T(0) ? v : T(0);
        case STB_ACT_SIGMOID: return sigmoid_f(v);
        case STB_ACT_ELU: return v > T(0) ? v : expm1_(v);
        case STB_ACT_SOFTPLUS: return softplus_f(v);
        case STB_ACT_LEAKY_RELU: return v > T(0) ? v : STB_LIT(0.01) * v;
        case STB_ACT_SILU: return v * sigmoid_f(v);
        case STB_ACT_GELU: return STB_LIT(0.5) * v * (T(1) + erf_(v * STB_LIT(0.70710678118654752440)));
        default: return v;
    }
}

// derivative of the activation given pre-activation v and post-activation a
template <class T>
__device__ __forceinline__ T activate_grad(int act, T v, T a) {
    switch (act) {
        case STB_ACT_TANH: return T(1) - a * a;
        case STB_ACT_RELU: return v > T(0) ? T(1) : T(0);
        case STB_ACT_SIGMOID: return a * (T(1) - a);
        case STB_ACT_ELU: return v > T(0) ? T(1) : a + T(1);
        case STB_ACT_SOFTPLUS: return sigmoid_f(v);
        case STB_ACT_LEAKY_RELU: return v > T(0) ? T(1) : STB_LIT(0.01);
        case STB_ACT_SILU: { T s = sigmoid_f(v); return s * (T(1) + v * (T(1) - s)); }
        case STB_ACT_GELU: {
            T cdf = STB_LIT(0.5) * (T(1) + erf_(v * STB_LIT(0.70710678118654752440)));
            T pdf = STB_LIT(0.39894228040143267794) * exp_(STB_LIT(-0.5) * v * v);
            return cdf + v * pdf;
        }
        default: return T(1);
    }
}

// view of a parameter object shifted by a fixed offset
template <class P>
struct OffsetView {
    P p;
    int o;
    __device__ __forceinline__ elem_t<P>& operator[](int i) const { return p[o + i]; }
};

// strided shared-memory column holding one element's parameters
template <class T>
struct SmemCol {
    T* base;
    int stride;
    __device__ __forceinline__ T& operator[](int i) const { return base[i * stride]; }
};

// ---------------------------------------------------------------------------------------
// softmax -> bin sizes, in place.   u[0..K) unnormalised  ->  u[i] = min + (1-min*K)*softmax_i
// rational_quadratic_spline.py:101-105, cubic_spline.py:104-105,111-112
// ---------------------------------------------------------------------------------------
template <class P>
__device__ __forceinline__ void softmax_bins(P u, int K, elem_t<P> min_size) {
    using T = elem_t<P>;
    T m = u[0];
    for (int i = 1; i < K; ++i) m = fmax_(m, u[i]);
    T s = T(0);
    for (int i = 0; i < K; ++i) {
        T e = exp_(u[i] - m);
        u[i] = e;
        s += e;
    }
    const T scale = T(1) - min_size * (T)K;
    for (int i = 0; i < K; ++i) u[i] = min_size + scale * (u[i] / s);
}

// ---------------------------------------------------------------------------------------
// spline constants
// ---------------------------------------------------------------------------------------
#define STB_RQS_MIN 1e-3f
// log(exp(1 - 1e-3) - 1): unconstrained value that makes the boundary derivative 1
// (rational_quadratic_spline.py:79-83)
#define STB_RQS_EDGE_CONST 0.5397424172369522f
#define STB_CUB_MIN 1e-2f
#define STB_CUB_EPS 1e-5f
#define STB_CUB_QUAD 1e-3f

// The spline functions take their constants as a template parameter O.  RqsDefaultsT / CubDefaultsT
// are the reference defaults above, folded in at compile time: the code the modules and the
// tensor-core kernels run.  In double they are the reference's Python float values (the edge pad
// log(exp(1 - 1e-3) - 1) evaluated in double), not the float constants widened.  SplineOptsT holds
// the functional API's own values (stb_spline_opts), read at run time by kernels instantiated for it.
template <class T>
struct RqsDefaultsT {
    static constexpr bool kRuntime = false;
    __device__ __forceinline__ T min_w() const { return STB_LIT(1e-3); }
    __device__ __forceinline__ T min_h() const { return STB_LIT(1e-3); }
    __device__ __forceinline__ T min_d() const { return STB_LIT(1e-3); }
    __device__ __forceinline__ T edge() const { return STB_LIT(0.5397424172369522); }
    __device__ __forceinline__ bool free_edge() const { return false; }
};

template <class T>
struct CubDefaultsT {
    static constexpr bool kRuntime = false;
    __device__ __forceinline__ T min_w() const { return STB_LIT(1e-2); }
    __device__ __forceinline__ T min_h() const { return STB_LIT(1e-2); }
    __device__ __forceinline__ T eps() const { return STB_LIT(1e-5); }
    __device__ __forceinline__ T quad() const { return STB_LIT(1e-3); }
};
using RqsDefaults = RqsDefaultsT<float>;
using CubDefaults = CubDefaultsT<float>;

template <class T>
struct SplineOptsT {
    static constexpr bool kRuntime = true;
    T mw, mh, md;
    T edge_;           // log(exp(1 - md) - 1), evaluated in double on the host (rounded once for float)
    T eps_, quad_;
    int free_edge_;
    __device__ __forceinline__ T min_w() const { return mw; }
    __device__ __forceinline__ T min_h() const { return mh; }
    __device__ __forceinline__ T min_d() const { return md; }
    __device__ __forceinline__ T edge() const { return edge_; }
    __device__ __forceinline__ bool free_edge() const { return free_edge_ != 0; }
    __device__ __forceinline__ T eps() const { return eps_; }
    __device__ __forceinline__ T quad() const { return quad_; }
};
// the fp32 kernels' parameter type
struct SplineOpts : SplineOptsT<float> {};

// the reference defaults of a transform kind
template <int KIND, class T = float>
using DefaultOpts = typename std::conditional<KIND == STB_CUBIC, CubDefaultsT<T>, RqsDefaultsT<T>>::type;

// The options of stb_spline_opts are float in both dtypes: a double kernel computes with the
// float values widened.
template <class Opts>
inline Opts make_spline_opts(const stb_spline_opts& s) {
    using T = decltype(Opts::mw);
    Opts o;
    o.mw = s.min_bin_width;
    o.mh = s.min_bin_height;
    o.md = s.min_derivative;
    o.edge_ = (T)log(exp(1.0 - (double)s.min_derivative) - 1.0);
    o.eps_ = s.cub_eps;
    o.quad_ = s.cub_quad_threshold;
    o.free_edge_ = s.free_edge_derivs;
    return o;
}

// ---------------------------------------------------------------------------------------
// rational-quadratic spline
// ---------------------------------------------------------------------------------------

// bin sizes u[0..K) -> knots: u[i] := knot_{i+1}, with knot_0 = lo and knot_K forced to hi.
// rational_quadratic_spline.py:180-184 / :187-191
template <class P, class T = elem_t<P>>
__device__ __forceinline__ void sizes_to_knots(P u, int K, T lo, T hi) {
    T cum = T(0);
    const T span = hi - lo;
    for (int i = 0; i < K; ++i) {
        cum += u[i];
        u[i] = span * cum + lo;
    }
    u[K - 1] = hi;
}

template <class P, class T = elem_t<P>>
__device__ __forceinline__ T knot_at(P kn, int i, T lo) { return i == 0 ? lo : kn[i - 1]; }

// search_sorted.py:3-5: sum(x >= knots) - 1 with the last knot nudged up by 1e-6.
template <class P, class T = elem_t<P>>
__device__ __forceinline__ int knot_search(P kn, int K, T lo, T x) {
    int cnt = (x >= lo) ? 1 : 0;
    for (int i = 0; i < K - 1; ++i) cnt += (x >= kn[i]) ? 1 : 0;
    cnt += (x >= kn[K - 1] + STB_LIT(1e-6)) ? 1 : 0;
    int k = cnt - 1;
    return k < 0 ? 0 : (k > K - 1 ? K - 1 : k);
}

template <class T>
struct RqsBinT {
    T xk, wk, yk, hk, delta, d0, d1;
};
using RqsBin = RqsBinT<float>;

// W, H: knot columns (after sizes_to_knots); D: K-1 unconstrained interior derivatives
// (K+1, the boundaries included, with o.free_edge()).
template <class PW, class PH, class PD, class T = elem_t<PW>, class O = RqsDefaultsT<T>>
__device__ __forceinline__ RqsBinT<T> rqs_bin(PW W, PH H, PD D, int K, int k, T left, T bottom,
                                              const O& o = O()) {
    RqsBinT<T> b;
    b.xk = knot_at(W, k, left);
    b.wk = W[k] - b.xk;                                   // widths re-derived from knots (:185)
    b.yk = knot_at(H, k, bottom);
    b.hk = H[k] - b.yk;
    b.delta = b.hk / b.wk;
    T u0, u1;
    if (o.free_edge()) {
        u0 = D[k];
        u1 = D[k + 1];
    } else {
        u0 = (k == 0) ? o.edge() : D[k - 1];
        u1 = (k == K - 1) ? o.edge() : D[k];
    }
    b.d0 = o.min_d() + softplus_f(u0);                    // :107
    b.d1 = o.min_d() + softplus_f(u1);
    return b;
}

// forward map and log-derivative inside bin b    (rational_quadratic_spline.py:236-248)
template <class T>
__device__ __forceinline__ void rqs_forward_in_bin(const RqsBinT<T>& b, T x, T& y, T& ld) {
    T theta = (x - b.xk) / b.wk;
    T tt = theta * (T(1) - theta);
    T num = b.hk * (b.delta * theta * theta + b.d0 * tt);
    T den = b.delta + (b.d0 + b.d1 - T(2) * b.delta) * tt;
    y = b.yk + num / den;
    T omt = T(1) - theta;
    T dnum = b.delta * b.delta * (b.d1 * theta * theta + T(2) * b.delta * tt + b.d0 * omt * omt);
    ld = log_(dnum) - T(2) * log_(den);
}

// inverse map and ITS log-derivative inside bin b  (rational_quadratic_spline.py:212-234)
template <class T>
__device__ __forceinline__ void rqs_inverse_in_bin(const RqsBinT<T>& b, T y, T& x, T& ld) {
    T dy = y - b.yk;
    T s = b.d0 + b.d1 - T(2) * b.delta;
    T qa = dy * s + b.hk * (b.delta - b.d0);
    T qb = b.hk * b.d0 - dy * s;
    T qc = -b.delta * dy;
    T disc = qb * qb - T(4) * qa * qc;
    T root = (T(2) * qc) / (-qb - sqrt_(disc));
    x = root * b.wk + b.xk;
    T tt = root * (T(1) - root);
    T den = b.delta + s * tt;
    T omr = T(1) - root;
    T num = b.delta * b.delta * (b.d1 * root * root + T(2) * b.delta * tt + b.d0 * omr * omr);
    ld = -log_(num) + T(2) * log_(den);
}

// Full element evaluation.  prm = [uw(K) | uh(K) | ud(K-1 or K+1)] (destroyed).
// Domain [left, right] -> codomain [bottom, top]  (rational_quadratic_spline.py:55-64).
//   inverse == false: out = f(x),      ld = log f'(x)
//   inverse == true : out = f^-1(x),   ld = own_ld ? log (f^-1)'(x) : -log f'(out)
// Identity (ld 0) outside the active box  (rational_quadratic_spline.py:71,86-87).
// (The scalar arguments take the element type of P: float box bounds convert.)
template <class P, class O = RqsDefaultsT<elem_t<P>>>
__device__ __forceinline__ void rqs_element(P prm, int K, elem_t<P> left, elem_t<P> right, elem_t<P> bottom,
                                            elem_t<P> top, bool inverse, bool own_ld, elem_t<P> x,
                                            elem_t<P>& out, elem_t<P>& ld, int* kbin = nullptr,
                                            const O& o = O()) {
    using T = elem_t<P>;
    out = x;
    ld = T(0);
    if (kbin) *kbin = -1;                     // identity tail: no search happens (:86-91)
    const T lo = inverse ? bottom : left, hi = inverse ? top : right;
    if (!(x >= lo && x <= hi)) return;
    OffsetView<P> W{prm, 0}, H{prm, K}, D{prm, 2 * K};
    softmax_bins(W, K, o.min_w());
    softmax_bins(H, K, o.min_h());
    sizes_to_knots(W, K, left, right);
    sizes_to_knots(H, K, bottom, top);
    if (!inverse) {
        int k = knot_search(W, K, left, x);
        if (kbin) *kbin = k;
        RqsBinT<T> b = rqs_bin(W, H, D, K, k, left, bottom, o);
        rqs_forward_in_bin(b, x, out, ld);
    } else {
        int k = knot_search(H, K, bottom, x);
        if (kbin) *kbin = k;
        RqsBinT<T> b = rqs_bin(W, H, D, K, k, left, bottom, o);
        T ld_own;
        rqs_inverse_in_bin(b, x, out, ld_own);
        if (own_ld) {
            ld = ld_own;
        } else {
            // flow.py:42-47 + coupling.py:84-95: forward log-derivative re-evaluated at the
            // recovered point (its own inside test and bin search), negated.
            ld = T(0);
            if (out >= left && out <= right) {
                int k2 = knot_search(W, K, left, out);
                RqsBinT<T> b2 = (k2 == k) ? b : rqs_bin(W, H, D, K, k2, left, bottom, o);
                T y2, ldf;
                rqs_forward_in_bin(b2, out, y2, ldf);
                ld = -ldf;
            }
        }
    }
}

// ---------------------------------------------------------------------------------------
// cubic spline
// ---------------------------------------------------------------------------------------
template <class T>
__device__ __forceinline__ T sign_f(T v) { return (v > T(0)) ? T(1) : ((v < T(0)) ? T(-1) : T(0)); }
// cubic_spline.py:18-20: sign(v) * |v|^(1/3), written as the reference writes it
template <class T>
__device__ __forceinline__ T cbrt_ref(T v) { return sign_f(v) * exp_(log_(fabs_(v)) / T(3)); }

template <class T>
struct CubBinT {
    T a, b, c, d, xl, xr;
};
using CubBin = CubBinT<float>;

// W, H: bin sizes (after softmax_bins); k: bin; cw/ch: cumulative sums BEFORE bin k.
// cubic_spline.py:118-138
template <class PW, class PH, class T = elem_t<PW>>
__device__ __forceinline__ CubBinT<T> cubic_bin(PW W, PH H, int K, int k, T cw, T ch, T ul, T ur) {
    T wk = W[k], hk = H[k];
    T sk = hk / wk;
    T dl, dr;
    if (k == 0) {
        dl = sigmoid_f(ul) * T(3) * sk;
    } else {
        T wp = W[k - 1], sp = H[k - 1] / wp;
        T m1 = fmin_(fabs_(sp), fabs_(sk));
        T m2 = STB_LIT(0.5) * (wk * sp + wp * sk) / (wp + wk);
        dl = fmin_(m1, m2) * (sign_f(sp) + sign_f(sk));
    }
    if (k == K - 1) {
        dr = sigmoid_f(ur) * T(3) * sk;
    } else {
        T wn = W[k + 1], sn = H[k + 1] / wn;
        T m1 = fmin_(fabs_(sk), fabs_(sn));
        T m2 = STB_LIT(0.5) * (wn * sk + wk * sn) / (wk + wn);
        dr = fmin_(m1, m2) * (sign_f(sk) + sign_f(sn));
    }
    CubBinT<T> r;
    r.a = (dl + dr - T(2) * sk) / (wk * wk);
    r.b = (T(3) * sk - T(2) * dl - dr) / wk;
    r.c = dl;
    r.d = ch;
    r.xl = cw;
    r.xr = (k == K - 1) ? T(1) : cw + wk;           // cumwidths[..., -1] = 1 (:108)
    return r;
}

// Walk the knots of `S` (the searched sizes) accumulating both cumulative sums; returns the bin
// of u and the cumulative widths/heights before it.   search_sorted.py:3-5 on cubic_spline.py:107-116
template <class PW, class PH, class T = elem_t<PW>>
__device__ __forceinline__ int cubic_search(PW W, PH H, int K, bool search_heights, T u, T& cw, T& ch) {
    T aw = T(0), ah = T(0);
    int k = 0;
    cw = T(0);
    ch = T(0);
    for (int i = 1; i < K; ++i) {
        aw += W[i - 1];
        ah += H[i - 1];
        T knot = search_heights ? ah : aw;
        if (u >= knot) { k = i; cw = aw; ch = ah; }
    }
    // the last knot is 1 + 1e-6: an inside u (<= 1) never reaches it
    return k;
}

template <class T>
__device__ __forceinline__ T cubic_forward_in_bin(const CubBinT<T>& b, T u, T& ld) {
    T s = u - b.xl;
    T out = b.a * s * s * s + b.b * s * s + b.c * s + b.d;
    ld = log_(T(3) * b.a * s * s + T(2) * b.b * s + b.c);
    return out;
}

// cubic_spline.py:153-228
template <class T, class O = CubDefaultsT<T>>
__device__ __forceinline__ T cubic_inverse_in_bin(const CubBinT<T>& k, T u, T& ld, const O& o = O()) {
    T b_ = (k.b / k.a) / T(3);
    T c_ = (k.c / k.a) / T(3);
    T d_ = (k.d - u) / k.a;
    T delta_1 = -b_ * b_ + c_;
    T delta_2 = -c_ * b_ + d_;
    T delta_3 = b_ * d_ - c_ * c_;
    T disc = T(4) * delta_1 * delta_3 - delta_2 * delta_2;
    T dep_1 = T(-2) * b_ * delta_1 + delta_2;
    T dep_2 = delta_1;
    T out;
    if (disc > T(0)) {
        T theta = atan2_(sqrt_(disc), -dep_1) / T(3);
        T c1 = cos_(theta), c2 = sin_(theta);
        T scale = T(2) * sqrt_(-dep_2);
        T shift = -b_ + k.xl;
        T r1 = c1 * scale + shift;
        T r2 = (STB_LIT(-0.5) * c1 - STB_LIT(0.5) * STB_LIT(1.7320508075688772) * c2) * scale + shift;
        T r3 = (STB_LIT(-0.5) * c1 + STB_LIT(0.5) * STB_LIT(1.7320508075688772) * c2) * scale + shift;
        T lo = k.xl - o.eps(), hi = k.xr + o.eps();
        bool ok1 = (lo < r1) && (r1 < hi), ok2 = (lo < r2) && (r2 < hi), ok3 = (lo < r3) && (r3 < hi);
        out = ok1 ? r1 : (ok2 ? r2 : (ok3 ? r3 : r1));      // argsort(masks, desc)[..., 0]  (:212)
    } else {
        T sq = sqrt_(-disc);
        T p = cbrt_ref((-dep_1 + sq) / T(2));
        T q = cbrt_ref((-dep_1 - sq) / T(2));
        out = (p + q) - b_ + k.xl;
    }
    if (fabs_(k.a) < o.quad()) {                             // :217-223
        T qc = k.d - u;
        T alpha = (-k.c + sqrt_(k.c * k.c - T(4) * k.b * qc)) / (T(2) * k.b);
        out = alpha + k.xl;
    }
    T s = out - k.xl;
    ld = -log_(T(3) * k.a * s * s + T(2) * k.b * s + k.c);
    return out;
}

// prm = [uw(K) | uh(K) | left, right]  (destroyed).  Same contract as rqs_element.
template <class P, class O = CubDefaultsT<elem_t<P>>>
__device__ __forceinline__ void cubic_element(P prm, int K, elem_t<P> lower, elem_t<P> upper, bool inverse,
                                              bool own_ld, elem_t<P> x, elem_t<P>& out, elem_t<P>& ld,
                                              int* kbin = nullptr, const O& o = O()) {
    using T = elem_t<P>;
    out = x;
    ld = T(0);
    if (kbin) *kbin = -1;
    if (!(x >= lower && x <= upper)) return;
    OffsetView<P> W{prm, 0}, H{prm, K};
    const T ul = prm[2 * K], ur = prm[2 * K + 1];
    softmax_bins(W, K, o.min_w());
    softmax_bins(H, K, o.min_h());
    const T span = upper - lower;
    T u = (x - lower) / span;                                // :99-102
    T cw, ch;
    if (!inverse) {
        int k = cubic_search(W, H, K, false, u, cw, ch);
        if (kbin) *kbin = k;
        CubBinT<T> b = cubic_bin(W, H, K, k, cw, ch, ul, ur);
        T v = cubic_forward_in_bin(b, u, ld);
        out = v * span + lower;                              // :244-245 (log terms cancel: same box)
    } else {
        int k = cubic_search(W, H, K, true, u, cw, ch);
        if (kbin) *kbin = k;
        CubBinT<T> b = cubic_bin(W, H, K, k, cw, ch, ul, ur);
        T ld_own;
        T v = cubic_inverse_in_bin(b, u, ld_own, o);
        out = v * span + lower;
        if (own_ld) {
            ld = ld_own;
        } else {
            ld = T(0);
            if (out >= lower && out <= upper) {
                T u2 = (out - lower) / span;
                int k2 = cubic_search(W, H, K, false, u2, cw, ch);
                CubBinT<T> b2 = (k2 == k) ? b : cubic_bin(W, H, K, k2, cw, ch, ul, ur);
                T ldf;
                (void)cubic_forward_in_bin(b2, u2, ldf);
                ld = -ldf;
            }
        }
    }
}

}  // namespace stb
