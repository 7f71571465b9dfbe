// Element-wise device math shared by every kernel: activations, the rational-quadratic
// spline (reference: stribor/util/rational_quadratic_spline.py) and the cubic spline
// (reference: stribor/util/cubic_spline.py).  Plain fp32, IEEE division and sqrt (the
// library is built WITHOUT --use_fast_math) so results track the reference's ATen CPU
// kernels to a few ulp.
//
// Parameter access is abstracted by an indexable "P" object (p[i] -> float&): the generic
// kernel keeps one element's parameters in a shared-memory column, the tensor-core kernel
// in registers.
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <type_traits>
#include "../../include/stribor_b200.h"

namespace stb {

// ---------------------------------------------------------------------------------------
// activations (torch.nn defaults)
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ float softplus_f(float v) {           // F.softplus: beta 1, threshold 20
    return v > 20.f ? v : log1pf(expf(v));
}
__device__ __forceinline__ float sigmoid_f(float v) { return 1.f / (1.f + expf(-v)); }

__device__ __forceinline__ float activate(int act, float v) {
    switch (act) {
        case STB_ACT_TANH: return tanhf(v);
        case STB_ACT_RELU: return v > 0.f ? v : 0.f;
        case STB_ACT_SIGMOID: return sigmoid_f(v);
        case STB_ACT_ELU: return v > 0.f ? v : expm1f(v);
        case STB_ACT_SOFTPLUS: return softplus_f(v);
        case STB_ACT_LEAKY_RELU: return v > 0.f ? v : 0.01f * v;
        case STB_ACT_SILU: return v * sigmoid_f(v);
        case STB_ACT_GELU: return 0.5f * v * (1.f + erff(v * 0.70710678118654752440f));
        default: return v;
    }
}

// derivative of the activation given pre-activation v and post-activation a
__device__ __forceinline__ float activate_grad(int act, float v, float a) {
    switch (act) {
        case STB_ACT_TANH: return 1.f - a * a;
        case STB_ACT_RELU: return v > 0.f ? 1.f : 0.f;
        case STB_ACT_SIGMOID: return a * (1.f - a);
        case STB_ACT_ELU: return v > 0.f ? 1.f : a + 1.f;
        case STB_ACT_SOFTPLUS: return sigmoid_f(v);
        case STB_ACT_LEAKY_RELU: return v > 0.f ? 1.f : 0.01f;
        case STB_ACT_SILU: { float s = sigmoid_f(v); return s * (1.f + v * (1.f - s)); }
        case STB_ACT_GELU: {
            float cdf = 0.5f * (1.f + erff(v * 0.70710678118654752440f));
            float pdf = 0.39894228040143267794f * expf(-0.5f * v * v);
            return cdf + v * pdf;
        }
        default: return 1.f;
    }
}

// view of a parameter object shifted by a fixed offset
template <class P>
struct OffsetView {
    P p;
    int o;
    __device__ __forceinline__ float& operator[](int i) const { return p[o + i]; }
};

// strided shared-memory column holding one element's parameters
struct SmemCol {
    float* base;
    int stride;
    __device__ __forceinline__ float& operator[](int i) const { return base[i * stride]; }
};

// ---------------------------------------------------------------------------------------
// softmax -> bin sizes, in place.   u[0..K) unnormalised  ->  u[i] = min + (1-min*K)*softmax_i
// rational_quadratic_spline.py:101-105, cubic_spline.py:104-105,111-112
// ---------------------------------------------------------------------------------------
template <class P>
__device__ __forceinline__ void softmax_bins(P u, int K, float min_size) {
    float m = u[0];
    for (int i = 1; i < K; ++i) m = fmaxf(m, u[i]);
    float s = 0.f;
    for (int i = 0; i < K; ++i) {
        float e = expf(u[i] - m);
        u[i] = e;
        s += e;
    }
    const float scale = 1.f - min_size * (float)K;
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

// The spline functions take their constants as a template parameter O.  RqsDefaults / CubDefaults
// are the reference defaults above, folded in at compile time: the code the modules and the
// tensor-core kernels run.  SplineOpts holds the functional API's own values (stb_spline_opts),
// read at run time by kernels instantiated for it.
struct RqsDefaults {
    static constexpr bool kRuntime = false;
    __device__ __forceinline__ float min_w() const { return STB_RQS_MIN; }
    __device__ __forceinline__ float min_h() const { return STB_RQS_MIN; }
    __device__ __forceinline__ float min_d() const { return STB_RQS_MIN; }
    __device__ __forceinline__ float edge() const { return STB_RQS_EDGE_CONST; }
    __device__ __forceinline__ bool free_edge() const { return false; }
};

struct CubDefaults {
    static constexpr bool kRuntime = false;
    __device__ __forceinline__ float min_w() const { return STB_CUB_MIN; }
    __device__ __forceinline__ float min_h() const { return STB_CUB_MIN; }
    __device__ __forceinline__ float eps() const { return STB_CUB_EPS; }
    __device__ __forceinline__ float quad() const { return STB_CUB_QUAD; }
};

struct SplineOpts {
    static constexpr bool kRuntime = true;
    float mw, mh, md;
    float edge_;       // log(exp(1 - md) - 1), evaluated in double on the host and rounded once
    float eps_, quad_;
    int free_edge_;
    __device__ __forceinline__ float min_w() const { return mw; }
    __device__ __forceinline__ float min_h() const { return mh; }
    __device__ __forceinline__ float min_d() const { return md; }
    __device__ __forceinline__ float edge() const { return edge_; }
    __device__ __forceinline__ bool free_edge() const { return free_edge_ != 0; }
    __device__ __forceinline__ float eps() const { return eps_; }
    __device__ __forceinline__ float quad() const { return quad_; }
};

// the reference defaults of a transform kind
template <int KIND>
using DefaultOpts = typename std::conditional<KIND == STB_CUBIC, CubDefaults, RqsDefaults>::type;

inline SplineOpts make_spline_opts(const stb_spline_opts& s) {
    SplineOpts o;
    o.mw = s.min_bin_width;
    o.mh = s.min_bin_height;
    o.md = s.min_derivative;
    o.edge_ = (float)log(exp(1.0 - (double)s.min_derivative) - 1.0);
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
template <class P>
__device__ __forceinline__ void sizes_to_knots(P u, int K, float lo, float hi) {
    float cum = 0.f;
    const float span = hi - lo;
    for (int i = 0; i < K; ++i) {
        cum += u[i];
        u[i] = span * cum + lo;
    }
    u[K - 1] = hi;
}

template <class P>
__device__ __forceinline__ float knot_at(P kn, int i, float lo) { return i == 0 ? lo : kn[i - 1]; }

// search_sorted.py:3-5: sum(x >= knots) - 1 with the last knot nudged up by 1e-6.
template <class P>
__device__ __forceinline__ int knot_search(P kn, int K, float lo, float x) {
    int cnt = (x >= lo) ? 1 : 0;
    for (int i = 0; i < K - 1; ++i) cnt += (x >= kn[i]) ? 1 : 0;
    cnt += (x >= kn[K - 1] + 1e-6f) ? 1 : 0;
    int k = cnt - 1;
    return k < 0 ? 0 : (k > K - 1 ? K - 1 : k);
}

struct RqsBin {
    float xk, wk, yk, hk, delta, d0, d1;
};

// W, H: knot columns (after sizes_to_knots); D: K-1 unconstrained interior derivatives
// (K+1, the boundaries included, with o.free_edge()).
template <class PW, class PH, class PD, class O = RqsDefaults>
__device__ __forceinline__ RqsBin rqs_bin(PW W, PH H, PD D, int K, int k, float left, float bottom,
                                          const O& o = O()) {
    RqsBin b;
    b.xk = knot_at(W, k, left);
    b.wk = W[k] - b.xk;                                   // widths re-derived from knots (:185)
    b.yk = knot_at(H, k, bottom);
    b.hk = H[k] - b.yk;
    b.delta = b.hk / b.wk;
    float u0, u1;
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
__device__ __forceinline__ void rqs_forward_in_bin(const RqsBin& b, float x, float& y, float& ld) {
    float theta = (x - b.xk) / b.wk;
    float tt = theta * (1.f - theta);
    float num = b.hk * (b.delta * theta * theta + b.d0 * tt);
    float den = b.delta + (b.d0 + b.d1 - 2.f * b.delta) * tt;
    y = b.yk + num / den;
    float omt = 1.f - theta;
    float dnum = b.delta * b.delta * (b.d1 * theta * theta + 2.f * b.delta * tt + b.d0 * omt * omt);
    ld = logf(dnum) - 2.f * logf(den);
}

// inverse map and ITS log-derivative inside bin b  (rational_quadratic_spline.py:212-234)
__device__ __forceinline__ void rqs_inverse_in_bin(const RqsBin& b, float y, float& x, float& ld) {
    float dy = y - b.yk;
    float s = b.d0 + b.d1 - 2.f * b.delta;
    float qa = dy * s + b.hk * (b.delta - b.d0);
    float qb = b.hk * b.d0 - dy * s;
    float qc = -b.delta * dy;
    float disc = qb * qb - 4.f * qa * qc;
    float root = (2.f * qc) / (-qb - sqrtf(disc));
    x = root * b.wk + b.xk;
    float tt = root * (1.f - root);
    float den = b.delta + s * tt;
    float omr = 1.f - root;
    float num = b.delta * b.delta * (b.d1 * root * root + 2.f * b.delta * tt + b.d0 * omr * omr);
    ld = -logf(num) + 2.f * logf(den);
}

// Full element evaluation.  prm = [uw(K) | uh(K) | ud(K-1 or K+1)] (destroyed).
// Domain [left, right] -> codomain [bottom, top]  (rational_quadratic_spline.py:55-64).
//   inverse == false: out = f(x),      ld = log f'(x)
//   inverse == true : out = f^-1(x),   ld = own_ld ? log (f^-1)'(x) : -log f'(out)
// Identity (ld 0) outside the active box  (rational_quadratic_spline.py:71,86-87).
template <class P, class O = RqsDefaults>
__device__ __forceinline__ void rqs_element(P prm, int K, float left, float right, float bottom,
                                            float top, bool inverse, bool own_ld, float x,
                                            float& out, float& ld, int* kbin = nullptr,
                                            const O& o = O()) {
    out = x;
    ld = 0.f;
    if (kbin) *kbin = -1;                     // identity tail: no search happens (:86-91)
    const float lo = inverse ? bottom : left, hi = inverse ? top : right;
    if (!(x >= lo && x <= hi)) return;
    OffsetView<P> W{prm, 0}, H{prm, K}, D{prm, 2 * K};
    softmax_bins(W, K, o.min_w());
    softmax_bins(H, K, o.min_h());
    sizes_to_knots(W, K, left, right);
    sizes_to_knots(H, K, bottom, top);
    if (!inverse) {
        int k = knot_search(W, K, left, x);
        if (kbin) *kbin = k;
        RqsBin b = rqs_bin(W, H, D, K, k, left, bottom, o);
        rqs_forward_in_bin(b, x, out, ld);
    } else {
        int k = knot_search(H, K, bottom, x);
        if (kbin) *kbin = k;
        RqsBin b = rqs_bin(W, H, D, K, k, left, bottom, o);
        float ld_own;
        rqs_inverse_in_bin(b, x, out, ld_own);
        if (own_ld) {
            ld = ld_own;
        } else {
            // flow.py:42-47 + coupling.py:84-95: forward log-derivative re-evaluated at the
            // recovered point (its own inside test and bin search), negated.
            ld = 0.f;
            if (out >= left && out <= right) {
                int k2 = knot_search(W, K, left, out);
                RqsBin b2 = (k2 == k) ? b : rqs_bin(W, H, D, K, k2, left, bottom, o);
                float y2, ldf;
                rqs_forward_in_bin(b2, out, y2, ldf);
                ld = -ldf;
            }
        }
    }
}

// ---------------------------------------------------------------------------------------
// cubic spline
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ float sign_f(float v) { return (v > 0.f) ? 1.f : ((v < 0.f) ? -1.f : 0.f); }
// cubic_spline.py:18-20
__device__ __forceinline__ float cbrt_ref(float v) { return sign_f(v) * expf(logf(fabsf(v)) / 3.0f); }

struct CubBin {
    float a, b, c, d, xl, xr;
};

// W, H: bin sizes (after softmax_bins); k: bin; cw/ch: cumulative sums BEFORE bin k.
// cubic_spline.py:118-138
template <class PW, class PH>
__device__ __forceinline__ CubBin cubic_bin(PW W, PH H, int K, int k, float cw, float ch, float ul,
                                            float ur) {
    float wk = W[k], hk = H[k];
    float sk = hk / wk;
    float dl, dr;
    if (k == 0) {
        dl = sigmoid_f(ul) * 3.f * sk;
    } else {
        float wp = W[k - 1], sp = H[k - 1] / wp;
        float m1 = fminf(fabsf(sp), fabsf(sk));
        float m2 = 0.5f * (wk * sp + wp * sk) / (wp + wk);
        dl = fminf(m1, m2) * (sign_f(sp) + sign_f(sk));
    }
    if (k == K - 1) {
        dr = sigmoid_f(ur) * 3.f * sk;
    } else {
        float wn = W[k + 1], sn = H[k + 1] / wn;
        float m1 = fminf(fabsf(sk), fabsf(sn));
        float m2 = 0.5f * (wn * sk + wk * sn) / (wk + wn);
        dr = fminf(m1, m2) * (sign_f(sk) + sign_f(sn));
    }
    CubBin r;
    r.a = (dl + dr - 2.f * sk) / (wk * wk);
    r.b = (3.f * sk - 2.f * dl - dr) / wk;
    r.c = dl;
    r.d = ch;
    r.xl = cw;
    r.xr = (k == K - 1) ? 1.f : cw + wk;            // cumwidths[..., -1] = 1 (:108)
    return r;
}

// Walk the knots of `S` (the searched sizes) accumulating both cumulative sums; returns the bin
// of u and the cumulative widths/heights before it.   search_sorted.py:3-5 on cubic_spline.py:107-116
template <class PW, class PH>
__device__ __forceinline__ int cubic_search(PW W, PH H, int K, bool search_heights, float u, float& cw,
                                            float& ch) {
    float aw = 0.f, ah = 0.f;
    int k = 0;
    cw = 0.f;
    ch = 0.f;
    for (int i = 1; i < K; ++i) {
        aw += W[i - 1];
        ah += H[i - 1];
        float knot = search_heights ? ah : aw;
        if (u >= knot) { k = i; cw = aw; ch = ah; }
    }
    // the last knot is 1 + 1e-6: an inside u (<= 1) never reaches it
    return k;
}

__device__ __forceinline__ float cubic_forward_in_bin(const CubBin& b, float u, float& ld) {
    float s = u - b.xl;
    float out = b.a * s * s * s + b.b * s * s + b.c * s + b.d;
    ld = logf(3.f * b.a * s * s + 2.f * b.b * s + b.c);
    return out;
}

// cubic_spline.py:153-228
template <class O = CubDefaults>
__device__ __forceinline__ float cubic_inverse_in_bin(const CubBin& k, float u, float& ld, const O& o = O()) {
    float b_ = (k.b / k.a) / 3.f;
    float c_ = (k.c / k.a) / 3.f;
    float d_ = (k.d - u) / k.a;
    float delta_1 = -b_ * b_ + c_;
    float delta_2 = -c_ * b_ + d_;
    float delta_3 = b_ * d_ - c_ * c_;
    float disc = 4.f * delta_1 * delta_3 - delta_2 * delta_2;
    float dep_1 = -2.f * b_ * delta_1 + delta_2;
    float dep_2 = delta_1;
    float out;
    if (disc > 0.f) {
        float theta = atan2f(sqrtf(disc), -dep_1) / 3.f;
        float c1 = cosf(theta), c2 = sinf(theta);
        float scale = 2.f * sqrtf(-dep_2);
        float shift = -b_ + k.xl;
        float r1 = c1 * scale + shift;
        float r2 = (-0.5f * c1 - 0.5f * 1.7320508075688772f * c2) * scale + shift;
        float r3 = (-0.5f * c1 + 0.5f * 1.7320508075688772f * c2) * scale + shift;
        float lo = k.xl - o.eps(), hi = k.xr + o.eps();
        bool ok1 = (lo < r1) && (r1 < hi), ok2 = (lo < r2) && (r2 < hi), ok3 = (lo < r3) && (r3 < hi);
        out = ok1 ? r1 : (ok2 ? r2 : (ok3 ? r3 : r1));      // argsort(masks, desc)[..., 0]  (:212)
    } else {
        float sq = sqrtf(-disc);
        float p = cbrt_ref((-dep_1 + sq) / 2.f);
        float q = cbrt_ref((-dep_1 - sq) / 2.f);
        out = (p + q) - b_ + k.xl;
    }
    if (fabsf(k.a) < o.quad()) {                             // :217-223
        float qc = k.d - u;
        float alpha = (-k.c + sqrtf(k.c * k.c - 4.f * k.b * qc)) / (2.f * k.b);
        out = alpha + k.xl;
    }
    float s = out - k.xl;
    ld = -logf(3.f * k.a * s * s + 2.f * k.b * s + k.c);
    return out;
}

// prm = [uw(K) | uh(K) | left, right]  (destroyed).  Same contract as rqs_element.
template <class P, class O = CubDefaults>
__device__ __forceinline__ void cubic_element(P prm, int K, float lower, float upper, bool inverse,
                                              bool own_ld, float x, float& out, float& ld,
                                              int* kbin = nullptr, const O& o = O()) {
    out = x;
    ld = 0.f;
    if (kbin) *kbin = -1;
    if (!(x >= lower && x <= upper)) return;
    OffsetView<P> W{prm, 0}, H{prm, K};
    const float ul = prm[2 * K], ur = prm[2 * K + 1];
    softmax_bins(W, K, o.min_w());
    softmax_bins(H, K, o.min_h());
    const float span = upper - lower;
    float u = (x - lower) / span;                            // :99-102
    float cw, ch;
    if (!inverse) {
        int k = cubic_search(W, H, K, false, u, cw, ch);
        if (kbin) *kbin = k;
        CubBin b = cubic_bin(W, H, K, k, cw, ch, ul, ur);
        float v = cubic_forward_in_bin(b, u, ld);
        out = v * span + lower;                              // :244-245 (log terms cancel: same box)
    } else {
        int k = cubic_search(W, H, K, true, u, cw, ch);
        if (kbin) *kbin = k;
        CubBin b = cubic_bin(W, H, K, k, cw, ch, ul, ur);
        float ld_own;
        float v = cubic_inverse_in_bin(b, u, ld_own, o);
        out = v * span + lower;
        if (own_ld) {
            ld = ld_own;
        } else {
            ld = 0.f;
            if (out >= lower && out <= upper) {
                float u2 = (out - lower) / span;
                int k2 = cubic_search(W, H, K, false, u2, cw, ch);
                CubBin b2 = (k2 == k) ? b : cubic_bin(W, H, K, k2, cw, ch, ul, ur);
                float ldf;
                (void)cubic_forward_in_bin(b2, u2, ldf);
                ld = -ldf;
            }
        }
    }
}

}  // namespace stb
