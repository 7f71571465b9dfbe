// Gradients of the element-wise transforms (what autograd derives for the reference's
// util/rational_quadratic_spline.py / util/cubic_spline.py / flows/affine.py).
//
// The in-bin maps are differentiated with small forward-mode dual numbers (value + N partials):
// S(x; q) and L = log dS/dx are evaluated once with all inputs seeded, which yields every partial
// the chain rule needs.  For the inverse direction x = S^-1(y; q), ld = -L(x; q) the implicit-
// function theorem gives
//     dx/dy = 1 / S_x,   dx/dq = -S_q / S_x,   dld/dy = -L_x / S_x,   dld/dq = -L_q + L_x S_q / S_x .
// The parameter normalisation (softmax -> cumulative knots, softplus / sigmoid derivatives) is
// back-propagated by hand.
#pragma once
#include "stb_math.cuh"

namespace stb {

template <int N>
struct Dual {
    float v;
    float d[N];
};

template <int N>
__device__ __forceinline__ Dual<N> dconst(float v) {
    Dual<N> r;
    r.v = v;
#pragma unroll
    for (int i = 0; i < N; ++i) r.d[i] = 0.f;
    return r;
}
template <int N>
__device__ __forceinline__ Dual<N> dvar(float v, int idx) {
    Dual<N> r = dconst<N>(v);
    r.d[idx] = 1.f;
    return r;
}
#define STB_DUAL_BIN(OP, EXPR_V, EXPR_D)                                                      \
    template <int N>                                                                          \
    __device__ __forceinline__ Dual<N> OP(const Dual<N>& a, const Dual<N>& b) {               \
        Dual<N> r;                                                                            \
        r.v = EXPR_V;                                                                         \
        _Pragma("unroll") for (int i = 0; i < N; ++i) r.d[i] = EXPR_D;                        \
        return r;                                                                             \
    }
STB_DUAL_BIN(operator+, a.v + b.v, a.d[i] + b.d[i])
STB_DUAL_BIN(operator-, a.v - b.v, a.d[i] - b.d[i])
STB_DUAL_BIN(operator*, a.v * b.v, a.d[i] * b.v + a.v * b.d[i])
#undef STB_DUAL_BIN
template <int N>
__device__ __forceinline__ Dual<N> operator/(const Dual<N>& a, const Dual<N>& b) {
    Dual<N> r;
    const float inv = 1.f / b.v;
    r.v = a.v * inv;
#pragma unroll
    for (int i = 0; i < N; ++i) r.d[i] = (a.d[i] - r.v * b.d[i]) * inv;
    return r;
}
template <int N>
__device__ __forceinline__ Dual<N> operator*(float s, const Dual<N>& a) {
    Dual<N> r;
    r.v = s * a.v;
#pragma unroll
    for (int i = 0; i < N; ++i) r.d[i] = s * a.d[i];
    return r;
}
template <int N>
__device__ __forceinline__ Dual<N> operator-(const Dual<N>& a) { return -1.f * a; }
template <int N>
__device__ __forceinline__ Dual<N> dlog(const Dual<N>& a) {
    Dual<N> r;
    r.v = logf(a.v);
    const float inv = 1.f / a.v;
#pragma unroll
    for (int i = 0; i < N; ++i) r.d[i] = a.d[i] * inv;
    return r;
}
template <int N>
__device__ __forceinline__ Dual<N> dabs(const Dual<N>& a) { return a.v >= 0.f ? a : -a; }   // |.|' = sign
template <int N>
__device__ __forceinline__ Dual<N> dmin(const Dual<N>& a, const Dual<N>& b) { return (a.v <= b.v) ? a : b; }
template <int N>
__device__ __forceinline__ Dual<N> dsigmoid(const Dual<N>& a) {
    Dual<N> r;
    r.v = sigmoid_f(a.v);
    const float g = r.v * (1.f - r.v);
#pragma unroll
    for (int i = 0; i < N; ++i) r.d[i] = a.d[i] * g;
    return r;
}

// --------------------------------------------------------------------------------------------
// rational-quadratic spline: S and log S' inside one bin, inputs (x, xk, xk1, yk, yk1, d0, d1)
// --------------------------------------------------------------------------------------------
enum { RQ_X = 0, RQ_XK, RQ_XK1, RQ_YK, RQ_YK1, RQ_D0, RQ_D1, RQ_N };

__device__ __forceinline__ void rqs_bin_dual(float x, float xk, float xk1, float yk, float yk1, float d0,
                                             float d1, Dual<RQ_N>& S, Dual<RQ_N>& L) {
    typedef Dual<RQ_N> D;
    const D X = dvar<RQ_N>(x, RQ_X), XK = dvar<RQ_N>(xk, RQ_XK), XK1 = dvar<RQ_N>(xk1, RQ_XK1);
    const D YK = dvar<RQ_N>(yk, RQ_YK), YK1 = dvar<RQ_N>(yk1, RQ_YK1);
    const D D0 = dvar<RQ_N>(d0, RQ_D0), D1 = dvar<RQ_N>(d1, RQ_D1);
    const D wk = XK1 - XK, hk = YK1 - YK;
    const D delta = hk / wk;
    const D theta = (X - XK) / wk;
    const D omt = dconst<RQ_N>(1.f) - theta;
    const D tt = theta * omt;
    const D den = delta + (D0 + D1 - 2.f * delta) * tt;
    S = YK + hk * (delta * theta * theta + D0 * tt) / den;
    const D dnum = delta * delta * (D1 * theta * theta + 2.f * (delta * tt) + D0 * omt * omt);
    L = dlog(dnum) - 2.f * dlog(den);
}

// Gradients of one RQS element.
//   sw, sh : NORMALISED bin sizes (min + scale * softmax), K each;  ud: K-1 raw derivative params
//            (K+1, the boundaries included, with o.free_edge())
//   direction / own_ld as rqs_element;  x: the element's input;  g_out, g_ld: incoming gradients
// Writes g_x and the gradient wrt the K + K + (K-1 or K+1) RAW parameters into gp[] (same indexable type).
// Domain [left, right] -> codomain [bottom, top] (rational_quadratic_spline.py:55-64); the common case is
// left == bottom == lower, right == top == upper.
template <class P, class O = RqsDefaults>
__device__ __forceinline__ void rqs_element_grad(P prm, P gp, int K, float left, float right, float bottom,
                                                 float top, bool inverse, float x, float g_out, float g_ld,
                                                 float& g_x, const O& o = O()) {
    const int Pn = o.free_edge() ? 3 * K + 1 : 3 * K - 1;
    for (int i = 0; i < Pn; ++i) gp[i] = 0.f;
    g_x = g_out;                                   // identity tails
    if (!(x >= (inverse ? bottom : left) && x <= (inverse ? top : right))) return;
    OffsetView<P> W{prm, 0}, H{prm, K}, D{prm, 2 * K};
    OffsetView<P> GW{gp, 0}, GH{gp, K}, GD{gp, 2 * K};
    const float mw = o.min_w(), mh = o.min_h();
    softmax_bins(W, K, mw);                        // normalised sizes, kept (not turned into knots)
    softmax_bins(H, K, mh);
    const float spanx = right - left, spany = top - bottom;
    // bin search by running sums (same arithmetic as sizes_to_knots + knot_search)
    int k = 0;
    float cwk = 0.f, chk = 0.f, cw = 0.f, ch = 0.f;
    for (int i = 1; i < K; ++i) {
        cw += W[i - 1];
        ch += H[i - 1];
        const float knot = inverse ? spany * ch + bottom : spanx * cw + left;
        if (x >= knot) { k = i; cwk = cw; chk = ch; }
    }
    const float wk_ = W[k], hk_ = H[k];
    const float xk = (k == 0) ? left : spanx * cwk + left;
    const float yk = (k == 0) ? bottom : spany * chk + bottom;
    const float xk1 = (k == K - 1) ? right : spanx * (cwk + wk_) + left;
    const float yk1 = (k == K - 1) ? top : spany * (chk + hk_) + bottom;
    float u0, u1;
    if (o.free_edge()) {
        u0 = D[k];
        u1 = D[k + 1];
    } else {
        u0 = (k == 0) ? o.edge() : D[k - 1];
        u1 = (k == K - 1) ? o.edge() : D[k];
    }
    const float d0 = o.min_d() + softplus_f(u0), d1 = o.min_d() + softplus_f(u1);

    float xe = x;                                  // point at which S, L are expanded
    if (inverse) {
        RqsBin b;
        b.xk = xk; b.wk = xk1 - xk; b.yk = yk; b.hk = yk1 - yk; b.delta = b.hk / b.wk; b.d0 = d0; b.d1 = d1;
        float ld_own;
        rqs_inverse_in_bin(b, x, xe, ld_own);
    }
    Dual<RQ_N> S, L;
    rqs_bin_dual(xe, xk, xk1, yk, yk1, d0, d1, S, L);
    float gq[RQ_N];                                // gradient wrt (x_in, xk, xk1, yk, yk1, d0, d1)
    if (!inverse) {
#pragma unroll
        for (int i = 0; i < RQ_N; ++i) gq[i] = g_out * S.d[i] + g_ld * L.d[i];
    } else {
        // coupling semantics: a recovered point outside the box gets ld = 0 (no gradient through ld)
        const float gl = (xe >= left && xe <= right) ? g_ld : 0.f;
        const float gy = (g_out - gl * L.d[RQ_X]) / S.d[RQ_X];
        gq[RQ_X] = gy;
#pragma unroll
        for (int i = 1; i < RQ_N; ++i) gq[i] = -S.d[i] * gy - gl * L.d[i];
    }
    g_x = gq[RQ_X];
    // knots -> normalised sizes (cumulative sums; the box ends are constants)
    const float g_cw = spanx * ((k > 0 ? gq[RQ_XK] : 0.f) + (k < K - 1 ? gq[RQ_XK1] : 0.f));
    const float g_wk = spanx * (k < K - 1 ? gq[RQ_XK1] : 0.f);
    const float g_ch = spany * ((k > 0 ? gq[RQ_YK] : 0.f) + (k < K - 1 ? gq[RQ_YK1] : 0.f));
    const float g_hk = spany * (k < K - 1 ? gq[RQ_YK1] : 0.f);
    // sizes -> raw (softmax backward): w_i = min + scale * s_i, s_i = (w_i - min) / scale
    // (min * K == 1 leaves scale 0: the sizes are constants and their raw parameters get no gradient)
    const float scale_w = 1.f - mw * (float)K, scale_h = 1.f - mh * (float)K;
    float dotw = 0.f, doth = 0.f;
    for (int i = 0; i <= k; ++i) {
        const float gwi = (i < k) ? g_cw : g_wk, ghi = (i < k) ? g_ch : g_hk;
        dotw += (W[i] - mw) * gwi;                 // = scale * s_i * g_w_i
        doth += (H[i] - mh) * ghi;
    }
    for (int i = 0; i < K; ++i) {
        const float gwi = (i < k) ? g_cw : ((i == k) ? g_wk : 0.f);
        const float ghi = (i < k) ? g_ch : ((i == k) ? g_hk : 0.f);
        const float sw = (O::kRuntime && scale_w == 0.f) ? 0.f : (W[i] - mw) / scale_w;
        const float sh = (O::kRuntime && scale_h == 0.f) ? 0.f : (H[i] - mh) / scale_h;
        GW[i] = sw * (scale_w * gwi - dotw);
        GH[i] = sh * (scale_h * ghi - doth);
    }
    // derivatives: d = min + softplus(u), softplus' = sigmoid (1 beyond the threshold)
    if (o.free_edge()) {                           // the boundary parameters are free too
        GD[k] = gq[RQ_D0] * (u0 > 20.f ? 1.f : sigmoid_f(u0));
        GD[k + 1] = gq[RQ_D1] * (u1 > 20.f ? 1.f : sigmoid_f(u1));
    } else {
        if (k > 0) GD[k - 1] = gq[RQ_D0] * (u0 > 20.f ? 1.f : sigmoid_f(u0));
        if (k < K - 1) GD[k] = gq[RQ_D1] * (u1 > 20.f ? 1.f : sigmoid_f(u1));
    }
}

// --------------------------------------------------------------------------------------------
// cubic spline: inputs (u, wp, wk, wn, hp, hk, hn, cw, ch, ul, ur) on the unit box
// --------------------------------------------------------------------------------------------
enum { CU_U = 0, CU_WP, CU_WK, CU_WN, CU_HP, CU_HK, CU_HN, CU_CW, CU_CH, CU_UL, CU_UR, CU_N };

__device__ __forceinline__ Dual<CU_N> dsign_sum(const Dual<CU_N>& a, const Dual<CU_N>& b) {
    return dconst<CU_N>(sign_f(a.v) + sign_f(b.v));                   // sign has zero gradient
}

__device__ __forceinline__ void cubic_bin_dual(int k, int K, float u, float wp, float wk, float wn, float hp,
                                               float hk, float hn, float cw, float ch, float ul, float ur,
                                               Dual<CU_N>& S, Dual<CU_N>& L) {
    typedef Dual<CU_N> D;
    const D U = dvar<CU_N>(u, CU_U), WP = dvar<CU_N>(wp, CU_WP), WK = dvar<CU_N>(wk, CU_WK), WN = dvar<CU_N>(wn, CU_WN);
    const D HP = dvar<CU_N>(hp, CU_HP), HK = dvar<CU_N>(hk, CU_HK), HN = dvar<CU_N>(hn, CU_HN);
    const D CW = dvar<CU_N>(cw, CU_CW), CH = dvar<CU_N>(ch, CU_CH);
    const D UL = dvar<CU_N>(ul, CU_UL), UR = dvar<CU_N>(ur, CU_UR);
    const D sk = HK / WK;
    D dl, dr;
    if (k == 0) {
        dl = 3.f * (dsigmoid(UL) * sk);
    } else {
        const D sp = HP / WP;
        const D m1 = dmin(dabs(sp), dabs(sk));
        const D m2 = 0.5f * ((WK * sp + WP * sk) / (WP + WK));
        dl = dmin(m1, m2) * dsign_sum(sp, sk);
    }
    if (k == K - 1) {
        dr = 3.f * (dsigmoid(UR) * sk);
    } else {
        const D sn = HN / WN;
        const D m1 = dmin(dabs(sk), dabs(sn));
        const D m2 = 0.5f * ((WN * sk + WK * sn) / (WK + WN));
        dr = dmin(m1, m2) * dsign_sum(sk, sn);
    }
    const D a = (dl + dr - 2.f * sk) / (WK * WK);
    const D b = (3.f * sk - 2.f * dl - dr) / WK;
    const D s = U - CW;
    S = a * s * s * s + b * s * s + dl * s + CH;
    L = dlog(3.f * (a * s * s) + 2.f * (b * s) + dl);
}

// prm = [uw(K) | uh(K) | left, right] raw; gp receives the gradient wrt those 2K + 2 values.
template <class P, class O = CubDefaults>
__device__ __forceinline__ void cubic_element_grad(P prm, P gp, int K, float lower, float upper, bool inverse,
                                                   float x, float g_out, float g_ld, float& g_x,
                                                   const O& o = O()) {
    const int Pn = 2 * K + 2;
    for (int i = 0; i < Pn; ++i) gp[i] = 0.f;
    g_x = g_out;
    if (!(x >= lower && x <= upper)) return;
    OffsetView<P> W{prm, 0}, H{prm, K};
    OffsetView<P> GW{gp, 0}, GH{gp, K};
    const float ul = prm[2 * K], ur = prm[2 * K + 1];
    const float mw = o.min_w(), mh = o.min_h();
    softmax_bins(W, K, mw);
    softmax_bins(H, K, mh);
    const float span = upper - lower;
    const float u = (x - lower) / span;
    float cw, ch;
    int k = cubic_search(W, H, K, inverse, u, cw, ch);
    float ue = u;
    if (inverse) {
        const CubBin b = cubic_bin(W, H, K, k, cw, ch, ul, ur);
        float ld_own;
        ue = cubic_inverse_in_bin(b, u, ld_own, o);
    }
    const float wp = k > 0 ? W[k - 1] : 1.f, hp = k > 0 ? H[k - 1] : 1.f;
    const float wn = k < K - 1 ? W[k + 1] : 1.f, hn = k < K - 1 ? H[k + 1] : 1.f;
    Dual<CU_N> S, L;
    cubic_bin_dual(k, K, ue, wp, W[k], wn, hp, H[k], hn, cw, ch, ul, ur, S, L);
    // out = span * S + lower, u = (x - lower) / span; ld = L (same box on both axes)
    float gq[CU_N];
    if (!inverse) {
#pragma unroll
        for (int i = 0; i < CU_N; ++i) gq[i] = g_out * span * S.d[i] + g_ld * L.d[i];
        g_x = gq[CU_U] / span;
    } else {
        const float xo = ue * span + lower;
        const float gl = (xo >= lower && xo <= upper) ? g_ld : 0.f;
        // x_out = span * ue + lower;  ue solves S(ue; q) = u;  ld = -L(ue; q)
        const float gu = (g_out * span - gl * L.d[CU_U]) / S.d[CU_U];      // gradient wrt u (input, unit box)
        gq[CU_U] = gu;
#pragma unroll
        for (int i = 1; i < CU_N; ++i) gq[i] = -S.d[i] * gu - gl * L.d[i];
        g_x = gu / span;
    }
    // neighbours / cumulative sums -> normalised sizes
    const float scale_w = 1.f - mw * (float)K, scale_h = 1.f - mh * (float)K;
    float dotw = 0.f, doth = 0.f;
    for (int i = 0; i < K; ++i) {
        float gwi = (i < k) ? gq[CU_CW] : 0.f, ghi = (i < k) ? gq[CU_CH] : 0.f;
        if (i == k - 1) { gwi += gq[CU_WP]; ghi += gq[CU_HP]; }
        if (i == k) { gwi += gq[CU_WK]; ghi += gq[CU_HK]; }
        if (i == k + 1) { gwi += gq[CU_WN]; ghi += gq[CU_HN]; }
        GW[i] = gwi;                                  // stash, converted below
        GH[i] = ghi;
        dotw += (W[i] - mw) * gwi;
        doth += (H[i] - mh) * ghi;
    }
    for (int i = 0; i < K; ++i) {
        const float sw = (O::kRuntime && scale_w == 0.f) ? 0.f : (W[i] - mw) / scale_w;
        const float sh = (O::kRuntime && scale_h == 0.f) ? 0.f : (H[i] - mh) / scale_h;
        GW[i] = sw * (scale_w * GW[i] - dotw);
        GH[i] = sh * (scale_h * GH[i] - doth);
    }
    gp[2 * K] = (k == 0) ? gq[CU_UL] : 0.f;
    gp[2 * K + 1] = (k == K - 1) ? gq[CU_UR] : 0.f;
}

}  // namespace stb
