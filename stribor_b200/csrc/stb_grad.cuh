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

template <int N, class T = float>
struct Dual {
    T v;
    T d[N];
};

template <int N, class T>
__device__ __forceinline__ Dual<N, T> dconst(T v) {
    Dual<N, T> r;
    r.v = v;
#pragma unroll
    for (int i = 0; i < N; ++i) r.d[i] = T(0);
    return r;
}
template <int N, class T>
__device__ __forceinline__ Dual<N, T> dvar(T v, int idx) {
    Dual<N, T> r = dconst<N>(v);
    r.d[idx] = T(1);
    return r;
}
#define STB_DUAL_BIN(OP, EXPR_V, EXPR_D)                                                      \
    template <int N, class T>                                                                 \
    __device__ __forceinline__ Dual<N, T> OP(const Dual<N, T>& a, const Dual<N, T>& b) {      \
        Dual<N, T> r;                                                                         \
        r.v = EXPR_V;                                                                         \
        _Pragma("unroll") for (int i = 0; i < N; ++i) r.d[i] = EXPR_D;                        \
        return r;                                                                             \
    }
STB_DUAL_BIN(operator+, a.v + b.v, a.d[i] + b.d[i])
STB_DUAL_BIN(operator-, a.v - b.v, a.d[i] - b.d[i])
STB_DUAL_BIN(operator*, a.v * b.v, a.d[i] * b.v + a.v * b.d[i])
#undef STB_DUAL_BIN
template <int N, class T>
__device__ __forceinline__ Dual<N, T> operator/(const Dual<N, T>& a, const Dual<N, T>& b) {
    Dual<N, T> r;
    const T inv = T(1) / b.v;
    r.v = a.v * inv;
#pragma unroll
    for (int i = 0; i < N; ++i) r.d[i] = (a.d[i] - r.v * b.d[i]) * inv;
    return r;
}
template <int N, class T>
__device__ __forceinline__ Dual<N, T> operator*(T s, const Dual<N, T>& a) {
    Dual<N, T> r;
    r.v = s * a.v;
#pragma unroll
    for (int i = 0; i < N; ++i) r.d[i] = s * a.d[i];
    return r;
}
template <int N, class T>
__device__ __forceinline__ Dual<N, T> operator-(const Dual<N, T>& a) { return T(-1) * a; }
template <int N, class T>
__device__ __forceinline__ Dual<N, T> dlog(const Dual<N, T>& a) {
    Dual<N, T> r;
    r.v = log_(a.v);
    const T inv = T(1) / a.v;
#pragma unroll
    for (int i = 0; i < N; ++i) r.d[i] = a.d[i] * inv;
    return r;
}
template <int N, class T>
__device__ __forceinline__ Dual<N, T> dabs(const Dual<N, T>& a) { return a.v >= T(0) ? a : -a; }   // |.|' = sign
template <int N, class T>
__device__ __forceinline__ Dual<N, T> dmin(const Dual<N, T>& a, const Dual<N, T>& b) { return (a.v <= b.v) ? a : b; }
template <int N, class T>
__device__ __forceinline__ Dual<N, T> dsigmoid(const Dual<N, T>& a) {
    Dual<N, T> r;
    r.v = sigmoid_f(a.v);
    const T g = r.v * (T(1) - r.v);
#pragma unroll
    for (int i = 0; i < N; ++i) r.d[i] = a.d[i] * g;
    return r;
}

// --------------------------------------------------------------------------------------------
// rational-quadratic spline: S and log S' inside one bin, inputs (x, xk, xk1, yk, yk1, d0, d1)
// --------------------------------------------------------------------------------------------
enum { RQ_X = 0, RQ_XK, RQ_XK1, RQ_YK, RQ_YK1, RQ_D0, RQ_D1, RQ_N };

template <class T>
__device__ __forceinline__ void rqs_bin_dual(T x, T xk, T xk1, T yk, T yk1, T d0, T d1, Dual<RQ_N, T>& S,
                                             Dual<RQ_N, T>& L) {
    typedef Dual<RQ_N, T> D;
    const D X = dvar<RQ_N>(x, RQ_X), XK = dvar<RQ_N>(xk, RQ_XK), XK1 = dvar<RQ_N>(xk1, RQ_XK1);
    const D YK = dvar<RQ_N>(yk, RQ_YK), YK1 = dvar<RQ_N>(yk1, RQ_YK1);
    const D D0 = dvar<RQ_N>(d0, RQ_D0), D1 = dvar<RQ_N>(d1, RQ_D1);
    const D wk = XK1 - XK, hk = YK1 - YK;
    const D delta = hk / wk;
    const D theta = (X - XK) / wk;
    const D omt = dconst<RQ_N>(T(1)) - theta;
    const D tt = theta * omt;
    const D den = delta + (D0 + D1 - T(2) * delta) * tt;
    S = YK + hk * (delta * theta * theta + D0 * tt) / den;
    const D dnum = delta * delta * (D1 * theta * theta + T(2) * (delta * tt) + D0 * omt * omt);
    L = dlog(dnum) - T(2) * dlog(den);
}

// Gradients of one RQS element.
//   sw, sh : NORMALISED bin sizes (min + scale * softmax), K each;  ud: K-1 raw derivative params
//            (K+1, the boundaries included, with o.free_edge())
//   direction / own_ld as rqs_element;  x: the element's input;  g_out, g_ld: incoming gradients
// Writes g_x and the gradient wrt the K + K + (K-1 or K+1) RAW parameters into gp[] (same indexable type).
// Domain [left, right] -> codomain [bottom, top] (rational_quadratic_spline.py:55-64); the common case is
// left == bottom == lower, right == top == upper.
template <class P, class O = RqsDefaultsT<elem_t<P>>>
__device__ __forceinline__ void rqs_element_grad(P prm, P gp, int K, elem_t<P> left, elem_t<P> right,
                                                 elem_t<P> bottom, elem_t<P> top, bool inverse, elem_t<P> x,
                                                 elem_t<P> g_out, elem_t<P> g_ld, elem_t<P>& g_x, const O& o = O()) {
    using T = elem_t<P>;
    const int Pn = o.free_edge() ? 3 * K + 1 : 3 * K - 1;
    for (int i = 0; i < Pn; ++i) gp[i] = T(0);
    g_x = g_out;                                   // identity tails
    if (!(x >= (inverse ? bottom : left) && x <= (inverse ? top : right))) return;
    OffsetView<P> W{prm, 0}, H{prm, K}, D{prm, 2 * K};
    OffsetView<P> GW{gp, 0}, GH{gp, K}, GD{gp, 2 * K};
    const T mw = o.min_w(), mh = o.min_h();
    softmax_bins(W, K, mw);                        // normalised sizes, kept (not turned into knots)
    softmax_bins(H, K, mh);
    const T spanx = right - left, spany = top - bottom;
    // bin search by running sums (same arithmetic as sizes_to_knots + knot_search)
    int k = 0;
    T cwk = T(0), chk = T(0), cw = T(0), ch = T(0);
    for (int i = 1; i < K; ++i) {
        cw += W[i - 1];
        ch += H[i - 1];
        const T knot = inverse ? spany * ch + bottom : spanx * cw + left;
        if (x >= knot) { k = i; cwk = cw; chk = ch; }
    }
    const T wk_ = W[k], hk_ = H[k];
    const T xk = (k == 0) ? left : spanx * cwk + left;
    const T yk = (k == 0) ? bottom : spany * chk + bottom;
    const T xk1 = (k == K - 1) ? right : spanx * (cwk + wk_) + left;
    const T yk1 = (k == K - 1) ? top : spany * (chk + hk_) + bottom;
    T u0, u1;
    if (o.free_edge()) {
        u0 = D[k];
        u1 = D[k + 1];
    } else {
        u0 = (k == 0) ? o.edge() : D[k - 1];
        u1 = (k == K - 1) ? o.edge() : D[k];
    }
    const T d0 = o.min_d() + softplus_f(u0), d1 = o.min_d() + softplus_f(u1);

    T xe = x;                                      // point at which S, L are expanded
    if (inverse) {
        RqsBinT<T> b;
        b.xk = xk; b.wk = xk1 - xk; b.yk = yk; b.hk = yk1 - yk; b.delta = b.hk / b.wk; b.d0 = d0; b.d1 = d1;
        T ld_own;
        rqs_inverse_in_bin(b, x, xe, ld_own);
    }
    Dual<RQ_N, T> S, L;
    rqs_bin_dual(xe, xk, xk1, yk, yk1, d0, d1, S, L);
    T gq[RQ_N];                                    // gradient wrt (x_in, xk, xk1, yk, yk1, d0, d1)
    if (!inverse) {
#pragma unroll
        for (int i = 0; i < RQ_N; ++i) gq[i] = g_out * S.d[i] + g_ld * L.d[i];
    } else {
        // coupling semantics: a recovered point outside the box gets ld = 0 (no gradient through ld)
        const T gl = (xe >= left && xe <= right) ? g_ld : T(0);
        const T gy = (g_out - gl * L.d[RQ_X]) / S.d[RQ_X];
        gq[RQ_X] = gy;
#pragma unroll
        for (int i = 1; i < RQ_N; ++i) gq[i] = -S.d[i] * gy - gl * L.d[i];
    }
    g_x = gq[RQ_X];
    // knots -> normalised sizes (cumulative sums; the box ends are constants)
    const T g_cw = spanx * ((k > 0 ? gq[RQ_XK] : T(0)) + (k < K - 1 ? gq[RQ_XK1] : T(0)));
    const T g_wk = spanx * (k < K - 1 ? gq[RQ_XK1] : T(0));
    const T g_ch = spany * ((k > 0 ? gq[RQ_YK] : T(0)) + (k < K - 1 ? gq[RQ_YK1] : T(0)));
    const T g_hk = spany * (k < K - 1 ? gq[RQ_YK1] : T(0));
    // sizes -> raw (softmax backward): w_i = min + scale * s_i, s_i = (w_i - min) / scale
    // (min * K == 1 leaves scale 0: the sizes are constants and their raw parameters get no gradient)
    const T scale_w = T(1) - mw * (T)K, scale_h = T(1) - mh * (T)K;
    T dotw = T(0), doth = T(0);
    for (int i = 0; i <= k; ++i) {
        const T gwi = (i < k) ? g_cw : g_wk, ghi = (i < k) ? g_ch : g_hk;
        dotw += (W[i] - mw) * gwi;                 // = scale * s_i * g_w_i
        doth += (H[i] - mh) * ghi;
    }
    for (int i = 0; i < K; ++i) {
        const T gwi = (i < k) ? g_cw : ((i == k) ? g_wk : T(0));
        const T ghi = (i < k) ? g_ch : ((i == k) ? g_hk : T(0));
        const T sw = (O::kRuntime && scale_w == T(0)) ? T(0) : (W[i] - mw) / scale_w;
        const T sh = (O::kRuntime && scale_h == T(0)) ? T(0) : (H[i] - mh) / scale_h;
        GW[i] = sw * (scale_w * gwi - dotw);
        GH[i] = sh * (scale_h * ghi - doth);
    }
    // derivatives: d = min + softplus(u), softplus' = sigmoid (1 beyond the threshold)
    if (o.free_edge()) {                           // the boundary parameters are free too
        GD[k] = gq[RQ_D0] * (u0 > T(20) ? T(1) : sigmoid_f(u0));
        GD[k + 1] = gq[RQ_D1] * (u1 > T(20) ? T(1) : sigmoid_f(u1));
    } else {
        if (k > 0) GD[k - 1] = gq[RQ_D0] * (u0 > T(20) ? T(1) : sigmoid_f(u0));
        if (k < K - 1) GD[k] = gq[RQ_D1] * (u1 > T(20) ? T(1) : sigmoid_f(u1));
    }
}

// --------------------------------------------------------------------------------------------
// cubic spline: inputs (u, wp, wk, wn, hp, hk, hn, cw, ch, ul, ur) on the unit box
// --------------------------------------------------------------------------------------------
enum { CU_U = 0, CU_WP, CU_WK, CU_WN, CU_HP, CU_HK, CU_HN, CU_CW, CU_CH, CU_UL, CU_UR, CU_N };

template <class T>
__device__ __forceinline__ Dual<CU_N, T> dsign_sum(const Dual<CU_N, T>& a, const Dual<CU_N, T>& b) {
    return dconst<CU_N>(sign_f(a.v) + sign_f(b.v));                   // sign has zero gradient
}

template <class T>
__device__ __forceinline__ void cubic_bin_dual(int k, int K, T u, T wp, T wk, T wn, T hp, T hk, T hn, T cw, T ch,
                                               T ul, T ur, Dual<CU_N, T>& S, Dual<CU_N, T>& L) {
    typedef Dual<CU_N, T> D;
    const D U = dvar<CU_N>(u, CU_U), WP = dvar<CU_N>(wp, CU_WP), WK = dvar<CU_N>(wk, CU_WK), WN = dvar<CU_N>(wn, CU_WN);
    const D HP = dvar<CU_N>(hp, CU_HP), HK = dvar<CU_N>(hk, CU_HK), HN = dvar<CU_N>(hn, CU_HN);
    const D CW = dvar<CU_N>(cw, CU_CW), CH = dvar<CU_N>(ch, CU_CH);
    const D UL = dvar<CU_N>(ul, CU_UL), UR = dvar<CU_N>(ur, CU_UR);
    const D sk = HK / WK;
    D dl, dr;
    if (k == 0) {
        dl = T(3) * (dsigmoid(UL) * sk);
    } else {
        const D sp = HP / WP;
        const D m1 = dmin(dabs(sp), dabs(sk));
        const D m2 = STB_LIT(0.5) * ((WK * sp + WP * sk) / (WP + WK));
        dl = dmin(m1, m2) * dsign_sum(sp, sk);
    }
    if (k == K - 1) {
        dr = T(3) * (dsigmoid(UR) * sk);
    } else {
        const D sn = HN / WN;
        const D m1 = dmin(dabs(sk), dabs(sn));
        const D m2 = STB_LIT(0.5) * ((WN * sk + WK * sn) / (WK + WN));
        dr = dmin(m1, m2) * dsign_sum(sk, sn);
    }
    const D a = (dl + dr - T(2) * sk) / (WK * WK);
    const D b = (T(3) * sk - T(2) * dl - dr) / WK;
    const D s = U - CW;
    S = a * s * s * s + b * s * s + dl * s + CH;
    L = dlog(T(3) * (a * s * s) + T(2) * (b * s) + dl);
}

// prm = [uw(K) | uh(K) | left, right] raw; gp receives the gradient wrt those 2K + 2 values.
template <class P, class O = CubDefaultsT<elem_t<P>>>
__device__ __forceinline__ void cubic_element_grad(P prm, P gp, int K, elem_t<P> lower, elem_t<P> upper,
                                                   bool inverse, elem_t<P> x, elem_t<P> g_out, elem_t<P> g_ld,
                                                   elem_t<P>& g_x, const O& o = O()) {
    using T = elem_t<P>;
    const int Pn = 2 * K + 2;
    for (int i = 0; i < Pn; ++i) gp[i] = T(0);
    g_x = g_out;
    if (!(x >= lower && x <= upper)) return;
    OffsetView<P> W{prm, 0}, H{prm, K};
    OffsetView<P> GW{gp, 0}, GH{gp, K};
    const T ul = prm[2 * K], ur = prm[2 * K + 1];
    const T mw = o.min_w(), mh = o.min_h();
    softmax_bins(W, K, mw);
    softmax_bins(H, K, mh);
    const T span = upper - lower;
    const T u = (x - lower) / span;
    T cw, ch;
    int k = cubic_search(W, H, K, inverse, u, cw, ch);
    T ue = u;
    if (inverse) {
        const CubBinT<T> b = cubic_bin(W, H, K, k, cw, ch, ul, ur);
        T ld_own;
        ue = cubic_inverse_in_bin(b, u, ld_own, o);
    }
    const T wp = k > 0 ? W[k - 1] : T(1), hp = k > 0 ? H[k - 1] : T(1);
    const T wn = k < K - 1 ? W[k + 1] : T(1), hn = k < K - 1 ? H[k + 1] : T(1);
    Dual<CU_N, T> S, L;
    cubic_bin_dual(k, K, ue, wp, T(W[k]), wn, hp, T(H[k]), hn, cw, ch, ul, ur, S, L);
    // out = span * S + lower, u = (x - lower) / span; ld = L (same box on both axes)
    T gq[CU_N];
    if (!inverse) {
#pragma unroll
        for (int i = 0; i < CU_N; ++i) gq[i] = g_out * span * S.d[i] + g_ld * L.d[i];
        g_x = gq[CU_U] / span;
    } else {
        const T xo = ue * span + lower;
        const T gl = (xo >= lower && xo <= upper) ? g_ld : T(0);
        // x_out = span * ue + lower;  ue solves S(ue; q) = u;  ld = -L(ue; q)
        const T gu = (g_out * span - gl * L.d[CU_U]) / S.d[CU_U];          // gradient wrt u (input, unit box)
        gq[CU_U] = gu;
#pragma unroll
        for (int i = 1; i < CU_N; ++i) gq[i] = -S.d[i] * gu - gl * L.d[i];
        g_x = gu / span;
    }
    // neighbours / cumulative sums -> normalised sizes
    const T scale_w = T(1) - mw * (T)K, scale_h = T(1) - mh * (T)K;
    T dotw = T(0), doth = T(0);
    for (int i = 0; i < K; ++i) {
        T gwi = (i < k) ? gq[CU_CW] : T(0), ghi = (i < k) ? gq[CU_CH] : T(0);
        if (i == k - 1) { gwi += gq[CU_WP]; ghi += gq[CU_HP]; }
        if (i == k) { gwi += gq[CU_WK]; ghi += gq[CU_HK]; }
        if (i == k + 1) { gwi += gq[CU_WN]; ghi += gq[CU_HN]; }
        GW[i] = gwi;                                  // stash, converted below
        GH[i] = ghi;
        dotw += (W[i] - mw) * gwi;
        doth += (H[i] - mh) * ghi;
    }
    for (int i = 0; i < K; ++i) {
        const T sw = (O::kRuntime && scale_w == T(0)) ? T(0) : (W[i] - mw) / scale_w;
        const T sh = (O::kRuntime && scale_h == T(0)) ? T(0) : (H[i] - mh) / scale_h;
        GW[i] = sw * (scale_w * GW[i] - dotw);
        GH[i] = sh * (scale_h * GH[i] - doth);
    }
    gp[2 * K] = (k == 0) ? gq[CU_UL] : T(0);
    gp[2 * K + 1] = (k == K - 1) ? gq[CU_UR] : T(0);
}

}  // namespace stb
