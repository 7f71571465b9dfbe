// Tile bodies of the CUDA-core layer kernels (generic_layer.cu), generic over the scalar type T:
// the fp32 kernels instantiate them for float (generic_layer.cu), the fp64 kernels for double
// (float64.cu).  The argument blocks keep the C ABI's float pointers; they point to T.
#pragma once
#include "common.cuh"
#include "stb_math.cuh"

namespace stb {

constexpr int kTileRows = 32;
constexpr int kGenWarps = 4;
constexpr int kGenThreads = kTileRows * kGenWarps;
constexpr int kXsStride = kTileRows + 1;
constexpr int kColStride = kGenThreads + 1;    // padded: conflict-free per-thread AND transposed access

struct GenArgs {
    LayerArgs L;
    int direction;
    int ldj_mode;
    int base_log_prob;
    int in_dim;        // conditioner input width (0 when there is no network)
    int buf_rows;      // rows of each ping-pong activation buffer
    int P;             // parameters per transformed dim
    const float* x;
    const float* latent;
    const float* t;
    float* y;
    float* ldj;
    float* ldiag;      // optional [rows, dim] per-dimension log-derivative
    int32_t* bins;     // optional [rows, dim] searched bin per element (pre-filled with -1 by the caller)
    long long rows;
};

// spline_params_per_dim, with the two free boundary derivatives of an rqs layer that asks for them
inline int layer_params_per_dim(const stb_layer* L) {
    const bool free_edge = L->kind == STB_RQS && L->spline.custom && L->spline.free_edge_derivs;
    return spline_params_per_dim(L->kind, L->n_bins) + (free_edge ? 2 : 0);
}

// ints between the tile's transformed-dim list and the T-typed block after it (keeps that block aligned)
template <class T>
__host__ __device__ constexpr int tr_list_ints(int d) {
    return (d + (int)(sizeof(T) / sizeof(int)) - 1) / (int)(sizeof(T) / sizeof(int)) * (int)(sizeof(T) / sizeof(int));
}

// dynamic shared memory of one generic_layer_tile<T>
template <class T>
size_t generic_smem_bytes(const stb_layer* L, int P, int buf_rows, bool ldiag) {
    return sizeof(T) * ((size_t)L->dim * kXsStride + 2 * (size_t)buf_rows * kTileRows + (size_t)P * kColStride +
                        kGenWarps * kTileRows + kTileRows) +
           sizeof(int) * (size_t)tr_list_ints<T>(L->dim) + (ldiag ? sizeof(T) * (size_t)L->dim * kXsStride : 0);
}

// row of the conditioner output holding parameter p of dim j
__device__ __forceinline__ int out_row(int kind, int dim, int P, int j, int p) {
    return (kind == STB_AFFINE || kind == STB_CONT_AFFINE) ? p * dim + j : j * P + p;
}

// acc[i] = sum_k W[rows[i]][k] * in_s[k][lane],  i < n (n <= 8)
template <int N, class T>
__device__ __forceinline__ void dot_rows(const T* __restrict__ W, int in_dim, const int* rows,
                                         int n, const T* in_s, int lane, T* acc) {
    const T* wp[N];
#pragma unroll
    for (int i = 0; i < N; ++i) {
        wp[i] = W + (size_t)rows[i < n ? i : 0] * in_dim;
        acc[i] = T(0);
    }
    if constexpr (std::is_same<T, float>::value) {
        const bool vec = ((in_dim & 3) == 0) && ((reinterpret_cast<uintptr_t>(W) & 15) == 0);
        int k = 0;
        if (vec) {
            for (; k + 4 <= in_dim; k += 4) {
                float a0 = in_s[(k + 0) * kTileRows + lane];
                float a1 = in_s[(k + 1) * kTileRows + lane];
                float a2 = in_s[(k + 2) * kTileRows + lane];
                float a3 = in_s[(k + 3) * kTileRows + lane];
#pragma unroll
                for (int i = 0; i < N; ++i) {
                    float4 w = __ldg(reinterpret_cast<const float4*>(wp[i] + k));
                    acc[i] = fmaf(w.x, a0, acc[i]);
                    acc[i] = fmaf(w.y, a1, acc[i]);
                    acc[i] = fmaf(w.z, a2, acc[i]);
                    acc[i] = fmaf(w.w, a3, acc[i]);
                }
            }
        }
        for (; k < in_dim; ++k) {
            float a = in_s[k * kTileRows + lane];
#pragma unroll
            for (int i = 0; i < N; ++i) acc[i] = fmaf(__ldg(wp[i] + k), a, acc[i]);
        }
    } else {
        for (int k = 0; k < in_dim; ++k) {
            const T a = in_s[k * kTileRows + lane];
#pragma unroll
            for (int i = 0; i < N; ++i) acc[i] = fma(__ldg(wp[i] + k), a, acc[i]);
        }
    }
}

// One tile of the generic layer kernel; O holds the spline constants (stb_math.cuh).  The kernel reads
// threadIdx.x itself: there the compiler knows its range from __launch_bounds__.
template <class T, int KIND, class O>
__device__ __forceinline__ void generic_layer_tile(const GenArgs& A, const O& o, const int tid) {
    extern __shared__ __align__(16) float smem[];
    const stb_layer& L = A.L.get();
    const int d = L.dim;
    const int lane = tid & 31, warp = tid >> 5;
    const long long row0 = (long long)blockIdx.x * kTileRows;
    const int nrows = (int)min((long long)kTileRows, A.rows - row0);
    const int P = A.P;

    T* xs = reinterpret_cast<T*>(smem);                   // [d][33]
    T* bufA = xs + d * kXsStride;                         // [buf_rows][32]
    T* bufB = bufA + A.buf_rows * kTileRows;              // [buf_rows][32]
    T* prm = bufB + A.buf_rows * kTileRows;               // [P][129]
    T* ldj_s = prm + P * kColStride;                      // [4][32]
    T* t_s = ldj_s + kGenWarps * kTileRows;               // [32]
    int* tr_list = reinterpret_cast<int*>(t_s + kTileRows);         // [d]
    T* lds = reinterpret_cast<T*>(tr_list + tr_list_ints<T>(d));    // [d][33], only with ldiag
    __shared__ int n_tr_s;

    // ---- stage the x tile (coalesced) and the list of transformed dims -------------------
    {
        const T* xg = reinterpret_cast<const T*>(A.x) + row0 * d;
        const int n = nrows * d;
        for (int i = tid; i < kTileRows * d; i += kGenThreads) {
            int r = i / d, c = i - r * d;
            xs[c * kXsStride + r] = (i < n) ? xg[i] : T(0);
            if (A.ldiag) lds[c * kXsStride + r] = T(0);
        }
        if (tid < kTileRows) t_s[tid] = (A.t != nullptr && tid < nrows) ? reinterpret_cast<const T*>(A.t)[row0 + tid] : T(0);
        if (warp == 0) {                      // ordered compaction of the transformed dims
            int n_tr = 0;
            for (int j0 = 0; j0 < d; j0 += 32) {
                const int j = j0 + lane;
                const bool tr = (j < d) && (!L.cond_x || L.mask[j] == 0);
                const unsigned b = __ballot_sync(0xffffffffu, tr);
                if (tr) tr_list[n_tr + __popc(b & ((1u << lane) - 1u))] = j;
                n_tr += __popc(b);
            }
            if (lane == 0) n_tr_s = n_tr;
        }
    }
    __syncthreads();
    const int n_tr = n_tr_s;

    // ---- conditioner input tile  [x*mask | latent | t]  -> bufA ------------------------------
    const int nl = L.net.n_linear;
    if (nl > 0) {
        const int xin = L.cond_x ? d : 0;
        for (int i = tid; i < xin * kTileRows; i += kGenThreads) {
            int c = i >> 5, r = i & 31;
            T v = (L.mask[c] != 0 && !L.zero_cond) ? xs[c * kXsStride + r] : T(0);
            bufA[c * kTileRows + r] = v;
        }
        const int ld_ = L.latent_dim;
        if (ld_ > 0) {
            const T* lg = reinterpret_cast<const T*>(A.latent) + row0 * ld_;
            for (int i = tid; i < kTileRows * ld_; i += kGenThreads) {
                int r = i / ld_, c = i - r * ld_;
                bufA[(xin + c) * kTileRows + r] = (r < nrows) ? lg[i] : T(0);
            }
        }
        if (L.time_input && tid < kTileRows) bufA[(xin + ld_) * kTileRows + tid] = t_s[tid];
    }
    __syncthreads();

    // ---- hidden layers ------------------------------------------------------------------------
    T* cur = bufA;
    T* nxt = bufB;
    for (int l = 0; l + 1 < nl; ++l) {
        const int in_dim = L.net.dims[l], out_dim = L.net.dims[l + 1];
        const T* W = reinterpret_cast<const T*>(L.net.W[l]);
        const T* b = reinterpret_cast<const T*>(L.net.b[l]);
        for (int o0 = warp * 8; o0 < out_dim; o0 += kGenWarps * 8) {
            int rows[8];
            const int n = min(8, out_dim - o0);
#pragma unroll
            for (int i = 0; i < 8; ++i) rows[i] = o0 + (i < n ? i : 0);
            T acc[8];
            dot_rows<8>(W, in_dim, rows, n, cur, lane, acc);
#pragma unroll
            for (int i = 0; i < 8; ++i)
                if (i < n) nxt[(o0 + i) * kTileRows + lane] = activate(L.net.activation, acc[i] + __ldg(b + o0 + i));
        }
        __syncthreads();
        T* tmp = cur; cur = nxt; nxt = tmp;
    }

    // ---- last linear + transform, one transformed dim at a time per warp ----------------------
    const bool inverse = (A.direction == STB_INVERSE);
    T ld_acc = T(0);
    SmemCol<T> col{prm + tid, kColStride};
    for (int it = warp; it < n_tr; it += kGenWarps) {
        const int j = tr_list[it];
        if (nl > 0) {
            const int in_dim = L.net.dims[nl - 1];
            const T* W = reinterpret_cast<const T*>(L.net.W[nl - 1]);
            const T* b = reinterpret_cast<const T*>(L.net.b[nl - 1]);
            for (int p0 = 0; p0 < P; p0 += 8) {
                int rows[8];
                const int n = min(8, P - p0);
#pragma unroll
                for (int i = 0; i < 8; ++i) rows[i] = out_row(KIND, d, P, j, p0 + (i < n ? i : 0));
                T acc[8];
                dot_rows<8>(W, in_dim, rows, n, cur, lane, acc);
#pragma unroll
                for (int i = 0; i < 8; ++i)
                    if (i < n) {
                        T v = acc[i] + __ldg(b + rows[i]);
                        if (L.net.final_activation != STB_ACT_NONE) v = activate(L.net.final_activation, v);
                        col[p0 + i] = v;
                    }
            }
        } else if (L.row_out) {
            const bool aff = (KIND == STB_AFFINE || KIND == STB_CONT_AFFINE);
            const size_t width = (size_t)(L.row_compact ? n_tr : d) * P;
            if (!aff) {
                // the P parameters of (row, dim) are contiguous: read row-wise (coalesced), 8 rows in
                // flight, and transpose through the padded column block of this warp
                T* pw = prm + warp * 32;
                const size_t c0 = (size_t)(L.row_compact ? it : j) * P;
                for (int r0 = 0; r0 < kTileRows; r0 += 8) {
                    for (int pb = 0; pb < P; pb += 32) {
                        const int p = pb + lane;
                        T v[8];
#pragma unroll
                        for (int u = 0; u < 8; ++u) {
                            const int r = r0 + u;
                            v[u] = (p < P && r < nrows) ? __ldg(reinterpret_cast<const T*>(L.row_out) + (size_t)(row0 + r) * width + c0 + p) : T(0);
                        }
                        if (p < P) {
#pragma unroll
                            for (int u = 0; u < 8; ++u) pw[p * kColStride + r0 + u] = v[u];
                        }
                    }
                }
                __syncwarp();
            } else {
                const T* ro = reinterpret_cast<const T*>(L.row_out) + (size_t)(row0 + (lane < nrows ? lane : 0)) * width;
                for (int p = 0; p < P; ++p)
                    col[p] = __ldg(ro + (L.row_compact ? p * n_tr + it : out_row(KIND, d, P, j, p)));
            }
        } else {
            for (int p = 0; p < P; ++p) col[p] = __ldg(reinterpret_cast<const T*>(L.const_out) + out_row(KIND, d, P, j, p));
        }
        const T xv = xs[j * kXsStride + lane];
        T out, ld;
        if constexpr (KIND == STB_AFFINE) {
            const T ls = col[0], sh = col[1];
            if (inverse) { out = (xv - sh) * exp_(-ls); ld = -ls; }
            else { out = xv * exp_(ls) + sh; ld = ls; }
        } else if constexpr (KIND == STB_CONT_AFFINE) {
            const T tv = t_s[lane];
            const T tls = __ldg(reinterpret_cast<const T*>(L.time_scale) + j) * tv;
            const T tsh = __ldg(reinterpret_cast<const T*>(L.time_scale) + d + j) * tv;
            const T a = col[0] * tls, sh = col[1] * tsh;
            if (inverse) { out = (xv - sh) * exp_(-a); ld = -a; }
            else { out = xv * exp_(a) + sh; ld = a; }
        } else if constexpr (KIND == STB_RQS) {
            const bool box = L.has_box != 0;
            int kb;
            rqs_element(col, L.n_bins, box ? L.left : L.lower, box ? L.right : L.upper,
                        box ? L.bottom : L.lower, box ? L.top : L.upper, inverse,
                        L.inverse_ldj_own != 0, xv, out, ld, &kb, o);
            if (A.bins && lane < nrows) A.bins[(row0 + lane) * d + j] = kb;
        } else if constexpr (KIND == STB_CUBIC) {
            int kb;
            cubic_element(col, L.n_bins, L.lower, L.upper, inverse, L.inverse_ldj_own != 0, xv, out, ld, &kb, o);
            if (A.bins && lane < nrows) A.bins[(row0 + lane) * d + j] = kb;
        }
        xs[j * kXsStride + lane] = out;
        if (A.ldiag) lds[j * kXsStride + lane] = ld;
        ld_acc += ld;
    }
    __syncthreads();

    // ---- UnitNormal log-density of the output row (dist/normal.py:37) --------------------------
    if (A.base_log_prob) {
        for (int c = warp; c < d; c += kGenWarps) {
            T v = xs[c * kXsStride + lane];
            ld_acc += STB_LIT(-0.5) * v * v - STB_LIT(0.91893853320467274178);
        }
    }

    // ---- per-row log|det J|: reduce over warps ----------------------------------------------------
    if (A.ldj_mode != STB_LDJ_NONE) {
        ldj_s[warp * kTileRows + lane] = ld_acc;
        __syncthreads();
        if (warp == 0 && lane < nrows) {
            T v = T(0);
#pragma unroll
            for (int w = 0; w < kGenWarps; ++w) v += ldj_s[w * kTileRows + lane];
            T* dst = reinterpret_cast<T*>(A.ldj) + row0 + lane;
            *dst = (A.ldj_mode == STB_LDJ_ADD) ? (*dst + v) : v;
        }
    }

    // ---- y tile out (coalesced) --------------------------------------------------------------------
    {
        T* yg = reinterpret_cast<T*>(A.y) + row0 * d;
        const int n = nrows * d;
        for (int i = tid; i < n; i += kGenThreads) {
            int r = i / d, c = i - r * d;
            yg[i] = xs[c * kXsStride + r];
        }
        if (A.ldiag) {
            T* lg = reinterpret_cast<T*>(A.ldiag) + row0 * d;
            for (int i = tid; i < n; i += kGenThreads) {
                int r = i / d, c = i - r * d;
                lg[i] = lds[c * kXsStride + r];
            }
        }
    }
}

// Parameter-free layers: one warp per row, lanes over dims (coalesced), shuffle-reduced log-det.
//   STB_PERMUTE  y[i] = x[perm[i]] (inverse: perm_inv), log-det 0            flows/permute.py:47-82
//   STB_SIGMOID  y = clamp(sigmoid(x), tiny, 1 - eps); log-diag(x) = -softplus(-x) - softplus(x);
//                inverse x = log(y) - log1p(-y) on the clamped y              flows/sigmoid.py:9-41
//                (tiny / eps: torch.finfo of T)
//   STB_LOGIT    the same maps with the roles swapped; its log-diag is evaluated at the LOGIT-side
//                value, as sigmoid.py:44-56 does
// Log-det conventions are the inherited ones (flow.py:35-47): inverse = -(forward log-det at the
// recovered / supplied point).
template <class T>
__device__ __forceinline__ void pointwise_row(int kind, int direction, const T* __restrict__ x, T* __restrict__ y,
                                              const int32_t* __restrict__ perm, T* __restrict__ ldj, int ldj_mode,
                                              int base_log_prob, int d, long long rows) {
    const long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (row >= rows) return;
    const bool f32 = std::is_same<T, float>::value;
    const T tiny = f32 ? T(1.17549435e-38f) : T(2.2250738585072014e-308);
    const T one_m_eps = f32 ? T(1.f - 1.1920929e-07f) : T(1) - T(2.220446049250313e-16);
    const bool to_unit = (kind == STB_SIGMOID) == (direction == STB_FORWARD);   // R -> (0,1) ?
    T ld = T(0), lp = T(0);
    if (kind == STB_PERMUTE && d <= 32 * 8) {
        // the whole row is gathered into registers before the first write: safe when y aliases x
        T v[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) { const int c = lane + 32 * k; v[k] = (c < d) ? x[row * d + perm[c]] : T(0); }
        __syncwarp();
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const int c = lane + 32 * k;
            if (c < d) { y[row * d + c] = v[k]; if (base_log_prob) lp += STB_LIT(-0.5) * v[k] * v[k] - STB_LIT(0.91893853320467274178); }
        }
    } else
    for (int c = lane; c < d; c += 32) {
        T v, out;
        if (kind == STB_PERMUTE) {
            out = x[row * d + perm[c]];
        } else {
            v = x[row * d + c];
            T u;                                           // the value on the unbounded (logit) side
            if (to_unit) {
                out = fmin_(fmax_(sigmoid_f(v), tiny), one_m_eps);
                u = v;
            } else {
                const T yc = fmin_(fmax_(v, tiny), one_m_eps);
                out = log_(yc) - log1p_(-yc);
                u = out;
            }
            const T ldiag = -softplus_f(-u) - softplus_f(u);          // log sigmoid'(u)
            // forward sigmoid: +ldiag; inverse sigmoid: -ldiag; logit: the opposite signs
            ld += to_unit ? ldiag : -ldiag;
        }
        if (base_log_prob) lp += STB_LIT(-0.5) * out * out - STB_LIT(0.91893853320467274178);
        y[row * d + c] = out;
    }
    if (ldj_mode != STB_LDJ_NONE) {
        T s = ld + lp;
#pragma unroll
        for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if (lane == 0) ldj[row] = (ldj_mode == STB_LDJ_ADD) ? ldj[row] + s : s;
    }
}

// fp64 launches (float64.cu): the double instantiations of the kernels above
int generic_layer_launch_f64(const stb_layer* L, const GenArgs& A, size_t smem, unsigned tiles, cudaStream_t stream);
int pointwise_launch_f64(int kind, int direction, const float* x, float* y, const int32_t* perm, float* ldj,
                         int ldj_mode, int base_log_prob, int d, long long rows, unsigned blocks, int threads,
                         cudaStream_t stream);

}  // namespace stb
