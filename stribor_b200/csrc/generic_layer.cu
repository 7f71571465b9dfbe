// Generic fused coupling-layer kernel (CUDA cores, shared-memory staged FMA).
//
// One CTA = one tile of 32 rows, 4 warps.  Lane = row; a warp owns a subset of the
// transformed dims (and of every hidden layer's output neurons), so weight reads are
// warp-uniform broadcasts and activations are read conflict-free from [k][row] tiles.
// Per layer the tile makes ONE HBM round trip: x tile in -> (conditioner MLP in smem/regs ->
// transform in registers -> per-row log|det J| reduced across warps) -> y tile out.
//
// This is the path for arbitrary configurations (any dim, mask, n_bins, hidden widths,
// activation, latent / time inputs, stand-alone Affine / Spline).  The tcgen05 kernel in
// tc_layer.cu takes over when the conditioner is a real dense contraction.
//
// Reference behaviour restated here: flows/coupling.py:53-95,188-213, flows/affine.py:59-109,
// flows/spline.py:76-105, net/mlp.py:46-58, net/time_net.py:24-25, dist/normal.py:37.
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

// row of the conditioner output holding parameter p of dim j
__device__ __forceinline__ int out_row(int kind, int dim, int P, int j, int p) {
    return (kind == STB_AFFINE || kind == STB_CONT_AFFINE) ? p * dim + j : j * P + p;
}

// acc[i] = sum_k W[rows[i]][k] * in_s[k][lane],  i < n (n <= 8)
template <int N>
__device__ __forceinline__ void dot_rows(const float* __restrict__ W, int in_dim, const int* rows,
                                         int n, const float* in_s, int lane, float* acc) {
    const float* wp[N];
#pragma unroll
    for (int i = 0; i < N; ++i) {
        wp[i] = W + (size_t)rows[i < n ? i : 0] * in_dim;
        acc[i] = 0.f;
    }
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
}

// One tile of generic_layer_kernel; O holds the spline constants (stb_math.cuh).  The kernel reads
// threadIdx.x itself: there the compiler knows its range from __launch_bounds__.
template <int KIND, class O>
__device__ __forceinline__ void generic_layer_tile(const GenArgs& A, const O& o, const int tid) {
    extern __shared__ __align__(16) float smem[];
    const stb_layer& L = A.L.get();
    const int d = L.dim;
    const int lane = tid & 31, warp = tid >> 5;
    const long long row0 = (long long)blockIdx.x * kTileRows;
    const int nrows = (int)min((long long)kTileRows, A.rows - row0);
    const int P = A.P;

    float* xs = smem;                                     // [d][33]
    float* bufA = xs + d * kXsStride;                     // [buf_rows][32]
    float* bufB = bufA + A.buf_rows * kTileRows;          // [buf_rows][32]
    float* prm = bufB + A.buf_rows * kTileRows;           // [P][129]
    float* ldj_s = prm + P * kColStride;                  // [4][32]
    float* t_s = ldj_s + kGenWarps * kTileRows;           // [32]
    int* tr_list = reinterpret_cast<int*>(t_s + kTileRows);   // [d]
    float* lds = reinterpret_cast<float*>(tr_list + d);       // [d][33], only with ldiag
    __shared__ int n_tr_s;

    // ---- stage the x tile (coalesced) and the list of transformed dims -------------------
    {
        const float* xg = A.x + row0 * d;
        const int n = nrows * d;
        for (int i = tid; i < kTileRows * d; i += kGenThreads) {
            int r = i / d, c = i - r * d;
            xs[c * kXsStride + r] = (i < n) ? xg[i] : 0.f;
            if (A.ldiag) lds[c * kXsStride + r] = 0.f;
        }
        if (tid < kTileRows) t_s[tid] = (A.t != nullptr && tid < nrows) ? A.t[row0 + tid] : 0.f;
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
            float v = (L.mask[c] != 0 && !L.zero_cond) ? xs[c * kXsStride + r] : 0.f;
            bufA[c * kTileRows + r] = v;
        }
        const int ld_ = L.latent_dim;
        if (ld_ > 0) {
            const float* lg = A.latent + row0 * ld_;
            for (int i = tid; i < kTileRows * ld_; i += kGenThreads) {
                int r = i / ld_, c = i - r * ld_;
                bufA[(xin + c) * kTileRows + r] = (r < nrows) ? lg[i] : 0.f;
            }
        }
        if (L.time_input && tid < kTileRows) bufA[(xin + ld_) * kTileRows + tid] = t_s[tid];
    }
    __syncthreads();

    // ---- hidden layers ------------------------------------------------------------------------
    float* cur = bufA;
    float* nxt = bufB;
    for (int l = 0; l + 1 < nl; ++l) {
        const int in_dim = L.net.dims[l], out_dim = L.net.dims[l + 1];
        const float* W = L.net.W[l];
        const float* b = L.net.b[l];
        for (int o0 = warp * 8; o0 < out_dim; o0 += kGenWarps * 8) {
            int rows[8];
            const int n = min(8, out_dim - o0);
#pragma unroll
            for (int i = 0; i < 8; ++i) rows[i] = o0 + (i < n ? i : 0);
            float acc[8];
            dot_rows<8>(W, in_dim, rows, n, cur, lane, acc);
#pragma unroll
            for (int i = 0; i < 8; ++i)
                if (i < n) nxt[(o0 + i) * kTileRows + lane] = activate(L.net.activation, acc[i] + __ldg(b + o0 + i));
        }
        __syncthreads();
        float* tmp = cur; cur = nxt; nxt = tmp;
    }

    // ---- last linear + transform, one transformed dim at a time per warp ----------------------
    const bool inverse = (A.direction == STB_INVERSE);
    float ld_acc = 0.f;
    SmemCol col{prm + tid, kColStride};
    for (int it = warp; it < n_tr; it += kGenWarps) {
        const int j = tr_list[it];
        if (nl > 0) {
            const int in_dim = L.net.dims[nl - 1];
            const float* W = L.net.W[nl - 1];
            const float* b = L.net.b[nl - 1];
            for (int p0 = 0; p0 < P; p0 += 8) {
                int rows[8];
                const int n = min(8, P - p0);
#pragma unroll
                for (int i = 0; i < 8; ++i) rows[i] = out_row(KIND, d, P, j, p0 + (i < n ? i : 0));
                float acc[8];
                dot_rows<8>(W, in_dim, rows, n, cur, lane, acc);
#pragma unroll
                for (int i = 0; i < 8; ++i)
                    if (i < n) {
                        float v = acc[i] + __ldg(b + rows[i]);
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
                float* pw = prm + warp * 32;
                const size_t c0 = (size_t)(L.row_compact ? it : j) * P;
                for (int r0 = 0; r0 < kTileRows; r0 += 8) {
                    for (int pb = 0; pb < P; pb += 32) {
                        const int p = pb + lane;
                        float v[8];
#pragma unroll
                        for (int u = 0; u < 8; ++u) {
                            const int r = r0 + u;
                            v[u] = (p < P && r < nrows) ? __ldg(L.row_out + (size_t)(row0 + r) * width + c0 + p) : 0.f;
                        }
                        if (p < P) {
#pragma unroll
                            for (int u = 0; u < 8; ++u) pw[p * kColStride + r0 + u] = v[u];
                        }
                    }
                }
                __syncwarp();
            } else {
                const float* ro = L.row_out + (size_t)(row0 + (lane < nrows ? lane : 0)) * width;
                for (int p = 0; p < P; ++p)
                    col[p] = __ldg(ro + (L.row_compact ? p * n_tr + it : out_row(KIND, d, P, j, p)));
            }
        } else {
            for (int p = 0; p < P; ++p) col[p] = __ldg(L.const_out + out_row(KIND, d, P, j, p));
        }
        const float xv = xs[j * kXsStride + lane];
        float out, ld;
        if constexpr (KIND == STB_AFFINE) {
            const float ls = col[0], sh = col[1];
            if (inverse) { out = (xv - sh) * expf(-ls); ld = -ls; }
            else { out = xv * expf(ls) + sh; ld = ls; }
        } else if constexpr (KIND == STB_CONT_AFFINE) {
            const float tv = t_s[lane];
            const float tls = __ldg(L.time_scale + j) * tv;
            const float tsh = __ldg(L.time_scale + d + j) * tv;
            const float a = col[0] * tls, sh = col[1] * tsh;
            if (inverse) { out = (xv - sh) * expf(-a); ld = -a; }
            else { out = xv * expf(a) + sh; ld = a; }
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
            float v = xs[c * kXsStride + lane];
            ld_acc += -0.5f * v * v - 0.91893853320467274178f;
        }
    }

    // ---- per-row log|det J|: reduce over warps ----------------------------------------------------
    if (A.ldj_mode != STB_LDJ_NONE) {
        ldj_s[warp * kTileRows + lane] = ld_acc;
        __syncthreads();
        if (warp == 0 && lane < nrows) {
            float v = 0.f;
#pragma unroll
            for (int w = 0; w < kGenWarps; ++w) v += ldj_s[w * kTileRows + lane];
            float* dst = A.ldj + row0 + lane;
            *dst = (A.ldj_mode == STB_LDJ_ADD) ? (*dst + v) : v;
        }
    }

    // ---- y tile out (coalesced) --------------------------------------------------------------------
    {
        float* yg = A.y + row0 * d;
        const int n = nrows * d;
        for (int i = tid; i < n; i += kGenThreads) {
            int r = i / d, c = i - r * d;
            yg[i] = xs[c * kXsStride + r];
        }
        if (A.ldiag) {
            float* lg = A.ldiag + row0 * d;
            for (int i = tid; i < n; i += kGenThreads) {
                int r = i / d, c = i - r * d;
                lg[i] = lds[c * kXsStride + r];
            }
        }
    }
}

template <int KIND>
__global__ void __launch_bounds__(kGenThreads) generic_layer_kernel(const GenArgs A) {
    generic_layer_tile<KIND>(A, DefaultOpts<KIND>(), threadIdx.x);
}

// splines with the functional API's non-default constants (stb_layer.spline.custom != 0)
template <int KIND>
__global__ void __launch_bounds__(kGenThreads) generic_layer_opts_kernel(const GenArgs A, const SplineOpts o) {
    generic_layer_tile<KIND>(A, o, threadIdx.x);
}

__global__ void unit_normal_kernel(const float* __restrict__ x, float* __restrict__ lp, int accumulate,
                                   int d, long long rows) {
    const long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (row >= rows) return;
    float s = 0.f;
    for (int c = lane; c < d; c += 32) {
        float v = x[row * d + c];
        s += -0.5f * v * v - 0.91893853320467274178f;
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) lp[row] = accumulate ? lp[row] + s : s;
}

// Parameter-free layers: one warp per row, lanes over dims (coalesced), shuffle-reduced log-det.
//   STB_PERMUTE  y[i] = x[perm[i]] (inverse: perm_inv), log-det 0            flows/permute.py:47-82
//   STB_SIGMOID  y = clamp(sigmoid(x), tiny, 1 - eps); log-diag(x) = -softplus(-x) - softplus(x);
//                inverse x = log(y) - log1p(-y) on the clamped y              flows/sigmoid.py:9-41
//   STB_LOGIT    the same maps with the roles swapped; its log-diag is evaluated at the LOGIT-side
//                value, as sigmoid.py:44-56 does
// Log-det conventions are the inherited ones (flow.py:35-47): inverse = -(forward log-det at the
// recovered / supplied point).
__global__ void pointwise_kernel(int kind, int direction, const float* __restrict__ x, float* __restrict__ y,
                                 const int32_t* __restrict__ perm, float* __restrict__ ldj, int ldj_mode,
                                 int base_log_prob, int d, long long rows) {
    const long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (row >= rows) return;
    const float tiny = 1.17549435e-38f, one_m_eps = 1.f - 1.1920929e-07f;
    const bool to_unit = (kind == STB_SIGMOID) == (direction == STB_FORWARD);   // R -> (0,1) ?
    float ld = 0.f, lp = 0.f;
    if (kind == STB_PERMUTE && d <= 32 * 8) {
        // the whole row is gathered into registers before the first write: safe when y aliases x
        float v[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) { const int c = lane + 32 * k; v[k] = (c < d) ? x[row * d + perm[c]] : 0.f; }
        __syncwarp();
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const int c = lane + 32 * k;
            if (c < d) { y[row * d + c] = v[k]; if (base_log_prob) lp += -0.5f * v[k] * v[k] - 0.91893853320467274178f; }
        }
    } else
    for (int c = lane; c < d; c += 32) {
        float v, out;
        if (kind == STB_PERMUTE) {
            out = x[row * d + perm[c]];
        } else {
            v = x[row * d + c];
            float u;                                       // the value on the unbounded (logit) side
            if (to_unit) {
                out = fminf(fmaxf(sigmoid_f(v), tiny), one_m_eps);
                u = v;
            } else {
                const float yc = fminf(fmaxf(v, tiny), one_m_eps);
                out = logf(yc) - log1pf(-yc);
                u = out;
            }
            const float ldiag = -softplus_f(-u) - softplus_f(u);      // log sigmoid'(u)
            // forward sigmoid: +ldiag; inverse sigmoid: -ldiag; logit: the opposite signs
            ld += to_unit ? ldiag : -ldiag;
        }
        if (base_log_prob) lp += -0.5f * out * out - 0.91893853320467274178f;
        y[row * d + c] = out;
    }
    if (ldj_mode != STB_LDJ_NONE) {
        float s = ld + lp;
#pragma unroll
        for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if (lane == 0) ldj[row] = (ldj_mode == STB_LDJ_ADD) ? ldj[row] + s : s;
    }
}

int pointwise_layer_apply(const stb_layer* L, int direction, const float* x, float* y, float* ldj, int ldj_mode,
                          int base_log_prob, int64_t rows, cudaStream_t stream) {
    if (x == y && L->kind == STB_PERMUTE && L->dim > 32 * 8)
        return set_error(STB_EINVAL, "a permutation of more than 256 dims cannot run in place");
    const int32_t* perm = nullptr;
    if (L->kind == STB_PERMUTE) {
        perm = (direction == STB_FORWARD) ? L->perm : L->perm_inv;
        if (!perm) return set_error(STB_EINVAL, "permutation layer without index arrays");
    }
    const int wpb = 8;
    const long long blocks = (rows + wpb - 1) / wpb;
    pointwise_kernel<<<(unsigned)blocks, wpb * 32, 0, stream>>>(L->kind, direction, x, y, perm, ldj,
                                                               ldj ? ldj_mode : STB_LDJ_NONE, base_log_prob, L->dim, rows);
    count_launch();
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return set_error(STB_ECUDA, "pointwise_kernel launch: %s", cudaGetErrorString(e));
    return STB_OK;
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
int validate_layer(const stb_layer* L) {
    if (!L) return set_error(STB_EINVAL, "layer is NULL");
    if (L->kind < STB_AFFINE || L->kind > STB_LOGIT) return set_error(STB_EINVAL, "unknown transform kind %d", L->kind);
    if (L->dim < 1) return set_error(STB_EINVAL, "dim must be >= 1");
    if (L->kind >= STB_PERMUTE) return STB_OK;
    if (L->cond_x && !L->mask) return set_error(STB_EINVAL, "coupling layer needs a mask");
    const stb_mlp& N = L->net;
    if (N.n_linear < 0 || N.n_linear > STB_MAX_LINEAR) return set_error(STB_EINVAL, "n_linear %d out of range", N.n_linear);
    const int P = layer_params_per_dim(L);
    if (L->kind == STB_RQS || L->kind == STB_CUBIC) {
        if (L->n_bins < 1) return set_error(STB_EINVAL, "n_bins must be >= 1");
        // rational_quadratic_spline.py:96-99 / cubic_spline.py:94-97
        const stb_spline_opts& so = L->spline;
        if (!so.custom) {
            const float mn = L->kind == STB_RQS ? 1e-3f : 1e-2f;
            if (mn * L->n_bins > 1.0f) return set_error(STB_EINVAL, "Minimal bin width too large for the number of bins");
        } else {
            const bool rqs = L->kind == STB_RQS;
            const bool finite = isfinite(so.min_bin_width) && isfinite(so.min_bin_height) &&
                                (rqs ? isfinite(so.min_derivative) : isfinite(so.cub_eps) && isfinite(so.cub_quad_threshold));
            if (!finite) return set_error(STB_EINVAL, "spline options must be finite");
            if (so.min_bin_width * L->n_bins > 1.0f) return set_error(STB_EINVAL, "Minimal bin width too large for the number of bins");
            if (so.min_bin_height * L->n_bins > 1.0f) return set_error(STB_EINVAL, "Minimal bin height too large for the number of bins");
            if (rqs && so.min_derivative < 0.f) return set_error(STB_EINVAL, "min_derivative must be >= 0");
        }
        if (L->has_box) {
            if (L->kind != STB_RQS) return set_error(STB_EINVAL, "separate domain/codomain boxes are rqs-only");
            if (!(L->right > L->left) || !(L->top > L->bottom)) return set_error(STB_EINVAL, "empty spline box");
        } else if (!(L->upper > L->lower)) {
            return set_error(STB_EINVAL, "spline box must have upper > lower");
        }
    }
    if (L->kind == STB_CONT_AFFINE && !L->time_scale) return set_error(STB_EINVAL, "cont-affine needs time_scale");
    if (N.n_linear == 0) {
        if (!L->const_out && !L->row_out) return set_error(STB_EINVAL, "no network and no const_out / row_out");
    } else {
        const int in_dim = (L->cond_x ? L->dim : 0) + L->latent_dim + (L->time_input ? 1 : 0);
        if (N.dims[0] != in_dim) return set_error(STB_EINVAL, "network input width %d != %d", N.dims[0], in_dim);
        if (N.dims[N.n_linear] != L->dim * P) return set_error(STB_EINVAL, "network output width %d != dim*P = %d", N.dims[N.n_linear], L->dim * P);
        for (int i = 0; i < N.n_linear; ++i)
            if (!N.W[i] || !N.b[i] || N.dims[i] < 1) return set_error(STB_EINVAL, "bad linear layer %d", i);
    }
    return STB_OK;
}

int generic_layer_apply(const stb_layer* L, int direction, const float* x, const float* latent,
                        const float* t, float* y, float* ldj, int ldj_mode, int base_log_prob,
                        float* ldiag, int64_t rows, cudaStream_t stream, int32_t* bins) {
    GenArgs A;
    A.L.set(L);
    A.direction = direction;
    A.ldj_mode = ldj ? ldj_mode : STB_LDJ_NONE;
    A.base_log_prob = base_log_prob;
    A.P = layer_params_per_dim(L);
    A.in_dim = L->net.n_linear > 0 ? L->net.dims[0] : 0;
    int buf_rows = 1;
    for (int i = 0; i < L->net.n_linear; ++i) buf_rows = max(buf_rows, L->net.dims[i]);
    A.buf_rows = buf_rows;
    A.x = x; A.latent = latent; A.t = t; A.y = y; A.ldj = ldj; A.ldiag = ldiag; A.bins = bins; A.rows = rows;

    size_t smem = sizeof(float) * ((size_t)L->dim * kXsStride + 2 * (size_t)buf_rows * kTileRows +
                                   (size_t)A.P * kColStride + kGenWarps * kTileRows + kTileRows) +
                  sizeof(int) * (size_t)L->dim + (ldiag ? sizeof(float) * (size_t)L->dim * kXsStride : 0);
    if (smem > 227 * 1024) return set_error(STB_ENOTSUP, "layer needs %zu B of shared memory per tile (> 227 KB)", smem);

    const bool custom = L->spline.custom && (L->kind == STB_RQS || L->kind == STB_CUBIC);
    void (*kern)(GenArgs) = nullptr;
    void (*kern_opts)(GenArgs, SplineOpts) = nullptr;
    switch (L->kind) {
        case STB_AFFINE: kern = generic_layer_kernel<STB_AFFINE>; break;
        case STB_RQS: kern = generic_layer_kernel<STB_RQS>; kern_opts = generic_layer_opts_kernel<STB_RQS>; break;
        case STB_CUBIC: kern = generic_layer_kernel<STB_CUBIC>; kern_opts = generic_layer_opts_kernel<STB_CUBIC>; break;
        default: kern = generic_layer_kernel<STB_CONT_AFFINE>; break;
    }
    if (smem > 48 * 1024) {
        cudaError_t e = custom ? cudaFuncSetAttribute(kern_opts, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)
                               : cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return set_error(STB_ECUDA, "cudaFuncSetAttribute: %s", cudaGetErrorString(e));
    }
    const long long tiles = (rows + kTileRows - 1) / kTileRows;
    if (tiles > 0x7fffffffLL) return set_error(STB_EINVAL, "too many rows");
    if (custom) kern_opts<<<(unsigned)tiles, kGenThreads, smem, stream>>>(A, make_spline_opts(L->spline));
    else kern<<<(unsigned)tiles, kGenThreads, smem, stream>>>(A);
    count_launch();
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return set_error(STB_ECUDA, "generic_layer_kernel launch: %s", cudaGetErrorString(e));
    return STB_OK;
}

int unit_normal_apply(const float* x, float* lp, int accumulate, int dim, int64_t rows, cudaStream_t stream) {
    if (rows == 0) return STB_OK;
    const int wpb = 8;
    const long long blocks = (rows + wpb - 1) / wpb;
    unit_normal_kernel<<<(unsigned)blocks, wpb * 32, 0, stream>>>(x, lp, accumulate, dim, rows);
    count_launch();
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return set_error(STB_ECUDA, "unit_normal_kernel launch: %s", cudaGetErrorString(e));
    return STB_OK;
}

}  // namespace stb
