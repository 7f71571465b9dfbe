// Backward of the element-wise transforms (affine / rational-quadratic / cubic) of a layer whose
// network output is supplied per row (row_out) or as a constant (const_out): what autograd derives
// for flows/affine.py:97-109, util/rational_quadratic_spline.py and util/cubic_spline.py.
//
// Same tiling as generic_layer.cu: one CTA = 32 rows, lane = row, a warp owns a subset of the
// transformed dims.  Parameters and their gradients live in padded shared-memory columns so both
// the per-thread access ([p][thread]) and the transposed, coalesced global access ([row][p]) are
// bank-conflict free.
#include "common.cuh"
#include "stb_grad.cuh"

namespace stb {

constexpr int kBTileRows = 32;
constexpr int kBWarps = 4;
constexpr int kBThreads = kBTileRows * kBWarps;
constexpr int kBColStride = kBThreads + 1;
constexpr int kBXsStride = kBTileRows + 1;

struct BwdArgs {
    LayerArgs L;
    int direction;
    int P, width, n_tr;
    const float* x;
    const float* g_out;
    const float* g_ldj;
    const float* g_ldiag;    // optional [rows, dim]: gradient wrt the per-dimension log-derivative (stb_layer_apply_diag)
    float* g_x;
    float* g_row;
    long long rows;
};

// index of parameter p of the it-th transformed dim (original dim j) in the network output
__device__ __forceinline__ int bwd_col(const stb_layer& L, int P, int n_tr, int it, int j, int p) {
    const bool aff = (L.kind == STB_AFFINE || L.kind == STB_CONT_AFFINE);
    if (L.row_compact) return aff ? p * n_tr + it : it * P + p;
    return aff ? p * L.dim + j : j * P + p;
}

// One tile of elementwise_backward_kernel; O holds the spline constants (stb_math.cuh).  The kernel
// reads threadIdx.x itself: there the compiler knows its range from __launch_bounds__.
template <int KIND, class O>
__device__ __forceinline__ void elementwise_backward_tile(const BwdArgs& A, const O& o, const int tid) {
    extern __shared__ __align__(16) float smem[];
    const stb_layer& L = A.L.get();
    const int d = L.dim, P = A.P;
    const int lane = tid & 31, warp = tid >> 5;
    const long long row0 = (long long)blockIdx.x * kBTileRows;
    const int nrows = (int)min((long long)kBTileRows, A.rows - row0);

    float* xs = smem;                                  // [d][33]   layer input
    float* gs = xs + d * kBXsStride;                   // [d][33]   g_out -> g_x
    float* prm = gs + d * kBXsStride;                  // [P][129]
    float* gpr = prm + P * kBColStride;                // [P][129]
    int* tr_list = reinterpret_cast<int*>(gpr + P * kBColStride);
    __shared__ int n_tr_s;

    {
        const float* xg = A.x + row0 * d;
        const float* gg = A.g_out + row0 * d;
        const int n = nrows * d;
        for (int i = tid; i < kBTileRows * d; i += kBThreads) {
            const int r = i / d, c = i - r * d;
            xs[c * kBXsStride + r] = (i < n) ? xg[i] : 0.f;
            gs[c * kBXsStride + r] = (i < n) ? gg[i] : 0.f;
        }
        if (warp == 0) {
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
    const bool inverse = (A.direction == STB_INVERSE);
    const float g_ld_row = (A.g_ldj != nullptr && lane < nrows) ? A.g_ldj[row0 + lane] : 0.f;
    SmemCol col{prm + tid, kBColStride};
    SmemCol gcol{gpr + tid, kBColStride};
    float* pw = prm + warp * 32;                       // this warp's 32 columns
    float* gw = gpr + warp * 32;

    for (int it = warp; it < n_tr; it += kBWarps) {
        const int j = tr_list[it];
        // ---- parameters of (rows of the tile, dim j) -> columns ------------------------------------
        if (L.row_out) {
            const bool contiguous = (KIND == STB_RQS || KIND == STB_CUBIC);
            if (contiguous) {                          // P consecutive values per row: coalesced rows
                const int c0 = bwd_col(L, P, n_tr, it, j, 0);
                // 8 rows per batch, all loads issued before the first store: the loop is otherwise a
                // chain of dependent L2 / HBM round trips (it was 45 % of a training step)
                for (int r0 = 0; r0 < kBTileRows; r0 += 8) {
                    for (int pb = 0; pb < P; pb += 32) {
                        const int p = pb + lane;
                        float v[8];
#pragma unroll
                        for (int u = 0; u < 8; ++u) {
                            const int r = r0 + u;
                            v[u] = (p < P && r < nrows) ? __ldg(L.row_out + (size_t)(row0 + r) * A.width + c0 + p) : 0.f;
                        }
                        if (p < P) {
#pragma unroll
                            for (int u = 0; u < 8; ++u) pw[p * kBColStride + r0 + u] = v[u];
                        }
                    }
                }
            } else {
                for (int p = 0; p < P; ++p)
                    col[p] = (lane < nrows) ? __ldg(L.row_out + (size_t)(row0 + lane) * A.width + bwd_col(L, P, n_tr, it, j, p)) : 0.f;
            }
        } else {
            for (int p = 0; p < P; ++p) col[p] = __ldg(L.const_out + bwd_col(L, P, n_tr, it, j, p));
        }
        __syncwarp();
        // ---- element gradient -------------------------------------------------------------------------
        const float xv = xs[j * kBXsStride + lane];
        const float go = gs[j * kBXsStride + lane];
        float g_ld = g_ld_row;
        if (A.g_ldiag != nullptr && lane < nrows) g_ld += A.g_ldiag[(row0 + lane) * d + j];
        float gx;
        if constexpr (KIND == STB_AFFINE) {
            const float ls = col[0], sh = col[1];
            if (inverse) {
                const float e = expf(-ls), out = (xv - sh) * e;
                gx = go * e; gcol[1] = -go * e; gcol[0] = -go * out - g_ld;
            } else {
                const float e = expf(ls);
                gx = go * e; gcol[1] = go; gcol[0] = go * xv * e + g_ld;
            }
        } else if constexpr (KIND == STB_RQS) {
            const bool box = L.has_box != 0;
            rqs_element_grad(col, gcol, L.n_bins, box ? L.left : L.lower, box ? L.right : L.upper,
                             box ? L.bottom : L.lower, box ? L.top : L.upper, inverse, xv, go, g_ld, gx, o);
        } else {
            cubic_element_grad(col, gcol, L.n_bins, L.lower, L.upper, inverse, xv, go, g_ld, gx, o);
        }
        gs[j * kBXsStride + lane] = gx;
        __syncwarp();
        // ---- parameter gradients out (per row) ------------------------------------------------------
        if (A.g_row) {
            if (KIND == STB_RQS || KIND == STB_CUBIC) {
                const int c0 = bwd_col(L, P, n_tr, it, j, 0);
                for (int r = 0; r < nrows; ++r) {
                    float* dst = A.g_row + (size_t)(row0 + r) * A.width + c0;
                    for (int p = lane; p < P; p += 32) dst[p] = gw[p * kBColStride + r];
                }
            } else if (lane < nrows) {
                for (int p = 0; p < P; ++p)
                    A.g_row[(size_t)(row0 + lane) * A.width + bwd_col(L, P, n_tr, it, j, p)] = gcol[p];
            }
        }
        __syncwarp();
    }
    __syncthreads();
    {
        float* gx = A.g_x + row0 * d;
        const int n = nrows * d;
        for (int i = tid; i < n; i += kBThreads) {
            const int r = i / d, c = i - r * d;
            gx[i] = gs[c * kBXsStride + r];
        }
    }
}

template <int KIND>
__global__ void __launch_bounds__(kBThreads) elementwise_backward_kernel(const BwdArgs A) {
    elementwise_backward_tile<KIND>(A, DefaultOpts<KIND>(), threadIdx.x);
}

// splines with the functional API's non-default constants (stb_layer.spline.custom != 0)
template <int KIND>
__global__ void __launch_bounds__(kBThreads) elementwise_backward_opts_kernel(const BwdArgs A, const SplineOpts o) {
    elementwise_backward_tile<KIND>(A, o, threadIdx.x);
}

// n_linear > 0 on the tensor-core path: the workspace receives the conditioner's hidden activations,
// augmented [rows, 72] = h(64) | 1 | 0 x 7
uint64_t layer_backward_workspace_bytes(const stb_layer* L, int64_t rows) {
    if (L->net.n_linear > 0 && tcw_backward_supported(L))
        return tcw_train_workspace_floats(L, rows > 0 ? rows : 0) * sizeof(float);
    return 0;
}

int layer_backward(const stb_layer* L, int direction, const float* x, const float* latent, const float* t,
                   const float* g_out, const float* g_ldj, float* g_x, float* g_latent, float* g_t,
                   const stb_layer_grads* grads, void* workspace, int64_t rows, cudaStream_t stream,
                   const float* g_ldiag) {
    (void)latent; (void)t; (void)g_latent; (void)g_t;
    if (L->net.n_linear > 0) {
        if (g_ldiag) return set_error(STB_ENOTSUP, "per-dimension log-derivative gradients need row_out / const_out parameters");
        // conditioner fused: recompute it on the tensor cores, differentiate the spline in registers
        // (tc_wide.cu).  Outputs: g_x, grads->g_row_out = gradient wrt the network output of the
        // transformed dims [rows, n_tr * 48], workspace = augmented hidden activations [rows, 72].
        const void* image = (L->packed && tcw_backward_supported(L)) ? tcw_image(L) : nullptr;
        if (!image)
            return set_error(STB_ENOTSUP, "fused conditioner backward needs the tensor-core path (quadratic spline, 16 bins, MLP[64], packed): run the MLP through autograd and pass its output as row_out");
        if (direction != STB_FORWARD && direction != STB_INVERSE) return set_error(STB_EINVAL, "bad direction");
        if (rows < 0 || !x || !g_out || !g_x || !workspace) return set_error(STB_EINVAL, "bad argument");
        if (rows == 0) return STB_OK;
        if (!grads || !grads->g_row_out)
            // fused variants (the training path): the last Linear's gradient products run in the same kernel.
            //   grads == NULL: the first Linear's too -- g_x is complete; workspace at float offset rows * 72:
            //     [n_chunks * 96, 72] image of [gW_last | gb_last] (packed column order), then gW_first over the
            //     conditioning slots [64 hidden, 64 slots], then gb_first [64]; all ACCUMULATED (caller zeroes)
            //   grads != NULL (g_row_out == NULL): workspace[0 : rows * 64] = g_pre and the image; the first
            //     Linear's three K = 64 products are left to the caller
            return tcw_layer_backward_fused(L, image, direction, x, g_out, g_ldj, g_x,
                                            static_cast<float*>(workspace), grads == nullptr, rows, stream);
        return tcw_layer_backward(L, image, direction, x, g_out, g_ldj, g_x, grads->g_row_out,
                                  static_cast<float*>(workspace), rows, stream);
    }
    if (L->kind == STB_CONT_AFFINE) return set_error(STB_ENOTSUP, "continuous-affine backward is not built yet");
    if (L->has_box && L->kind != STB_RQS) return set_error(STB_EINVAL, "separate domain/codomain boxes are rqs-only");
    if (direction != STB_FORWARD && direction != STB_INVERSE) return set_error(STB_EINVAL, "bad direction");
    if (rows < 0 || !x || !g_out || !g_x) return set_error(STB_EINVAL, "bad argument");
    if (rows == 0) return STB_OK;
    if (L->row_compact && !L->mask_host && L->cond_x) return set_error(STB_EINVAL, "row_compact needs mask_host");

    const bool custom = L->spline.custom && (L->kind == STB_RQS || L->kind == STB_CUBIC);
    BwdArgs A;
    A.L.set(L);
    A.direction = direction;
    A.P = spline_params_per_dim(L->kind, L->n_bins) + (custom && L->kind == STB_RQS && L->spline.free_edge_derivs ? 2 : 0);
    int n_tr = L->dim;
    if (L->cond_x && L->mask_host) {
        n_tr = 0;
        for (int j = 0; j < L->dim; ++j) n_tr += L->mask_host[j] == 0;
    }
    A.n_tr = n_tr;
    A.width = (L->row_compact ? n_tr : L->dim) * A.P;
    A.x = x; A.g_out = g_out; A.g_ldj = g_ldj; A.g_ldiag = g_ldiag; A.g_x = g_x;
    A.g_row = grads ? grads->g_row_out : nullptr;
    A.rows = rows;
    const size_t smem = sizeof(float) * (2 * (size_t)L->dim * kBXsStride + 2 * (size_t)A.P * kBColStride) +
                        sizeof(int) * (size_t)L->dim;
    if (smem > 227 * 1024) return set_error(STB_ENOTSUP, "layer needs %zu B of shared memory per tile", smem);
    void (*kern)(BwdArgs) = nullptr;
    void (*kern_opts)(BwdArgs, SplineOpts) = nullptr;
    switch (L->kind) {
        case STB_AFFINE: kern = elementwise_backward_kernel<STB_AFFINE>; break;
        case STB_RQS: kern = elementwise_backward_kernel<STB_RQS>; kern_opts = elementwise_backward_opts_kernel<STB_RQS>; break;
        default: kern = elementwise_backward_kernel<STB_CUBIC>; kern_opts = elementwise_backward_opts_kernel<STB_CUBIC>; break;
    }
    if (smem > 48 * 1024) {
        cudaError_t e = custom ? cudaFuncSetAttribute(kern_opts, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)
                               : cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return set_error(STB_ECUDA, "cudaFuncSetAttribute: %s", cudaGetErrorString(e));
    }
    const long long tiles = (rows + kBTileRows - 1) / kBTileRows;
    if (custom) kern_opts<<<(unsigned)tiles, kBThreads, smem, stream>>>(A, make_spline_opts(L->spline));
    else kern<<<(unsigned)tiles, kBThreads, smem, stream>>>(A);
    count_launch();
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return set_error(STB_ECUDA, "elementwise_backward_kernel launch: %s", cudaGetErrorString(e));
    return STB_OK;
}

}  // namespace stb
