// Tile body of the element-wise backward kernels (backward.cu), generic over the scalar type T: the fp32
// kernels instantiate it for float (backward.cu), the fp64 kernels for double (float64.cu).  The argument
// block keeps the C ABI's float pointers; they point to T.
#pragma once
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

// dynamic shared memory of one elementwise_backward_tile<T>
template <class T>
size_t backward_smem_bytes(const stb_layer* L, int P) {
    return sizeof(T) * (2 * (size_t)L->dim * kBXsStride + 2 * (size_t)P * kBColStride) + sizeof(int) * (size_t)L->dim;
}

// One tile of the element-wise backward kernel, scalar type T; O holds the spline constants (stb_math.cuh).
// The kernel reads threadIdx.x itself: there the compiler knows its range from __launch_bounds__.
template <class T, int KIND, class O>
__device__ __forceinline__ void elementwise_backward_tile(const BwdArgs& A, const O& o, const int tid) {
    extern __shared__ __align__(16) float smem[];
    const stb_layer& L = A.L.get();
    const int d = L.dim, P = A.P;
    const int lane = tid & 31, warp = tid >> 5;
    const long long row0 = (long long)blockIdx.x * kBTileRows;
    const int nrows = (int)min((long long)kBTileRows, A.rows - row0);

    T* xs = reinterpret_cast<T*>(smem);                // [d][33]   layer input
    T* gs = xs + d * kBXsStride;                       // [d][33]   g_out -> g_x
    T* prm = gs + d * kBXsStride;                      // [P][129]
    T* gpr = prm + P * kBColStride;                    // [P][129]
    int* tr_list = reinterpret_cast<int*>(gpr + P * kBColStride);
    __shared__ int n_tr_s;

    {
        const T* xg = reinterpret_cast<const T*>(A.x) + row0 * d;
        const T* gg = reinterpret_cast<const T*>(A.g_out) + row0 * d;
        const int n = nrows * d;
        for (int i = tid; i < kBTileRows * d; i += kBThreads) {
            const int r = i / d, c = i - r * d;
            xs[c * kBXsStride + r] = (i < n) ? xg[i] : T(0);
            gs[c * kBXsStride + r] = (i < n) ? gg[i] : T(0);
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
    const T g_ld_row = (A.g_ldj != nullptr && lane < nrows) ? reinterpret_cast<const T*>(A.g_ldj)[row0 + lane] : T(0);
    SmemCol<T> col{prm + tid, kBColStride};
    SmemCol<T> gcol{gpr + tid, kBColStride};
    T* pw = prm + warp * 32;                           // this warp's 32 columns
    T* gw = gpr + warp * 32;

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
                        T v[8];
#pragma unroll
                        for (int u = 0; u < 8; ++u) {
                            const int r = r0 + u;
                            v[u] = (p < P && r < nrows) ? __ldg(reinterpret_cast<const T*>(L.row_out) + (size_t)(row0 + r) * A.width + c0 + p) : T(0);
                        }
                        if (p < P) {
#pragma unroll
                            for (int u = 0; u < 8; ++u) pw[p * kBColStride + r0 + u] = v[u];
                        }
                    }
                }
            } else {
                for (int p = 0; p < P; ++p)
                    col[p] = (lane < nrows) ? __ldg(reinterpret_cast<const T*>(L.row_out) + (size_t)(row0 + lane) * A.width + bwd_col(L, P, n_tr, it, j, p)) : T(0);
            }
        } else {
            for (int p = 0; p < P; ++p) col[p] = __ldg(reinterpret_cast<const T*>(L.const_out) + bwd_col(L, P, n_tr, it, j, p));
        }
        __syncwarp();
        // ---- element gradient -------------------------------------------------------------------------
        const T xv = xs[j * kBXsStride + lane];
        const T go = gs[j * kBXsStride + lane];
        T g_ld = g_ld_row;
        if (A.g_ldiag != nullptr && lane < nrows) g_ld += reinterpret_cast<const T*>(A.g_ldiag)[(row0 + lane) * d + j];
        T gx;
        if constexpr (KIND == STB_AFFINE) {
            const T ls = col[0], sh = col[1];
            if (inverse) {
                const T e = exp_(-ls), out = (xv - sh) * e;
                gx = go * e; gcol[1] = -go * e; gcol[0] = -go * out - g_ld;
            } else {
                const T e = exp_(ls);
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
                    T* dst = reinterpret_cast<T*>(A.g_row) + (size_t)(row0 + r) * A.width + c0;
                    for (int p = lane; p < P; p += 32) dst[p] = gw[p * kBColStride + r];
                }
            } else if (lane < nrows) {
                for (int p = 0; p < P; ++p)
                    reinterpret_cast<T*>(A.g_row)[(size_t)(row0 + lane) * A.width + bwd_col(L, P, n_tr, it, j, p)] = gcol[p];
            }
        }
        __syncwarp();
    }
    __syncthreads();
    {
        T* gx = reinterpret_cast<T*>(A.g_x) + row0 * d;
        const int n = nrows * d;
        for (int i = tid; i < n; i += kBThreads) {
            const int r = i / d, c = i - r * d;
            gx[i] = gs[c * kBXsStride + r];
        }
    }
}

// fp64 launch (float64.cu): the double instantiation of the kernel above
int elementwise_backward_launch_f64(const stb_layer* L, const BwdArgs& A, size_t smem, unsigned tiles,
                                    cudaStream_t stream);

}  // namespace stb
