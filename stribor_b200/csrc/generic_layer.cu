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
#include "generic_tile.cuh"

namespace stb {

template <int KIND>
__global__ void __launch_bounds__(kGenThreads) generic_layer_kernel(const GenArgs A) {
    generic_layer_tile<float, KIND>(A, DefaultOpts<KIND>(), threadIdx.x);
}

// splines with the functional API's non-default constants (stb_layer.spline.custom != 0)
template <int KIND>
__global__ void __launch_bounds__(kGenThreads) generic_layer_opts_kernel(const GenArgs A, const SplineOpts o) {
    generic_layer_tile<float, KIND>(A, o, threadIdx.x);
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

// Parameter-free layers (generic_tile.cuh)
__global__ void pointwise_kernel(int kind, int direction, const float* __restrict__ x, float* __restrict__ y,
                                 const int32_t* __restrict__ perm, float* __restrict__ ldj, int ldj_mode,
                                 int base_log_prob, int d, long long rows) {
    pointwise_row<float>(kind, direction, x, y, perm, ldj, ldj_mode, base_log_prob, d, rows);
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
    const int mode = ldj ? ldj_mode : STB_LDJ_NONE;
    if (L->dtype == STB_F64)
        return pointwise_launch_f64(L->kind, direction, x, y, perm, ldj, mode, base_log_prob, L->dim, rows,
                                    (unsigned)blocks, wpb * 32, stream);
    return launch_kernel(pointwise_kernel, (unsigned)blocks, wpb * 32, 0, stream, "pointwise_kernel", L->kind, direction,
                         x, y, perm, ldj, mode, base_log_prob, L->dim, (long long)rows);
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
int validate_layer(const stb_layer* L) {
    if (!L) return set_error(STB_EINVAL, "layer is NULL");
    if (L->kind < STB_AFFINE || L->kind > STB_LOGIT) return set_error(STB_EINVAL, "unknown transform kind %d", L->kind);
    if (L->dim < 1) return set_error(STB_EINVAL, "dim must be >= 1");
    if (L->dtype != STB_F32 && L->dtype != STB_F64) return set_error(STB_EINVAL, "unknown dtype %d", L->dtype);
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

    const size_t smem = L->dtype == STB_F64 ? generic_smem_bytes<double>(L, A.P, buf_rows, ldiag != nullptr)
                                            : generic_smem_bytes<float>(L, A.P, buf_rows, ldiag != nullptr);
    if (smem > 227 * 1024) return set_error(STB_ENOTSUP, "layer needs %zu B of shared memory per tile (> 227 KB)", smem);
    const long long tiles = (rows + kTileRows - 1) / kTileRows;
    if (tiles > 0x7fffffffLL) return set_error(STB_EINVAL, "too many rows");
    if (L->dtype == STB_F64) return generic_layer_launch_f64(L, A, smem, (unsigned)tiles, stream);

    const bool custom = L->spline.custom && (L->kind == STB_RQS || L->kind == STB_CUBIC);
    void (*kern)(GenArgs) = nullptr;
    void (*kern_opts)(GenArgs, SplineOpts) = nullptr;
    switch (L->kind) {
        case STB_AFFINE: kern = generic_layer_kernel<STB_AFFINE>; break;
        case STB_RQS: kern = generic_layer_kernel<STB_RQS>; kern_opts = generic_layer_opts_kernel<STB_RQS>; break;
        case STB_CUBIC: kern = generic_layer_kernel<STB_CUBIC>; kern_opts = generic_layer_opts_kernel<STB_CUBIC>; break;
        default: kern = generic_layer_kernel<STB_CONT_AFFINE>; break;
    }
    if (custom)
        return launch_kernel(kern_opts, (unsigned)tiles, kGenThreads, smem, stream, "generic_layer_kernel", A,
                             make_spline_opts<SplineOpts>(L->spline));
    return launch_kernel(kern, (unsigned)tiles, kGenThreads, smem, stream, "generic_layer_kernel", A);
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
