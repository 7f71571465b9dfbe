// Backward of the element-wise transforms (affine / rational-quadratic / cubic) of a layer whose
// network output is supplied per row (row_out) or as a constant (const_out): what autograd derives
// for flows/affine.py:97-109, util/rational_quadratic_spline.py and util/cubic_spline.py.
//
// Same tiling as generic_layer.cu: one CTA = 32 rows, lane = row, a warp owns a subset of the
// transformed dims.  Parameters and their gradients live in padded shared-memory columns so both
// the per-thread access ([p][thread]) and the transposed, coalesced global access ([row][p]) are
// bank-conflict free.
#include "backward_tile.cuh"

namespace stb {

template <int KIND>
__global__ void __launch_bounds__(kBThreads) elementwise_backward_kernel(const BwdArgs A) {
    elementwise_backward_tile<float, KIND>(A, DefaultOpts<KIND>(), threadIdx.x);
}

// splines with the functional API's non-default constants (stb_layer.spline.custom != 0)
template <int KIND>
__global__ void __launch_bounds__(kBThreads) elementwise_backward_opts_kernel(const BwdArgs A, const SplineOpts o) {
    elementwise_backward_tile<float, KIND>(A, o, threadIdx.x);
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
    const size_t smem = L->dtype == STB_F64 ? backward_smem_bytes<double>(L, A.P) : backward_smem_bytes<float>(L, A.P);
    if (smem > 227 * 1024) return set_error(STB_ENOTSUP, "layer needs %zu B of shared memory per tile", smem);
    const long long tiles = (rows + kBTileRows - 1) / kBTileRows;
    if (L->dtype == STB_F64) return elementwise_backward_launch_f64(L, A, smem, (unsigned)tiles, stream);
    void (*kern)(BwdArgs) = nullptr;
    void (*kern_opts)(BwdArgs, SplineOpts) = nullptr;
    switch (L->kind) {
        case STB_AFFINE: kern = elementwise_backward_kernel<STB_AFFINE>; break;
        case STB_RQS: kern = elementwise_backward_kernel<STB_RQS>; kern_opts = elementwise_backward_opts_kernel<STB_RQS>; break;
        default: kern = elementwise_backward_kernel<STB_CUBIC>; kern_opts = elementwise_backward_opts_kernel<STB_CUBIC>; break;
    }
    if (custom)
        return launch_kernel(kern_opts, (unsigned)tiles, kBThreads, smem, stream, "elementwise_backward_kernel", A,
                             make_spline_opts<SplineOpts>(L->spline));
    return launch_kernel(kern, (unsigned)tiles, kBThreads, smem, stream, "elementwise_backward_kernel", A);
}

}  // namespace stb
