// The parts of tc_pack.cuh with one definition: the mask split, the spline-coupling gate and the softmax-bound pass.
#include "tc_pack.cuh"

namespace stb {
namespace tc {

bool split_mask(const stb_layer* L, int max_cond, int max_tr, MaskSplit& m) {
    if (!L->mask_host) return false;
    m = MaskSplit{};
    for (int j = 0; j < L->dim; ++j) {
        if (L->mask_host[j]) { if (m.n_cond >= max_cond) return false; m.cond_idx[m.n_cond++] = j; }
        else { if (m.n_tr >= max_tr) return false; m.tr_idx[m.n_tr++] = j; }
    }
    return m.n_tr >= 1;
}

bool tc_epilogue_ok(const stb_layer* L) {
    // The hidden activations feed the next GEMM as fp16 hi | lo parts: only activations bounded by 1 are safe
    // (a ReLU / ELU / ... output above 65504 would split into +inf, -inf -> NaN, where the reference and the
    // CUDA-core kernel stay finite).  Other activations take the generic kernel.
    if (L->net.activation != STB_ACT_TANH && L->net.activation != STB_ACT_SIGMOID) return false;
    // the tensor-core epilogues evaluate the inverse log-det as -(forward log-derivative): the Coupling convention
    return !L->inverse_ldj_own;
}

bool spline_gate(const stb_layer* L, int max_dim, int k1, MaskSplit& m) {
    if (L->kind != STB_RQS && L->kind != STB_CUBIC) return false;
    if (L->n_bins < 2 || L->n_bins > kBins || !L->cond_x || L->zero_cond || L->latent_dim < 0 || L->time_input) return false;
    if (L->has_box || L->row_out || L->dim < 2 || L->dim > max_dim) return false;
    if (L->spline.custom) return false;                    // non-default spline constants: CUDA-core kernels only
    if (!tc_epilogue_ok(L)) return false;
    const stb_mlp& N = L->net;
    if (N.n_linear < 2 || N.n_linear > 3 || N.final_activation != STB_ACT_NONE) return false;
    if (N.dims[0] != L->dim + L->latent_dim) return false;
    if (N.dims[N.n_linear] != L->dim * spline_params_per_dim(L->kind, L->n_bins)) return false;
    // [conditioning columns | latent] share GEMM1's K columns
    return split_mask(L, k1, k1, m) && m.n_cond + L->latent_dim <= k1;
}

// One warp per transformed dim: |logit_p| <= |b_p| + sum_k |W[p][k]| when the hidden activation is bounded by 1 (tanh,
// sigmoid).  If that bound is <= 100 in log2 units for all 2 K softmax rows of the dim, 2^logit cannot overflow or
// flush to zero and the spline kernels skip the max subtraction.
__global__ void tc_bound_kernel(const BoundArgs a) {
    const int ji = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), p = threadIdx.x & 31;
    bool ok = false;
    if (ji < a.n_tr && (a.act == STB_ACT_TANH || a.act == STB_ACT_SIGMOID)) {
        ok = true;
        if (p < 2 * a.n_bins) {                              // the 2 K softmax rows of the dim: [w(K) | h(K)]
            const size_t row = (size_t)a.tr_idx[ji] * a.P + p;
            float l1 = fabsf(a.b[row]);
            for (int k = 0; k < a.H; ++k) l1 += fabsf(a.W[row * a.H + k]);
            ok = (l1 * 1.4426950408889634f <= 100.f);        // false for NaN / inf
        }
    }
    ok = __all_sync(0xffffffffu, ok);
    if (p == 0 && ok) atomicOr(&a.noshift[ji >> 5], 1u << (ji & 31));
}

}  // namespace tc
}  // namespace stb
