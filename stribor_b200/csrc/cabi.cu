// extern "C" surface of libstribor_b200.so (see include/stribor_b200.h).
#include <stdarg.h>
#include <stdio.h>
#include "common.cuh"

namespace stb {

static thread_local char g_err[512] = "";
static thread_local uint64_t g_launches = 0;

int set_error(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}
void count_launch() { ++g_launches; }

int sm_count() {
    static thread_local int n_sm = 0;
    if (n_sm == 0) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev);
        if (n_sm <= 0) n_sm = 148;
    }
    return n_sm;
}

int layer_images(const stb_layer* L, PackedImage img[2]) {
    int n = 0;
    uint64_t off = 0;
    auto add = [&](int family, uint64_t bytes) { img[n++] = PackedImage{family, off, bytes}; off += bytes; };
    if (tc_layer_supported(L)) {
        add(IMG_TC, tc_packed_bytes(L));
        if (tcw_layer_supported(L)) add(IMG_TCW, tcw_packed_bytes(L));
    } else if (tcw_layer_supported(L)) add(IMG_TCW, tcw_packed_bytes(L));
    else if (tch_layer_supported(L)) add(IMG_TCH, tch_packed_bytes(L));
    else if (tcm_layer_supported(L)) add(IMG_TCM, tcm_packed_bytes(L));
    return n;
}

const void* tcw_image(const stb_layer* L) {
    PackedImage img[2];
    const int n = layer_images(L, img);
    for (int i = 0; i < n; ++i)
        if (img[i].family == IMG_TCW && L->packed && L->packed_bytes >= img[i].offset + img[i].bytes)
            return static_cast<const uint8_t*>(L->packed) + img[i].offset;
    return nullptr;
}

static int apply_one(const stb_layer* L, int direction, const float* x, const float* latent,
                     const float* t, float* y, float* ldj, int ldj_mode, int base_lp, int64_t rows,
                     cudaStream_t s, float* ldiag = nullptr, int32_t* bins = nullptr) {
    int rc = validate_layer(L);
    if (rc) return rc;
    if (rows < 0) return set_error(STB_EINVAL, "rows < 0");
    if (rows == 0) return STB_OK;
    if (!x || !y) return set_error(STB_EINVAL, "x / y is NULL");
    if (bins) {                                   // -1 everywhere the kernels do not search
        cudaError_t e = cudaMemsetAsync(bins, 0xff, (size_t)rows * L->dim * sizeof(int32_t), s);
        if (e != cudaSuccess) return set_error(STB_ECUDA, "memset: %s", cudaGetErrorString(e));
    }
    if (L->kind >= STB_PERMUTE) {
        if (ldiag) return set_error(STB_ENOTSUP, "no per-dimension log-derivative for this layer kind");
        if (ldj_mode != STB_LDJ_NONE && !ldj) return set_error(STB_EINVAL, "ldj_mode set but ldj is NULL");
        return pointwise_layer_apply(L, direction, x, y, ldj, ldj_mode, base_lp, rows, s);
    }
    if (L->latent_dim > 0 && !latent) return set_error(STB_EINVAL, "layer expects a latent input");
    if ((L->kind == STB_CONT_AFFINE) && !t) return set_error(STB_EINVAL, "layer expects a time input");
    if (ldj_mode != STB_LDJ_NONE && !ldj) return set_error(STB_EINVAL, "ldj_mode set but ldj is NULL");
    if (L->packed && !ldiag && tc_layer_supported(L) && !(bins && L->n_bins != 16))
        return tc_layer_apply(L, direction, x, latent, y, ldj, ldj_mode, base_lp, rows, s, bins);
    const void* wide = (L->packed && !ldiag) ? tcw_image(L) : nullptr;
    if (wide)
        return tcw_layer_apply(L, wide, direction, x, latent, y, ldj, ldj_mode, base_lp, rows, s, bins);
    if (L->packed && !ldiag && tch_layer_supported(L))
        return tch_layer_apply(L, direction, x, latent, y, ldj, ldj_mode, base_lp, rows, s, bins);
    if (L->packed && !ldiag && tcm_layer_supported(L))
        return tcm_layer_apply(L, direction, x, latent, t, y, ldj, ldj_mode, base_lp, rows, s);
    return generic_layer_apply(L, direction, x, latent, t, y, ldj, ldj_mode, base_lp, ldiag, rows, s, bins);
}

// A run of layers that goes out as ONE chained launch: 2..8 packed couplings of one tensor-core family -- spline
// couplings of the 256-row kernel (tc_layer.cu, CHAIN) or affine / continuous-affine couplings with small conditioners
// (tc_mlp.cu, CHAIN) -- of the same dim, with any permutations (flows/permute.py) before, between or after them folded
// into the kernels' gather / scatter lists (ChainPerm): the tile keeps its original column order on chip.
struct ChainRun {
    const stb_layer* couplings[8];
    int n;                  // couplings
    int consumed;           // layers of the sequence covered (couplings + folded permutations)
    bool mlp;               // tc_mlp.cu family
    bool permuted;
    ChainPerm perm;
};

static bool pair_ok(const stb_layer* a, const stb_layer* b, bool mlp) {
    const stb_layer* two[2] = {a, b};
    return mlp ? tcm_chain_supported(two, 2) : tc_chain_supported(two, 2);
}

static bool scan_run(const stb_layer* const* seq, int n, int direction, ChainRun* run) {
    run->n = 0; run->consumed = 0; run->permuted = false; run->mlp = false;
    int d = 0;
    uint8_t phys[kChainPermMaxDim];
    int k = 0, last_good = 0;
    bool permuted = false;
    for (; k < n; ++k) {
        const stb_layer* L = seq[k];
        if (validate_layer(L) != 0) break;
        if (d == 0) {
            d = L->dim;
            if (d > kChainPermMaxDim) return false;
            for (int c = 0; c < d; ++c) phys[c] = (uint8_t)c;
        }
        if (L->dim != d) break;
        if (L->kind == STB_PERMUTE) {
            const int32_t* p = (direction == STB_FORWARD) ? L->perm_host : L->perm_inv_host;
            if (!p) break;
            uint8_t np[kChainPermMaxDim];
            for (int c = 0; c < d; ++c) {
                if (p[c] < 0 || p[c] >= d) return false;
                np[c] = phys[p[c]];                          // y[c] = x[p[c]]
            }
            for (int c = 0; c < d; ++c) phys[c] = np[c];
            permuted = true;
            if (run->n >= 2) { last_good = k + 1; for (int c = 0; c < d; ++c) run->perm.out_phys[c] = phys[c]; run->permuted = true; }
            continue;
        }
        if (L->kind >= STB_PERMUTE || run->n >= 8) break;
        if (run->n == 0) {
            if (pair_ok(L, L, false)) run->mlp = false;
            else if (pair_ok(L, L, true)) run->mlp = true;
            else break;
        } else {
            run->couplings[run->n] = L;
            const bool ok = run->mlp ? tcm_chain_supported(run->couplings, run->n + 1) : tc_chain_supported(run->couplings, run->n + 1);
            if (!ok) break;
        }
        run->couplings[run->n] = L;
        for (int c = 0; c < d; ++c) run->perm.phys[run->n][c] = phys[c];
        ++run->n;
        if (run->n >= 2) {
            last_good = k + 1;
            for (int c = 0; c < d; ++c) run->perm.out_phys[c] = phys[c];
            run->permuted = permuted;
        }
    }
    if (run->n < 2) return false;
    // `last_good` is the end of the longest prefix that ends in (coupling | trailing permutation) with >= 2 couplings;
    // couplings collected beyond it cannot exist (the loop only breaks on a non-member)
    run->consumed = last_good;
    return true;
}

// Is the whole sequence ONE chained launch (tile resident on chip from the first layer to the last)?  Then a
// log_prob caller may leave out the [rows, dim] latent output: nothing needs an HBM scratch between layers.
static bool single_chain(const stb_layer* const* seq, int n, int direction) {
    ChainRun run;
    return n >= 2 && scan_run(seq, n, direction, &run) && run.consumed == n;
}

// A sequence of layers (already in application order).  Maximal chainable runs (ChainRun) go out as ONE launch each;
// everything else layer by layer.
static int apply_sequence(const stb_layer* const* seq, int n, int direction, const float* x, const float* latent,
                          const float* t, float* out, float* ldj, int ldj_mode, int base_lp_last, int64_t rows,
                          cudaStream_t s) {
    const float* cur = x;
    int mode = ldj_mode;
    int i = 0;
    while (i < n) {
        ChainRun run;
        bool chained = false;
        if (rows > 0 && x && !(ldj_mode != STB_LDJ_NONE && !ldj))
            chained = scan_run(seq + i, n - i, direction, &run) && (out || (i == 0 && run.consumed == n));
        const int j = chained ? i + run.consumed : i + 1;
        const int last = (j == n);
        int rc;
        if (chained) {
            const ChainPerm* pm = run.permuted ? &run.perm : nullptr;
            rc = run.mlp ? tcm_chain_apply(run.couplings, run.n, direction, cur, t, out, ldj, ldj ? mode : STB_LDJ_NONE,
                                           last && base_lp_last, rows, s, pm)
                         : tc_chain_apply(run.couplings, run.n, direction, cur, latent, out, ldj, ldj ? mode : STB_LDJ_NONE,
                                          last && base_lp_last, rows, s, pm);
        } else {
            if (!out) return set_error(STB_EINVAL, "the output / scratch buffer is NULL but this flow needs several launches");
            rc = apply_one(seq[i], direction, cur, latent, t, out, ldj, ldj ? mode : STB_LDJ_NONE,
                           last && base_lp_last, rows, s);
        }
        if (rc) return rc;
        cur = out;
        if (mode == STB_LDJ_SET) mode = STB_LDJ_ADD;       // later layers accumulate
        i = j;
    }
    return STB_OK;
}

// one dtype per chain: the kernels hand each layer's output to the next as it is
static int check_one_dtype(const stb_layer* layers, int n_layers) {
    for (int i = 1; i < n_layers; ++i)
        if (layers[i].dtype != layers[0].dtype)
            return set_error(STB_EINVAL, "layer %d has dtype %d but layer 0 has %d: a flow runs in one dtype", i,
                             layers[i].dtype, layers[0].dtype);
    return STB_OK;
}

}  // namespace stb

using namespace stb;

extern "C" {

int stb_abi_version(void) { return STB_ABI_VERSION; }
const char* stb_last_error(void) { return g_err; }
uint64_t stb_launch_count(void) { return g_launches; }
uint64_t stb_sizeof_layer(void) { return sizeof(stb_layer); }

int stb_layer_apply(const stb_layer* layer, int direction, const float* x, const float* latent,
                    const float* t, float* y, float* ldj, int ldj_mode, int base_log_prob,
                    int64_t rows, void* stream) {
    if (direction != STB_FORWARD && direction != STB_INVERSE) return set_error(STB_EINVAL, "bad direction");
    return apply_one(layer, direction, x, latent, t, y, ldj, ldj_mode, base_log_prob, rows,
                     (cudaStream_t)stream);
}

int stb_layer_apply_bins(const stb_layer* layer, int direction, const float* x, const float* latent,
                         const float* t, float* y, float* ldj, int ldj_mode, int32_t* bins,
                         int64_t rows, void* stream) {
    if (direction != STB_FORWARD && direction != STB_INVERSE) return set_error(STB_EINVAL, "bad direction");
    if (!bins) return set_error(STB_EINVAL, "bins is NULL");
    return apply_one(layer, direction, x, latent, t, y, ldj, ldj_mode, 0, rows, (cudaStream_t)stream, nullptr, bins);
}

int stb_layer_apply_diag(const stb_layer* layer, int direction, const float* x, const float* latent,
                         const float* t, float* y, float* ldiag, int64_t rows, void* stream) {
    if (direction != STB_FORWARD && direction != STB_INVERSE) return set_error(STB_EINVAL, "bad direction");
    if (!ldiag) return set_error(STB_EINVAL, "ldiag is NULL");
    return apply_one(layer, direction, x, latent, t, y, nullptr, STB_LDJ_NONE, 0, rows,
                     (cudaStream_t)stream, ldiag);
}

int stb_flow_apply(const stb_layer* layers, int n_layers, int direction, const float* x,
                   const float* latent, const float* t, float* out, float* ldj, int ldj_mode,
                   int64_t rows, void* stream) {
    if (n_layers < 0 || (n_layers > 0 && !layers)) return set_error(STB_EINVAL, "bad layer list");
    if (direction != STB_FORWARD && direction != STB_INVERSE) return set_error(STB_EINVAL, "bad direction");
    cudaStream_t s = (cudaStream_t)stream;
    if (n_layers == 0) return set_error(STB_EINVAL, "empty flow: nothing to apply");
    if (n_layers > 64) return set_error(STB_EINVAL, "more than 64 layers");
    if (int rc = check_one_dtype(layers, n_layers)) return rc;
    const stb_layer* order[64];
    for (int i = 0; i < n_layers; ++i) order[i] = &layers[direction == STB_FORWARD ? i : n_layers - 1 - i];
    return apply_sequence(order, n_layers, direction, x, latent, t, out, ldj, ldj_mode, 0, rows, s);
}

int stb_flow_log_prob_needs_x_out(const stb_layer* layers, int n_layers) {
    if (n_layers < 2 || n_layers > 8 || !layers) return 1;
    const stb_layer* order[8];
    for (int i = 0; i < n_layers; ++i) order[i] = &layers[n_layers - 1 - i];
    return single_chain(order, n_layers, STB_INVERSE) ? 0 : 1;
}

int stb_flow_log_prob(const stb_layer* layers, int n_layers, const float* y, const float* latent,
                      const float* t, float* x_out, float* lp, int64_t rows, void* stream) {
    if (n_layers < 1 || !layers) return set_error(STB_EINVAL, "log_prob needs at least one layer");
    if (!lp) return set_error(STB_EINVAL, "lp is NULL");
    cudaStream_t s = (cudaStream_t)stream;
    if (n_layers > 64) return set_error(STB_EINVAL, "more than 64 layers");
    if (int rc = check_one_dtype(layers, n_layers)) return rc;
    const stb_layer* order[64];
    for (int i = 0; i < n_layers; ++i) order[i] = &layers[n_layers - 1 - i];
    if (!x_out && !(stb_flow_log_prob_needs_x_out(layers, n_layers) == 0))
        return set_error(STB_EINVAL, "x_out is NULL but this flow is evaluated in several launches and needs the [rows, dim] scratch");
    return apply_sequence(order, n_layers, STB_INVERSE, y, latent, t, x_out, lp, STB_LDJ_SET, 1, rows, s);
}

int stb_unit_normal_log_prob(const float* x, float* lp, int accumulate, int32_t dim, int64_t rows,
                             void* stream) {
    if (!x || !lp || dim < 1 || rows < 0) return set_error(STB_EINVAL, "bad argument");
    return unit_normal_apply(x, lp, accumulate, dim, rows, (cudaStream_t)stream);
}

uint64_t stb_layer_backward_workspace_bytes(const stb_layer* layer, int64_t rows) {
    return layer_backward_workspace_bytes(layer, rows);
}

int stb_layer_backward(const stb_layer* layer, int direction, const float* x, const float* latent,
                       const float* t, const float* g_out, const float* g_ldj, float* g_x,
                       float* g_latent, float* g_t, const stb_layer_grads* grads, void* workspace,
                       int64_t rows, void* stream) {
    int rc = validate_layer(layer);
    if (rc) return rc;
    return layer_backward(layer, direction, x, latent, t, g_out, g_ldj, g_x, g_latent, g_t, grads,
                          workspace, rows, (cudaStream_t)stream);
}

int stb_layer_backward_diag(const stb_layer* layer, int direction, const float* x, const float* g_out,
                            const float* g_ldiag, float* g_x, const stb_layer_grads* grads, int64_t rows,
                            void* stream) {
    int rc = validate_layer(layer);
    if (rc) return rc;
    if (layer->net.n_linear > 0 || layer->kind >= STB_CONT_AFFINE)
        return set_error(STB_ENOTSUP, "stb_layer_backward_diag: affine / spline layers with row_out or const_out parameters only");
    return layer_backward(layer, direction, x, nullptr, nullptr, g_out, nullptr, g_x, nullptr, nullptr, grads,
                          nullptr, rows, (cudaStream_t)stream, g_ldiag);
}

uint64_t stb_packed_bytes(const stb_layer* layer) {
    if (validate_layer(layer)) return 0;
    PackedImage img[2];
    const int n = layer_images(layer, img);
    return n ? img[n - 1].offset + img[n - 1].bytes : 0;
}

int stb_pack_layer(const stb_layer* layer, void* packed_out, void* stream) {
    int rc = validate_layer(layer);
    if (rc) return rc;
    if (!packed_out) return set_error(STB_EINVAL, "packed_out is NULL");
    if (layer->dtype != STB_F32) return set_error(STB_EINVAL, "fp64 layers have no packed image (CUDA-core kernels only)");
    PackedImage img[2];
    const int n = layer_images(layer, img);
    if (n == 0) return set_error(STB_ENOTSUP, "layer has no tensor-core path");
    for (int i = 0; i < n && rc == 0; ++i) {
        void* out = static_cast<uint8_t*>(packed_out) + img[i].offset;
        const cudaStream_t s = (cudaStream_t)stream;
        switch (img[i].family) {
            case IMG_TC: rc = tc_pack_layer(layer, out, s); break;
            case IMG_TCW: rc = tcw_pack_layer(layer, out, s); break;
            case IMG_TCH: rc = tch_pack_layer(layer, out, s); break;
            default: rc = tcm_pack_layer(layer, out, s); break;
        }
    }
    return rc;
}

int stb_layer_uses_tensor_path(const stb_layer* layer) {
    if (validate_layer(layer)) return 0;
    PackedImage img[2];
    return (layer->packed && layer_images(layer, img) > 0) ? 1 : 0;
}

}  // extern "C"
