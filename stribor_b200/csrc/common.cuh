// Host-side plumbing shared by the translation units of libstribor_b200.so:
// thread-local error text, launch counter, SM count, internal entry points.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>
#include <string.h>
#include "../../include/stribor_b200.h"

namespace stb {

// A kernel's by-value copy of a stb_layer: its fields up to, not including, `spline`.  The spline options reach
// only the kernels instantiated for non-default options, as a kernel parameter of their own, so the argument
// layout of every other kernel is the one it had before the options were appended to stb_layer.
struct LayerArgs {
    alignas(stb_layer) unsigned char raw[offsetof(stb_layer, spline)];
    void set(const stb_layer* L) { memcpy(raw, L, sizeof raw); }
    __host__ __device__ __forceinline__ const stb_layer& get() const { return *reinterpret_cast<const stb_layer*>(raw); }
};

int set_error(int code, const char* fmt, ...);
void count_launch();
// multiprocessors of the current device, looked up once per host thread (148, a B200's count, if the query fails)
int sm_count();

int validate_layer(const stb_layer* L);

// network outputs per transformed dim: rqs 3K - 1, cubic 2K + 2, affine kinds 2 (log-scale, shift)
__host__ __device__ inline int spline_params_per_dim(int kind, int K) {
    return kind == STB_RQS ? 3 * K - 1 : (kind == STB_CUBIC ? 2 * K + 2 : 2);
}

int generic_layer_apply(const stb_layer* L, int direction, const float* x, const float* latent,
                        const float* t, float* y, float* ldj, int ldj_mode, int base_log_prob,
                        float* ldiag, int64_t rows, cudaStream_t stream, int32_t* bins = nullptr);
int pointwise_layer_apply(const stb_layer* L, int direction, const float* x, float* y, float* ldj,
                          int ldj_mode, int base_log_prob, int64_t rows, cudaStream_t stream);
int unit_normal_apply(const float* x, float* lp, int accumulate, int dim, int64_t rows,
                      cudaStream_t stream);

// tcgen05 path (tc_layer.cu)
bool tc_layer_supported(const stb_layer* L);
uint64_t tc_packed_bytes(const stb_layer* L);
int tc_pack_layer(const stb_layer* L, void* out, cudaStream_t stream);
int tc_layer_apply(const stb_layer* L, int direction, const float* x, const float* latent, float* y, float* ldj,
                   int ldj_mode, int base_log_prob, int64_t rows, cudaStream_t stream, int32_t* bins = nullptr);

// Permutations (flows/permute.py:11-82) between chained couplings are folded into the kernels' index lists: the tile
// keeps its ORIGINAL column order on chip, layer l gathers / scatters logical column j at physical column phys[l][j],
// and the tile is written back as y[:, i] = tile[:, out_phys[i]].  Built by cabi.cu from stb_layer.perm_host.
constexpr int kChainPermMaxLayers = 8, kChainPermMaxDim = 64;
struct ChainPerm {
    uint8_t phys[kChainPermMaxLayers][kChainPermMaxDim];
    uint8_t out_phys[kChainPermMaxDim];
};

// several layers of one flow in one launch (tc_layer.cu, CHAIN kernels); layers[] in application order
bool tc_chain_supported(const stb_layer* const* layers, int n);
int tc_chain_apply(const stb_layer* const* layers, int n, int direction, const float* x, const float* latent, float* y,
                   float* ldj, int ldj_mode, int base_log_prob, int64_t rows, cudaStream_t stream,
                   const ChainPerm* perm = nullptr);

// tcgen05 path for dim <= 128 and the training backward (tc_wide.cu).  `image` is the wide packed image (tcw_image).
bool tcw_layer_supported(const stb_layer* L);
bool tcw_backward_supported(const stb_layer* L);
uint64_t tcw_packed_bytes(const stb_layer* L);
int tcw_pack_layer(const stb_layer* L, void* out, cudaStream_t stream);
int tcw_layer_apply(const stb_layer* L, const void* image, int direction, const float* x, const float* latent, float* y,
                    float* ldj, int ldj_mode, int base_log_prob, int64_t rows, cudaStream_t stream,
                    int32_t* bins = nullptr);
int tcw_layer_backward(const stb_layer* L, const void* image, int direction, const float* x, const float* g_out,
                       const float* g_ldj, float* g_x, float* g_net, float* hidden, int64_t rows,
                       cudaStream_t stream);
uint64_t tcw_train_workspace_floats(const stb_layer* L, int64_t rows);
int tcw_layer_backward_fused(const stb_layer* L, const void* image, int direction, const float* x, const float* g_out,
                             const float* g_ldj, float* g_x, float* workspace, int first_linear, int64_t rows,
                             cudaStream_t stream);
// the layer's wide image (layer_images), NULL when it has none or `packed` is too small to hold it
const void* tcw_image(const stb_layer* L);

// tcgen05 path for spline couplings with a wide conditioner, MLP[H] / MLP[H,H], H <= 256 (tc_hwide.cu)
bool tch_layer_supported(const stb_layer* L);
uint64_t tch_packed_bytes(const stb_layer* L);
int tch_pack_layer(const stb_layer* L, void* out, cudaStream_t stream);
int tch_layer_apply(const stb_layer* L, int direction, const float* x, const float* latent, float* y, float* ldj,
                    int ldj_mode, int base_log_prob, int64_t rows, cudaStream_t stream, int32_t* bins = nullptr);

// tcgen05 path for affine couplings with a wide conditioner (tc_mlp.cu)
bool tcm_layer_supported(const stb_layer* L);
uint64_t tcm_packed_bytes(const stb_layer* L);
int tcm_pack_layer(const stb_layer* L, void* out, cudaStream_t stream);
int tcm_layer_apply(const stb_layer* L, int direction, const float* x, const float* latent, const float* t, float* y,
                    float* ldj, int ldj_mode, int base_log_prob, int64_t rows, cudaStream_t stream);

// every layer of an affine / continuous-affine flow with small conditioners in one launch (tc_mlp.cu, CHAIN kernel)
bool tcm_chain_supported(const stb_layer* const* layers, int n);
int tcm_chain_apply(const stb_layer* const* layers, int n, int direction, const float* x, const float* t, float* y,
                    float* ldj, int ldj_mode, int base_log_prob, int64_t rows, cudaStream_t stream,
                    const ChainPerm* perm = nullptr);

// The packed images of a layer (stb_pack_layer), in the order they sit in stb_layer.packed: an MLP[64] spline layer
// that fits tc_layer.cu carries that image and then the tc_wide.cu one.  Returns how many (0 .. 2).  (cabi.cu)
enum { IMG_TC, IMG_TCW, IMG_TCH, IMG_TCM };
struct PackedImage { int family; uint64_t offset, bytes; };
int layer_images(const stb_layer* L, PackedImage img[2]);

// backward (backward.cu)
uint64_t layer_backward_workspace_bytes(const stb_layer* L, int64_t rows);
int layer_backward(const stb_layer* L, int direction, const float* x, const float* latent,
                   const float* t, const float* g_out, const float* g_ldj, float* g_x,
                   float* g_latent, float* g_t, const stb_layer_grads* grads, void* workspace,
                   int64_t rows, cudaStream_t stream, const float* g_ldiag = nullptr);

}  // namespace stb
