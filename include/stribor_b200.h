/* stribor_b200 -- C ABI of the B200 (sm_100a) coupling-flow kernels.
 *
 * This header is the drop-in boundary.  The reference (mbilos/stribor 0.2.0) is pure
 * PyTorch and has no FFI layer; what a binding replaces is the arithmetic done inside
 * these reference methods (paths relative to the reference checkout):
 *
 *   stb_layer_apply      <- Coupling.forward / inverse / log_det_jacobian
 *                           (stribor/flows/coupling.py:69-95), with Affine
 *                           (flows/affine.py:97-123) or Spline (flows/spline.py:89-143 ->
 *                           util/rational_quadratic_spline.py:11-251, util/cubic_spline.py:22-247)
 *                           and the latent MLP (net/mlp.py:46-65); also the inherited
 *                           forward_and_/inverse_and_log_det_jacobian (flow.py:35-47) and
 *                           ContinuousAffineCoupling (flows/coupling.py:188-213) with
 *                           TimeLinear (net/time_net.py:18-28)
 *   stb_flow_apply       <- NormalizingFlow.forward / inverse / *_and_log_det_jacobian
 *                           (flow.py:99-125) and NeuralFlow.forward (flow.py:172-184)
 *   stb_flow_log_prob    <- NormalizingFlow.log_prob (flow.py:127-130) with UnitNormal
 *                           (dist/normal.py:40-54)
 *   stb_layer_backward   <- what autograd derives for the above in the NLL training step
 *   stb_pack_layer       <- (new) one-off repack of nn.Linear weights for the tcgen05 path
 *
 * Conventions: plain C, no C++ types, no exceptions.  Every function returns 0 on success
 * or a negative STB_E* code; stb_last_error() gives a thread-local message.  The CALLER owns
 * every buffer (device pointers unless stated), the library never allocates device memory,
 * never synchronises and keeps no global mutable state, so calls are re-entrant across
 * streams, devices and host threads.  All tensors are fp32, row-major, rows contiguous:
 * x/y [rows, dim], latent [rows, latent_dim], t [rows, 1], ldj/lp [rows].
 */
#ifndef STRIBOR_B200_H_
#define STRIBOR_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define STB_ABI_VERSION 3
#define STB_MAX_LINEAR 8

/* error codes */
#define STB_OK 0
#define STB_EINVAL (-1)      /* bad argument / unsupported configuration  */
#define STB_ECUDA (-2)       /* CUDA runtime error (launch, attribute)     */
#define STB_ENOTSUP (-3)     /* valid in the reference, not built here yet */

/* transform kinds (flows/affine.py, flows/spline.py, flows/coupling.py:98) */
enum { STB_AFFINE = 0, STB_RQS = 1, STB_CUBIC = 2, STB_CONT_AFFINE = 3,
       /* parameter-free layers that sit between couplings ("next" rows of the scope table):
        * flows/permute.py:11-82 (Flip of the last dim is the permutation dim-1..0) and
        * flows/sigmoid.py:9-56 */
       STB_PERMUTE = 4, STB_SIGMOID = 5, STB_LOGIT = 6 };

/* activations by torch.nn class name (net/mlp.py:38-41) */
enum { STB_ACT_NONE = 0, STB_ACT_TANH = 1, STB_ACT_RELU = 2, STB_ACT_SIGMOID = 3, STB_ACT_ELU = 4,
       STB_ACT_SOFTPLUS = 5, STB_ACT_LEAKY_RELU = 6, STB_ACT_SILU = 7, STB_ACT_GELU = 8 };

/* directions */
enum { STB_FORWARD = 0, STB_INVERSE = 1 };

/* what to do with the per-row log|det J| of a layer */
enum { STB_LDJ_NONE = 0,      /* not computed                                          */
       STB_LDJ_SET = 1,       /* ldj[row]  = value                                     */
       STB_LDJ_ADD = 2 };     /* ldj[row] += value                                     */

/* Latent network: Linear -> (act -> Linear)* [-> final act]   (net/mlp.py:46-58)
 * W[i] is nn.Linear layout [dims[i+1], dims[i]] row-major, b[i] is [dims[i+1]]. */
typedef struct stb_mlp {
    int32_t n_linear;                  /* 0 = no network: `const_out` below is used     */
    int32_t activation;
    int32_t final_activation;
    int32_t dims[STB_MAX_LINEAR + 1];
    const float* W[STB_MAX_LINEAR];
    const float* b[STB_MAX_LINEAR];
} stb_mlp;

/* One invertible layer.
 *   cond_x = 1: a Coupling -- the network input is [x*mask | latent | t?]; dims with
 *               mask 0 are transformed, dims with mask 1 pass through.
 *   cond_x = 0: a stand-alone element-wise transform -- the network input is [latent];
 *               every dim is transformed (`mask` ignored).
 * Network output layout (flows/affine.py:66, flows/spline.py:82-86):
 *   affine / cont-affine: [log_scale(dim) | shift(dim)]
 *   rqs:   per dim [widths(K) | heights(K) | derivatives(K-1)]
 *          (K+1 derivatives, boundary ones included, when spline.free_edge_derivs is set)
 *   cubic: per dim [widths(K) | heights(K) | left, right derivative]
 */

/* Spline constants of the functional API: the keyword arguments of the reference's
 * unconstrained_rational_quadratic_spline / unconstrained_cubic_spline.  custom == 0 (a zero-filled block) means the reference
 * defaults -- rqs: minimum bin width / height / derivative 1e-3, K-1 derivatives;
 * cubic: minimum bin width / height 1e-2, eps 1e-5, quadratic_threshold 1e-3 -- and every
 * other field is ignored.  With custom != 0 all fields of the layer's kind are used.
 * Layers with custom != 0 run on the CUDA-core kernels only (row_out / const_out
 * parameters); they never take a tensor-core path. */
typedef struct stb_spline_opts {
    int32_t custom;
    float min_bin_width, min_bin_height;  /* rqs and cubic; min * n_bins <= 1 each        */
    float min_derivative;                 /* rqs: derivative = min + softplus(param), >= 0 */
    int32_t free_edge_derivs;             /* rqs: 1 = K+1 derivative parameters per dim, the
                                             boundary derivatives included; 0 = K-1, the
                                             boundaries padded with log(exp(1 - min) - 1),
                                             i.e. a boundary derivative of exactly 1       */
    float cub_eps;                        /* cubic: root window of the inverse            */
    float cub_quad_threshold;             /* cubic: |a| below it -> quadratic formula     */
} stb_spline_opts;

typedef struct stb_layer {
    int32_t kind;
    int32_t dim;
    int32_t latent_dim;
    int32_t cond_x;
    int32_t time_input;        /* cont-affine: t is the last network input                */
    int32_t n_bins;
    int32_t inverse_ldj_own;   /* inverse: 1 = log-derivative of the inverse map itself
                                  (Spline.inverse_and_log_det_jacobian, spline.py:119-123);
                                  0 = -(forward log-derivative at the recovered point),
                                  the inherited default (flow.py:42-47) Coupling uses      */
    int32_t zero_cond;         /* dim == 1: conditioning on x is multiplied by 0
                                  (coupling.py:62-63)                                      */
    float lower, upper;        /* spline box: domain == codomain == [lower, upper]        */
    float left, right;         /* rqs only, used when has_box != 0: domain [left, right]  */
    float bottom, top;         /*   and codomain [bottom, top]
                                  (rational_quadratic_spline.py:55-64)                     */
    int32_t has_box;
    int32_t row_compact;       /* row_out holds only the transformed dims' parameters, in mask
                                  order: [rows, n_tr * P] (affine: [log_scale(n_tr) | shift(n_tr)]) */
    const uint8_t* mask;       /* device, [dim], 1 = pass through / conditions            */
    const uint8_t* mask_host;  /* HOST copy of the mask (optional; needed by stb_pack_layer
                                  and for the tensor-core path to be selected)            */
    const float* const_out;    /* device, network-output-shaped vector when n_linear == 0 */
    const float* row_out;      /* device, [rows, out_width]: a precomputed network output
                                  PER ROW (n_linear == 0; takes precedence over const_out) */
    const float* time_scale;   /* device, [2*dim] TimeLinear.scale (cont-affine)          */
    const int32_t* perm;       /* device, [dim]: STB_PERMUTE forward is y[i] = x[perm[i]];
                                  perm_inv the inverse permutation                        */
    const int32_t* perm_inv;
    stb_mlp net;
    const void* packed;        /* device, from stb_pack_layer (NULL = generic path only)  */
    uint64_t packed_bytes;
    const int32_t* perm_host;      /* HOST copies of perm / perm_inv (optional).  With them a permutation  */
    const int32_t* perm_inv_host;  /* between chained couplings is folded into the neighbouring kernels'    */
                                   /* gather / scatter index lists instead of costing an HBM pass           */
    stb_spline_opts spline;        /* rqs / cubic constants; zero-filled = the reference defaults          */
} stb_layer;

int stb_abi_version(void);
uint64_t stb_sizeof_layer(void);          /* sizeof(stb_layer), for binding self-checks */
const char* stb_last_error(void);

/* y = T(x) (STB_FORWARD) or T^-1(x) (STB_INVERSE) for one layer; optionally the per-row
 * log|det J| with the reference's sign conventions (see inverse_ldj_own).  x and y may
 * alias.  `base_log_prob` != 0 additionally adds the UnitNormal log-density of the OUTPUT
 * row to ldj (used for the last layer of log_prob). */
int stb_layer_apply(const stb_layer* layer, int direction, const float* x, const float* latent,
                    const float* t, float* y, float* ldj, int ldj_mode, int base_log_prob,
                    int64_t rows, void* stream);

/* Element-wise variant: additionally writes the per-dimension log-derivative
 * ldiag [rows, dim] (0 for pass-through dims) -- ElementwiseTransform.log_diag_jacobian
 * (flow.py:50-69, affine.py:115-123, spline.py:135-143). */
int stb_layer_apply_diag(const stb_layer* layer, int direction, const float* x, const float* latent,
                         const float* t, float* y, float* ldiag, int64_t rows, void* stream);

/* Parity instrument: stb_layer_apply that ALSO reports, per element, the bin the spline's knot search chose
 * -- util/search_sorted.py:3-5 as called from util/rational_quadratic_spline.py:194-197 and
 * util/cubic_spline.py:140-143 (STB_FORWARD searches the cumulative widths, STB_INVERSE the cumulative
 * heights).  bins [rows, dim] int32: the bin index in [0, n_bins), or -1 for pass-through dims, for elements
 * outside the spline box (identity tails) and for non-spline layers.  The call takes exactly the kernel
 * path stb_layer_apply takes for this layer (tensor-core kernels when `packed` is set), so what it reports
 * is the product path's own search, not a re-computation. */
int stb_layer_apply_bins(const stb_layer* layer, int direction, const float* x, const float* latent,
                         const float* t, float* y, float* ldj, int ldj_mode, int32_t* bins,
                         int64_t rows, void* stream);

/* Chain of layers, applied first-to-last (STB_FORWARD) or last-to-first with each layer
 * inverted (STB_INVERSE).  `out` may alias `x`.  ldj (nullable) receives the summed
 * log|det J| according to ldj_mode. */
int stb_flow_apply(const stb_layer* layers, int n_layers, int direction, const float* x,
                   const float* latent, const float* t, float* out, float* ldj, int ldj_mode,
                   int64_t rows, void* stream);

/* lp[row] = log N(x; 0, I) + sum_layers ldj, x = inverse chain of y  (flow.py:127-130).
 * `x_out` [rows, dim] receives the latent x and doubles as the scratch between launches.  It may be NULL when
 * stb_flow_log_prob_needs_x_out() returns 0 -- the whole flow is one chained launch whose tile never leaves the
 * chip -- which halves the compulsory HBM traffic of log_prob (4d + 4 instead of 8d + 4 bytes per row). */
int stb_flow_log_prob_needs_x_out(const stb_layer* layers, int n_layers);
int stb_flow_log_prob(const stb_layer* layers, int n_layers, const float* y, const float* latent,
                      const float* t, float* x_out, float* lp, int64_t rows, void* stream);

/* lp[row] (+)= sum_j -x_j^2/2 - log(sqrt(2 pi))   (dist/normal.py:37) */
int stb_unit_normal_log_prob(const float* x, float* lp, int accumulate, int32_t dim, int64_t rows,
                             void* stream);

/* Gradient of one layer application, recomputing the layer from its saved INPUT `x`
 * (the tensor stb_layer_apply was called with).  g_out [rows,dim] and g_ldj [rows]
 * (nullable) are the incoming gradients of the layer's outputs; g_x [rows,dim],
 * g_latent, g_t (nullable) receive input gradients; gW[i]/gb[i] (same shapes as the
 * weights; accumulated into, caller zeroes) receive parameter gradients;
 * g_const_out / g_time_scale likewise.  `workspace` must hold
 * stb_layer_backward_workspace_bytes(layer, rows) bytes.
 * Two families are built:
 *  (1) n_linear == 0 (row_out / const_out): the element-wise gradient -- g_x and grads->g_row_out are
 *      written; the caller runs a conditioner through autograd (library GEMMs) around it.
 *  (2) n_linear > 0 with a packed image (stb_pack_layer), quadratic or cubic spline, 16 bins, MLP[64], dim <= 128,
 *      Tanh / Sigmoid / ReLU hidden activation: the conditioner is RECOMPUTED on the tensor cores from the
 *      saved input and the spline differentiated in registers (tc_wide.cu).  g_x receives the transformed
 *      dims' gradient and g_out for the pass-through dims (the conditioner's contribution to them is
 *      g_pre W1 over the conditioning columns, see below).  With W = stb_layer_backward_workspace_bytes:
 *        grads == NULL  (everything fused -- the training path): g_x is COMPLETE (pass-through dims include
 *          the conditioner's contribution); at float offset rows*72 of the workspace, all ACCUMULATED into
 *          (caller zeroes), summed over row tiles with atomics (order not deterministic):
 *            [n_tr_pad*48, 72]   [gW_last | gb_last | 0..] for the transformed dims' rows of the last Linear,
 *                                48 rows per transformed dim in packed column order
 *                                (w_0, h_0, w_1, h_1, ... w_15, h_15, d_0..d_14 (cubic: left, right), pad)
 *            [64, 64]            gW_first over the conditioning SLOTS (slot k = k-th pass-through dim)
 *            [64]                gb_first
 *        grads != NULL, grads->g_row_out == NULL: as above without the first Linear -- workspace[0 : rows*64]
 *          receives g_pre (gradient wrt the hidden pre-activation), g_x carries g_out on the pass-through dims,
 *          and the caller forms gW_first[:, cond] = g_pre^T x[:, cond], gb_first = sum g_pre,
 *          g_x[:, cond] += g_pre W_first[:, cond]
 *        grads->g_row_out != NULL  (two-step variant, quadratic only: exact fp32 products left to the caller)
 *          grads->g_row_out [rows, n_tr*48]  gradient wrt the network output of the transformed dims,
 *                                            natural order [w(16) | h(16) | d(15) | 0]
 *          workspace[0 : rows*72]            [hidden(64) | 1 | 0 x 7] per row; the caller forms
 *                                            g_pre = (g_row_out W_last) * act'(hidden) and all four products
 *      gW / gb pointers of stb_layer_grads are not used by this family.
 *      Any other layer with n_linear > 0 returns STB_ENOTSUP. */
typedef struct stb_layer_grads {
    float* gW[STB_MAX_LINEAR];
    float* gb[STB_MAX_LINEAR];
    float* g_const_out;
    float* g_time_scale;
    float* g_row_out;          /* n_linear == 0: per-row gradient wrt the network output,
                                  [rows, out_width] in the layout of row_out (also produced for
                                  const_out layers: the caller sums it over rows)                */
} stb_layer_grads;

uint64_t stb_layer_backward_workspace_bytes(const stb_layer* layer, int64_t rows);
int stb_layer_backward(const stb_layer* layer, int direction, const float* x, const float* latent,
                       const float* t, const float* g_out, const float* g_ldj, float* g_x,
                       float* g_latent, float* g_t, const stb_layer_grads* grads, void* workspace,
                       int64_t rows, void* stream);

/* Gradient of stb_layer_apply_diag for layers whose parameters are supplied (n_linear == 0: row_out or
 * const_out) -- what autograd derives for ElementwiseTransform.forward_and_log_diag_jacobian
 * (flow.py:57-69; affine.py:97-123, spline.py:101-105 -> util/rational_quadratic_spline.py:11-251 incl.
 * the separate left/right/bottom/top boxes, util/cubic_spline.py:22-247).  g_out [rows, dim] and
 * g_ldiag [rows, dim] (nullable) are the incoming gradients of y and of the per-dimension log-derivative;
 * g_x [rows, dim] and grads->g_row_out (layout of row_out; also written for const_out layers, the caller
 * sums it over rows) receive the results. */
int stb_layer_backward_diag(const stb_layer* layer, int direction, const float* x, const float* g_out,
                            const float* g_ldiag, float* g_x, const stb_layer_grads* grads, int64_t rows,
                            void* stream);

/* tcgen05 path: size of / build the packed weight image for a layer (0 bytes = this layer
 * configuration only runs on the generic path).  Layers with an image (round 2): spline couplings
 * (quadratic / cubic, 2 <= n_bins <= 16) with an MLP[64] conditioner at dim <= 128 or an MLP[H] / MLP[H,H]
 * conditioner (H in {64, 128, 192, 256}) at dim <= 64; affine and continuous-affine couplings with MLP[H] /
 * MLP[H,H]; Tanh / Sigmoid hidden activations; `latent_dim` > 0 as long as conditioning columns + latent (+ t)
 * fit the first GEMM's K columns (32; 64 in the dim <= 128 kernel); inverse_ldj_own == 0. */
uint64_t stb_packed_bytes(const stb_layer* layer);
int stb_pack_layer(const stb_layer* layer, void* packed_out, void* stream);

/* 1 if stb_layer_apply would take the tcgen05 path for this (packed) layer. */
int stb_layer_uses_tensor_path(const stb_layer* layer);

/* Bring-up check of the tcgen05 building blocks: D[128,N] = A[128,K] * B[N,K]^T on one CTA.
 * mode bit0: 0 = fp16, 1 = tf32 operands; bit1: 3-pass hi/lo split.  variant bit0 must be 0
 * (descriptor bring-up switch); bit1: issue the small correction passes before hi*hi; bit2 / bit3:
 * A is given as [K,128] / B as [K,N] (transposed) and consumed as an MN-major operand in place; bit4 (fp16 modes): the
 * A operand is written to TMEM with tcgen05.st and consumed by TMEM-sourced UMMAs (no shared-memory copy of A). */
int stb_tc_selftest(const float* A, const float* B, float* D, int32_t K, int32_t N, int32_t mode,
                    int32_t variant, void* stream);

/* number of kernels this library has launched from the calling thread (bench bookkeeping) */
uint64_t stb_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* STRIBOR_B200_H_ */
