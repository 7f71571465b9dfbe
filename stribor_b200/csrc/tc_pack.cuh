// What the four tensor-core families (tc_layer.cu, tc_wide.cu, tc_hwide.cu, tc_mlp.cu) do the same way around their
// kernels: the packed weight image's layout helpers and device passes, the host-side mask split and spline-coupling
// admission, the pack driver and the persistent-kernel launch.  Each family keeps its Header and offsets.
#pragma once
#include <type_traits>
#include "common.cuh"
#include "tc_common.cuh"

namespace stb {
namespace tc {

constexpr int kBins = 16;        // bins of the packed spline layout (fewer real bins: weight 0, bias -inf)
constexpr int kSplitMax = 64;    // most conditioning / transformed slots of any family (tc_wide.cu)

// ---- layout ---------------------------------------------------------------------------------------------------------
// column c of a transformed dim's 48 packed columns -> parameter index in the network's [w(K) | h(K) | rest] order, -1
// for padding: the 32 softmax columns are interleaved (w_i, h_i), i < 16; columns 32 .. 47 carry the K - 1 derivatives
// (cubic: the 2 end slopes)
__host__ __device__ __forceinline__ int param_of_col(int c, int K, int P) {
    if (c < 2 * kBins) {
        const int i = c >> 1;
        return (i < K) ? ((c & 1) ? K + i : i) : -1;
    }
    const int p = 2 * K + (c - 2 * kBins);
    return (p < P) ? p : -1;
}

// byte offset of element (r, k) of an operand with K elements per row in the core-matrix layout (tc_common.cuh)
__device__ __forceinline__ uint32_t core_off(int r, int k, int K, int elem) {
    const int epc = 16 / elem, chunks = K / epc;
    return (uint32_t)((r >> 3) * (chunks * 128) + (k / epc) * 128 + (r & 7) * 16 + (k % epc) * elem);
}

// element (n, k) of an [N x 16] K-major block: 2 chunks of 8 elements per row
__device__ __forceinline__ uint32_t blk_off(int n, int k) {
    return (uint32_t)((n >> 3) * 256 + (k >> 3) * 128 + (n & 7) * 16 + (k & 7) * 2);
}

// power of two >= max |W|, so W / s is exact and within [-1, 1] (1 when the maximum is 0, inf or NaN)
__device__ __forceinline__ float pow2_scale(float mx) {
    if (!(mx > 0.f) || !isfinite(mx)) return 1.f;
    int ex;
    const float fr = frexpf(mx, &ex);            // mx = fr * 2^ex, fr in [0.5, 1)
    return ldexpf(1.f, (fr == 0.5f) ? ex - 1 : ex);
}

// max of the warp's m into *bits (a header word zeroed before the pass): non-negative floats order like their bits
__device__ __forceinline__ void warp_max_to(uint32_t* bits, float m) {
#pragma unroll
    for (int o = 16; o; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((threadIdx.x & 31) == 0) atomicMax(bits, __float_as_uint(m));
}

// ---- the mask split -------------------------------------------------------------------------------------------------
struct MaskSplit {
    int n_cond, n_tr;
    int cond_idx[kSplitMax];     // conditioning slot -> column (0 past n_cond)
    int tr_idx[kSplitMax];       // transformed slot -> column (0 past n_tr)
};

// false without a host mask, with more conditioning / transformed columns than the family holds, or with nothing to
// transform
bool split_mask(const stb_layer* L, int max_cond, int max_tr, MaskSplit& m);

// What every tensor-core epilogue needs of a coupling: fp32 tensors (STB_F32), a hidden activation bounded by 1 (tanh, sigmoid) and the Coupling's
// inverse log-det convention.
bool tc_epilogue_ok(const stb_layer* L);

// The spline couplings the spline families (tc_layer.cu, tc_wide.cu, tc_hwide.cu) take, before their own conditioner
// shape: a quadratic or cubic spline of 2 .. 16 bins with default constants on dim <= max_dim columns, conditioned on x
// (+ latent) through an MLP with one or two hidden layers and a bounded activation, whose conditioning + latent columns
// fit GEMM1's K = k1 and whose transformed dims number <= k1.  Fills the mask split.
bool spline_gate(const stb_layer* L, int max_dim, int k1, MaskSplit& m);

// ---- device passes --------------------------------------------------------------------------------------------------
// weight of the first Linear for hidden unit n at GEMM1 slot k.  The Linear reads [x * mask | latent | t] (in_dim
// columns); the slots are [conditioning columns | t at time_col (-1: none) | latent at lat0 .. lat0 + n_lat - 1 | 0].
__device__ __forceinline__ float first_linear_w(const float* W1, int n, int k, int in_dim, int dim, const MaskSplit& m,
                                                int time_col, int lat0, int n_lat) {
    const float* row = W1 + (size_t)n * in_dim;
    if (k < m.n_cond) return row[m.cond_idx[k]];
    if (k == time_col) return row[in_dim - 1];
    if (k >= lat0 && k < lat0 + n_lat) return row[dim + (k - lat0)];
    return 0.f;
}

// W1 of the wide-conditioner families as blocks (pb = 2, 1, 0) x (kb = 0, 1), each [H x 16] of bf16 part pb
__device__ __forceinline__ void store_w1_blocks(uint8_t* w, int H, int n, int k, float v) {
    __nv_bfloat16 q[3];
    split_bf16x3(v, q[0], q[1], q[2]);
    for (int pb = 0; pb < 3; ++pb) {
        const int b = (2 - pb) * 2 + (k >> 4);
        *reinterpret_cast<__nv_bfloat16*>(w + (size_t)b * H * 32 + blk_off(n, k & 15)) = q[pb];
    }
}

// element (n, k) of an [N x K] weight as K / 16 blocks, each [N x 16] fp16 hi then [N x 16] fp16 lo
__device__ __forceinline__ void store_hilo_blocks(uint8_t* w, int N, int n, int k, float v) {
    __half hi, lo;
    split_f16(v, hi, lo);
    uint8_t* blk = w + (size_t)(k >> 4) * N * 64;
    *reinterpret_cast<__half*>(blk + blk_off(n, k & 15)) = hi;
    *reinterpret_cast<__half*>(blk + N * 32 + blk_off(n, k & 15)) = lo;
}

// the last Linear's biases of n_slots transformed slots, 48 packed columns each: softmax columns in log2 units, padded
// bins -inf (numerator 2^-inf = 0 exactly)
__device__ __forceinline__ void fill_spline_bias(float* dst, int n_slots, const float* b, const MaskSplit& m, int P,
                                                 int K, int gtid, int gsz) {
    for (int i = gtid; i < n_slots * 48; i += gsz) {
        const int ji = i / 48, col = i % 48, p = param_of_col(col, K, P);
        float bv = (ji < m.n_tr && p >= 0) ? b[m.tr_idx[ji] * P + p] : 0.f;
        if (col < 2 * kBins && p < 0 && ji < m.n_tr) bv = -INFINITY;
        dst[i] = (col < 2 * kBins) ? bv * 1.4426950408889634f : bv;
    }
}

// The softmax rows of the transformed dims for tc_bound_kernel (tc_pack.cu).
struct BoundArgs {
    const float *W, *b;          // last Linear: [dim * P, H], [dim * P]
    uint32_t* noshift;           // header words: bit ji % 32 of word ji / 32 for transformed slot ji
    int H, P, n_bins, n_tr, act;
    int tr_idx[kSplitMax];
};
__global__ void tc_bound_kernel(const BoundArgs a);

// Image of a spline coupling with an MLP[64] conditioner, shared by tc_layer.cu and tc_wide.cu:
//   Header | b1 [64] | b2 [max_tr x 48] ... | W1 at kOffW1: three bf16 parts of [64 x K1] | W2: chunks of two
//   transformed dims x 48 padded parameters x 64, fp16 hi (12 KB) | lo (12 KB), scaled by the power of two s2
struct SplinePackArgs {
    const float *W1, *b1, *W2, *b2;
    uint8_t* out;
    int kind, dim, n_chunks, P, act, n_lat, n_bins;
    MaskSplit m;
};

// F: the family's layout -- Hdr (with the fields written below), kMagic, kK1, kMaxTr, kOffB1, kOffW1 and
// header_extra(Hdr*, const SplinePackArgs&) for its own header fields.
template <class F>
__global__ void spline64_maxabs_kernel(const SplinePackArgs a) {
    float m = 0.f;
    const int total = a.m.n_tr * a.P * 64;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        const int k = i % 64, rp = i / 64, p = rp % a.P, ji = rp / a.P;
        m = fmaxf(m, fabsf(a.W2[((size_t)a.m.tr_idx[ji] * a.P + p) * 64 + k]));
    }
    warp_max_to(&reinterpret_cast<typename F::Hdr*>(a.out)->maxbits, m);
}

template <class F>
__global__ void spline64_pack_kernel(const SplinePackArgs a) {
    constexpr int kHid = 64, kChunkN = 96, kMaxChunks = F::kMaxTr / 2;
    constexpr uint32_t kW1Part = kHid * F::kK1 * 2, kOffW2 = F::kOffW1 + 3 * kW1Part, kChunkBytes = 2 * kChunkN * kHid * 2;
    auto* hdr = reinterpret_cast<typename F::Hdr*>(a.out);
    const float s2 = pow2_scale(__uint_as_float(hdr->maxbits));
    const int gtid = blockIdx.x * blockDim.x + threadIdx.x, gsz = gridDim.x * blockDim.x;
    if (gtid == 0) {
        hdr->magic = F::kMagic; hdr->kind = a.kind; hdr->dim = a.dim; hdr->n_cond = a.m.n_cond; hdr->n_tr = a.m.n_tr;
        hdr->n_chunks = a.n_chunks; hdr->P = a.P; hdr->act = a.act; hdr->s2 = s2; hdr->n_lat = a.n_lat;
        hdr->n_bins = a.n_bins;
        for (int i = 0; i < F::kK1; ++i) hdr->cond_idx[i] = a.m.cond_idx[i];
        for (int i = 0; i < F::kMaxTr; ++i) hdr->tr_idx[i] = a.m.tr_idx[i];
        F::header_extra(hdr, a);
    }
    float* b1 = reinterpret_cast<float*>(a.out + F::kOffB1);
    for (int i = gtid; i < kHid; i += gsz) b1[i] = a.b1[i];
    fill_spline_bias(b1 + kHid, F::kMaxTr, a.b2, a.m, a.P, a.n_bins, gtid, gsz);
    for (int i = gtid; i < kHid * F::kK1; i += gsz) {
        const int n = i / F::kK1, k = i % F::kK1;
        __nv_bfloat16 q0, q1, q2;
        split_bf16x3(first_linear_w(a.W1, n, k, a.dim + a.n_lat, a.dim, a.m, -1, a.m.n_cond, a.n_lat), q0, q1, q2);
        const uint32_t off = F::kOffW1 + core_off(n, k, F::kK1, 2);
        *reinterpret_cast<__nv_bfloat16*>(a.out + off) = q0;
        *reinterpret_cast<__nv_bfloat16*>(a.out + off + kW1Part) = q1;
        *reinterpret_cast<__nv_bfloat16*>(a.out + off + 2 * kW1Part) = q2;
    }
    const float inv = 1.f / s2;
    for (int i = gtid; i < kMaxChunks * kChunkN * kHid; i += gsz) {
        const int k = i % kHid, rn = i / kHid, n = rn % kChunkN, c = rn / kChunkN;
        const int ji = c * 2 + n / 48, p = param_of_col(n % 48, a.n_bins, a.P);
        float v = 0.f;
        if (c < a.n_chunks && ji < a.m.n_tr && p >= 0) v = a.W2[((size_t)a.m.tr_idx[ji] * a.P + p) * kHid + k] * inv;
        __half hi, lo;
        split_f16(v, hi, lo);
        const uint32_t off = kOffW2 + (uint32_t)c * kChunkBytes + core_off(n, k, kHid, 2);
        *reinterpret_cast<__half*>(a.out + off) = hi;
        *reinterpret_cast<__half*>(a.out + off + kChunkBytes / 2) = lo;
    }
}

inline BoundArgs spline_bound_args(const MaskSplit& m, const float* W, const float* b, int H, int P, int n_bins, int act,
                                   void* noshift) {
    BoundArgs a;
    a.W = W; a.b = b; a.noshift = static_cast<uint32_t*>(noshift);
    a.H = H; a.P = P; a.n_bins = n_bins; a.n_tr = m.n_tr; a.act = act;
    for (int i = 0; i < kSplitMax; ++i) a.tr_idx[i] = m.tr_idx[i];
    return a;
}

// ---- host: packing and launching ------------------------------------------------------------------------------------
// one pass of a pack: a counted launch
template <class A>
void pack_pass(void (*kern)(A), int grid, int block, cudaStream_t s, const A& a) {
    kern<<<grid, block, 0, s>>>(a);
    count_launch();
}

// Zero the image's first `zero_bytes` (its header: the passes accumulate maxima and noshift bits there), then run the
// family's passes in order.
template <class Passes>
int pack_image(void* out, size_t zero_bytes, cudaStream_t s, const char* what, Passes passes) {
    cudaError_t e = cudaMemsetAsync(out, 0, zero_bytes, s);
    if (e != cudaSuccess) return set_error(STB_ECUDA, "memset: %s", cudaGetErrorString(e));
    passes();
    e = cudaGetLastError();
    if (e != cudaSuccess) return set_error(STB_ECUDA, "%s launch: %s", what, cudaGetErrorString(e));
    return STB_OK;
}

// One launch of a persistent kernel: `per_sm` CTAs per multiprocessor, no more than `work` (tiles) of them.
template <class A>
int launch_persistent(void (*kern)(A), const A& args, long long work, int per_sm, int threads, uint32_t smem,
                      cudaStream_t s, const char* name) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return set_error(STB_ECUDA, "cudaFuncSetAttribute: %s", cudaGetErrorString(e));
    const int grid = (int)min((long long)per_sm * sm_count(), work);
    kern<<<grid, threads, smem, s>>>(args);
    count_launch();
    e = cudaGetLastError();
    if (e != cudaSuccess) return set_error(STB_ECUDA, "%s launch: %s", name, cudaGetErrorString(e));
    return STB_OK;
}

// The kernel variant for a spline kind and direction (and one more flag): f(Kind, Inverse[, Flag]) gets each as a
// std::integral_constant and names the instantiation, e.g. [](auto K, auto I) { return my_kernel<K, I>; }.
template <class F>
auto pick_variant(int kind, bool inverse, F f) {
    using Rqs = std::integral_constant<int, STB_RQS>;
    using Cubic = std::integral_constant<int, STB_CUBIC>;
    if (kind == STB_RQS) return inverse ? f(Rqs{}, std::true_type{}) : f(Rqs{}, std::false_type{});
    return inverse ? f(Cubic{}, std::true_type{}) : f(Cubic{}, std::false_type{});
}
template <class F>
auto pick_variant(int kind, bool inverse, bool flag, F f) {
    return flag ? pick_variant(kind, inverse, [&](auto k, auto i) { return f(k, i, std::true_type{}); })
                : pick_variant(kind, inverse, [&](auto k, auto i) { return f(k, i, std::false_type{}); });
}

}  // namespace tc
}  // namespace stb
