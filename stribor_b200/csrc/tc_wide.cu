// Tensor-core coupling layer for dim <= 128 and its training backward (sm_100a, tcgen05 + TMEM).
//
// Scope: st.Coupling(st.Spline(dim <= 128, n_bins = 16 (forward: 2..16), 'quadratic' | 'cubic',
// latent_net = MLP(dim (+ latent, forward only), [64], dim * P)), mask) with <= 64 conditioning (+ latent) columns and
// <= 64 transformed dims -- BASELINE.json configs[4] (d = 128) -- in three modes:
//   FWD  y = T(x) or T^-1(x), per-row log|det J|          (flows/coupling.py:69-95, as tc_layer.cu)
//   BWD  the gradient of that application from its saved input: recomputes the conditioner on the
//        tensor cores, differentiates the spline element in registers and writes
//          g_x  [rows, dim]          transformed dims; pass-through dims carry g_out (the conditioner's
//                                    contribution to them is added by the caller from g_net / hidden)
//          g_net [rows, n_tr * 48]   gradient wrt the network output of the transformed dims, natural
//                                    parameter order [w(16) | h(16) | d(15) | 0] per dim
//          hidden [rows, 72]         the conditioner's hidden activations | 1 | 0 x 7 (augmented so that
//                                    g_net^T hidden = [gW | gb] of the last Linear in one product)
//        (what autograd derives for util/rational_quadratic_spline.py + flows/coupling.py)
//
// One persistent CTA per SM, 18 warps, tiles of 128 rows:
//   warp 0      producer: streams the packed first Linear (24 KB) and then the last-Linear chunks
//               (24 KB = 2 transformed dims x 48 padded parameters x 64, fp16 hi | lo) through one
//               3-stage cp.async.bulk ring
//   warp 1      UMMA issuer: GEMM1 [128 x K1] x [K1 x 64] as bf16x3 split products, GEMM2
//               [128 x 64] x [64 x 96] per chunk as 3 fp16 passes; accumulators in TMEM
//   warps 2-17  loader + epilogue: the x tile is split on the fly (conditioning columns -> bf16x3 A
//               operand, transformed columns -> smem), tanh of GEMM1 -> fp16 hi | lo A operand of
//               GEMM2, then thread = row: 48 parameters of one element out of TMEM, spline (or its
//               gradient) in registers.
#include <stdlib.h>
#include "common.cuh"
#include "stb_math.cuh"
#include "tc_common.cuh"
#include "tc_pack.cuh"
#include "tc_spline16.cuh"

namespace stb {
using namespace tc;

namespace tcw {
using namespace sp16;

constexpr int kHid = 64;
constexpr int kK1 = 64;              // max conditioning columns (GEMM1 K)
constexpr int kPPad = 48;
constexpr int kG = 2;
constexpr int kChunkN = kG * kPPad;  // 96
constexpr int kMaxDim = 128;
constexpr int kMaxTr = 64;
constexpr int kMaxChunks = kMaxTr / kG;
constexpr int kTileRows = 128;
constexpr int kTrStride = kMaxTr + 1;
constexpr int kStages = 3;
constexpr int kEpiWarps = 16;
constexpr int kEpiWarp0 = 2;
constexpr int kThreads = (kEpiWarp0 + kEpiWarps) * 32;
constexpr int kEpiThreads = kEpiWarps * 32;
constexpr int kHAug = 72;            // row of the hidden-activation output: h(64) | 1 | 0 x 7

constexpr uint32_t kMagic = 0x53544257u;
struct Header {                      // 2048 bytes
    uint32_t magic;
    int32_t kind, dim, n_cond, n_tr, n_chunks, P, act, k1pad;
    float s2;
    uint32_t maxbits;
    uint32_t noshift_mask[2];
    int32_t n_lat;                   // `latent=` columns: conditioning slots n_cond .. n_cond + n_lat - 1 (forward kernels only)
    uint32_t m_d, m_d4;              // division magics (div_magic) of dim, dim / 4 ...
    int32_t cond_idx[kK1];           // conditioning slot -> column
    int32_t tr_idx[kMaxTr];          // transformed slot -> column
    int16_t colmap[kMaxDim];         // column -> slot: >= 0 conditioning slot, < 0: -(transformed slot) - 1
    uint32_t m_ntr, m_npad, m_npad64; // ... n_tr, k1pad - n_cond - n_lat, 64 - n_cond
    int32_t n_bins;                  // 2 .. 16 real bins in the padded 16-bin layout (forward kernels; the gradient kernels need 16)
    int32_t pad1[512 - 20 - kK1 - kMaxTr - kMaxDim / 2];
};
static_assert(sizeof(Header) == 2048, "header layout");
constexpr uint32_t kOffB1 = 2048;                                  // float[64]
constexpr uint32_t kOffB2 = kOffB1 + kHid * 4;                     // float[kMaxChunks * 96]
constexpr uint32_t kSmallBytes = kOffB2 + kMaxChunks * kChunkN * 4;
constexpr uint32_t kOffW1 = 16384;                                 // 3 bf16 parts of [64][64], 8 KB each
constexpr uint32_t kW1Part = kHid * kK1 * 2;
constexpr uint32_t kChunkBytes = 2 * kChunkN * kHid * 2;           // 24576
static_assert(3 * kW1Part == kChunkBytes, "the first Linear travels through the chunk ring");
constexpr uint32_t kOffW2 = kOffW1 + kChunkBytes;
constexpr uint32_t kPackedBytes = kOffW2 + kMaxChunks * kChunkBytes;
static_assert(kSmallBytes % 16 == 0 && kSmallBytes <= kOffW1, "small block");

constexpr uint32_t kA1Part = kTileRows * kK1 * 2;                  // 16384
// shared memory map
constexpr uint32_t kSmXs = 0;                                      // float [128][65]  transformed columns of x
constexpr uint32_t kSmGs = kSmXs + kTileRows * kTrStride * 4;      // float [128][65]  same of g_out (BWD)
constexpr uint32_t kSmA = (kSmGs + kTileRows * kTrStride * 4 + 1023) & ~1023u;   // 48 KB: A1 bf16x3 / h fp16 hi | lo
constexpr uint32_t kABytes = 3 * kA1Part;
constexpr uint32_t kSmB = kSmA + kABytes;
constexpr uint32_t kSmSmall = kSmB + kStages * kChunkBytes;
constexpr uint32_t kSmBar = (kSmSmall + kSmallBytes + 15) & ~15u;
constexpr uint32_t kSmLd = kSmBar + 256;                           // float [3][128]
constexpr uint32_t kSmemBytes = kSmLd + 3 * kTileRows * 4;
static_assert(kSmemBytes <= 227 * 1024, "shared memory budget");

struct Bars {
    uint64_t setup;
    uint64_t b_full[kStages], b_empty[kStages];
    uint64_t a1_ready, acc1_full, h_ready;
    uint64_t acc_full[2], acc_empty[2];
    uint32_t tmem_base;
};
static_assert(sizeof(Bars) <= 256, "barrier block");

constexpr uint32_t kColAcc1 = 0;
constexpr uint32_t kColAcc2 = 128;               // + buf * 96
constexpr uint32_t kTmemCols = 512;

struct Args {
    const uint8_t* packed;
    const float* x;
    float* y;                 // FWD: output rows; BWD: g_x
    float* ldj;
    int ldj_mode;
    int base_log_prob;
    float lower, upper;
    long long rows;
    int n_tiles;
    // BWD
    const float* g_out;
    const float* g_ldj;
    float* g_net;
    float* hidden;
    int32_t* bins;            // FWD, optional: [rows, dim] searched bin per element (stb_layer_apply_bins)
    const float* latent;      // FWD, optional: [rows, n_lat]
};

// i / dv for 0 <= i < 2^16, 1 <= dv <= 2^7 with a precomputed magic = ceil(2^32 / dv): exact (i * (magic * dv - 2^32) <
// 2^23), one IMAD.HI instead of the ~20-instruction runtime division in the tile staging loops
// (dv == 1: the magic 2^32 does not fit and is stored as 0 = "divide by one")
__device__ __forceinline__ uint32_t div_magic(int dv) { return (uint32_t)((0x100000000ull + (uint32_t)dv - 1) / (uint32_t)dv); }
__device__ __forceinline__ int fast_div(int i, uint32_t magic) { return magic ? (int)__umulhi((uint32_t)i, magic) : i; }
__device__ __forceinline__ void stg256(float* p, const float* v) {
    asm volatile("st.global.v8.f32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(p), "f"(v[0]), "f"(v[1]), "f"(v[2]),
                 "f"(v[3]), "f"(v[4]), "f"(v[5]), "f"(v[6]), "f"(v[7])
                 : "memory");
}

// One conditioning value -> its three bf16 parts at (row r, slot m) of the A1 operand (K-major core-matrix
// layout, 64 slots: 1024 B per 8-row group, 128 B per 8-slot group)
__device__ __forceinline__ uint8_t* a1_addr(uint8_t* abuf, int r, int m) {
    return abuf + (uint32_t)(r >> 3) * 1024 + (uint32_t)(m >> 3) * 128 + (uint32_t)(r & 7) * 16 + (uint32_t)(m & 7) * 2;
}
__device__ __forceinline__ void a1_put(uint8_t* abuf, int r, int m, float v) {
    __nv_bfloat16 p0, p1, p2;
    split_bf16x3(v, p0, p1, p2);
    uint8_t* dst = a1_addr(abuf, r, m);
    *reinterpret_cast<__nv_bfloat16*>(dst) = p0;
    *reinterpret_cast<__nv_bfloat16*>(dst + kA1Part) = p1;
    *reinterpret_cast<__nv_bfloat16*>(dst + 2 * kA1Part) = p2;
}
// four consecutive slots (m % 4 == 0): 8-byte stores
__device__ __forceinline__ void a1_put4(uint8_t* abuf, int r, int m, const float4& v) {
    __align__(8) __nv_bfloat16 q0[4], q1[4], q2[4];
    split_bf16x3(v.x, q0[0], q1[0], q2[0]); split_bf16x3(v.y, q0[1], q1[1], q2[1]);
    split_bf16x3(v.z, q0[2], q1[2], q2[2]); split_bf16x3(v.w, q0[3], q1[3], q2[3]);
    uint8_t* dst = a1_addr(abuf, r, m);
    *reinterpret_cast<uint2*>(dst) = *reinterpret_cast<const uint2*>(q0);
    *reinterpret_cast<uint2*>(dst + kA1Part) = *reinterpret_cast<const uint2*>(q1);
    *reinterpret_cast<uint2*>(dst + 2 * kA1Part) = *reinterpret_cast<const uint2*>(q2);
}
__device__ __forceinline__ void a1_zero(uint8_t* abuf, int r, int m) {
    uint8_t* dst = a1_addr(abuf, r, m);
    *reinterpret_cast<uint16_t*>(dst) = 0;
    *reinterpret_cast<uint16_t*>(dst + kA1Part) = 0;
    *reinterpret_cast<uint16_t*>(dst + 2 * kA1Part) = 0;
}

// FULL = false (forward only): 2 .. 15 real bins in the padded 16-bin layout (tc_spline16.cuh)
template <int KIND, bool INVERSE, bool BWD, bool FULL = true>
__global__ void __launch_bounds__(kThreads, 1) tc_wide_kernel(const Args A) {
    extern __shared__ __align__(1024) uint8_t smem[];
    float* xs = reinterpret_cast<float*>(smem + kSmXs);
    float* gs = reinterpret_cast<float*>(smem + kSmGs);
    uint8_t* abuf = smem + kSmA;
    uint8_t* bst = smem + kSmB;
    const Header* hdr = reinterpret_cast<const Header*>(smem + kSmSmall);
    const float* b1s = reinterpret_cast<const float*>(smem + kSmSmall + kOffB1);
    const float* b2s = reinterpret_cast<const float*>(smem + kSmSmall + kOffB2);
    Bars* bars = reinterpret_cast<Bars*>(smem + kSmBar);
    float* ld_s = reinterpret_cast<float*>(smem + kSmLd);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

    if (tid == 0) {
        mbar_init(&bars->setup, 1);
        for (int i = 0; i < kStages; ++i) { mbar_init(&bars->b_full[i], 1); mbar_init(&bars->b_empty[i], 1); }
        mbar_init(&bars->a1_ready, kEpiWarps);
        mbar_init(&bars->acc1_full, 1);
        mbar_init(&bars->h_ready, kEpiWarps);
        for (int b = 0; b < 2; ++b) { mbar_init(&bars->acc_full[b], 1); mbar_init(&bars->acc_empty[b], 8); }
        fence_mbar_init();
    }
    __shared__ uint32_t tmem_base_s;      // own word: the allocator writes it, keep it away from the mbarrier block
    if (warp == 1) tmem_alloc(&tmem_base_s, kTmemCols);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_base_s;

    if (tid == 0) {
        mbar_arrive_expect_tx(&bars->setup, kSmallBytes);
        bulk_g2s(smem + kSmSmall, A.packed, kSmallBytes, &bars->setup);
    }
    mbar_wait(&bars->setup, 0);

    const int d = hdr->dim, n_tr = hdr->n_tr, n_cond = hdr->n_cond, n_chunks = hdr->n_chunks;
    const int k1pad = hdr->k1pad;
    const int K = FULL ? kBins : hdr->n_bins;
    const int act = hdr->act;
    const float s2 = hdr->s2;
    const float s2l = s2 * 1.4426950408889634f;
    const int my_tiles = (A.n_tiles > (int)blockIdx.x) ? (A.n_tiles - 1 - (int)blockIdx.x) / (int)gridDim.x + 1 : 0;

    if (warp == 0) {
        // ======================= producer =========================================================
        if (lane == 0) {
            uint32_t cc = 0;
            for (int it = 0; it < my_tiles; ++it) {
                for (int c = -1; c < n_chunks; ++c, ++cc) {       // item -1: the packed first Linear
                    const uint32_t st = cc % kStages, use = cc / kStages;
                    mbar_wait_relaxed(&bars->b_empty[st], (use & 1) ^ 1);
                    mbar_arrive_expect_tx(&bars->b_full[st], kChunkBytes);
                    const uint8_t* src = (c < 0) ? A.packed + kOffW1 : A.packed + kOffW2 + (size_t)c * kChunkBytes;
                    bulk_g2s(bst + st * kChunkBytes, src, kChunkBytes, &bars->b_full[st]);
                }
            }
        }
    } else if (warp == 1) {
        // ======================= UMMA issuer ======================================================
        if (lane == 0) {
            const uint32_t idesc1 = make_idesc(FMT_BF16, 128, kHid);
            const uint32_t idesc2 = make_idesc(FMT_F16, 128, kChunkN);
            uint32_t cc = 0, cb = 0;
            for (int it = 0; it < my_tiles; ++it) {
                const uint32_t tpar = it & 1;
                {
                    const uint32_t st = cc % kStages, use = cc / kStages;
                    mbar_wait_relaxed(&bars->b_full[st], use & 1);
                    mbar_wait_relaxed(&bars->a1_ready, tpar);
                    tc_fence_after();
                    const uint32_t a0 = smem_u32(abuf), b0 = smem_u32(bst + st * kChunkBytes);
                    const uint32_t dcol = tmem + kColAcc1;
                    uint32_t acc = 0;
                    // x = x0 + x1 + x2, W = W0 + W1 + W2 (bf16 parts): every product except x2*W2, smallest
                    // first (the tensor core truncates the running accumulator at every step)
#pragma unroll
                    for (int p = 0; p < 8; ++p) {
                        const int pa = (p == 0 || p == 3 || p == 6) ? 1 : ((p == 1 || p == 4) ? 2 : 0);
                        const int pb = (p == 0 || p == 2) ? 2 : ((p == 1 || p == 3 || p == 5) ? 1 : 0);
                        for (int ks = 0; ks < k1pad / 16; ++ks) {
                            umma_f16(dcol, make_smem_desc(a0 + pa * kA1Part + ks * 256, 128, 1024),
                                     make_smem_desc(b0 + pb * kW1Part + ks * 256, 128, 1024), idesc1, acc);
                            acc = 1;
                        }
                    }
                    umma_commit(&bars->acc1_full);
                    umma_commit(&bars->b_empty[st]);
                    ++cc;
                }
                for (int c = 0; c < n_chunks; ++c, ++cc, ++cb) {
                    const uint32_t st = cc % kStages, use = cc / kStages;
                    mbar_wait_relaxed(&bars->b_full[st], use & 1);
                    const uint32_t buf = cb & 1, buse = cb >> 1;
                    if (c == 0) mbar_wait_relaxed(&bars->h_ready, tpar);
                    mbar_wait_relaxed(&bars->acc_empty[buf], (buse & 1) ^ 1);
                    tc_fence_after();
                    const uint32_t a_hi = smem_u32(abuf), a_lo = a_hi + 16384;
                    const uint32_t b_hi = smem_u32(bst + st * kChunkBytes), b_lo = b_hi + 12288;
                    const uint32_t dcol = tmem + kColAcc2 + buf * kChunkN;
                    uint32_t acc = 0;
#pragma unroll
                    for (int p = 0; p < 3; ++p) {                  // lo*hi, hi*lo, then hi*hi
                        const uint32_t aa = (p == 0) ? a_lo : a_hi, bb = (p == 1) ? b_lo : b_hi;
#pragma unroll
                        for (int ks = 0; ks < kHid / 16; ++ks) {
                            umma_f16(dcol, make_smem_desc(aa + ks * 256, 128, 1024),
                                     make_smem_desc(bb + ks * 256, 128, 1024), idesc2, acc);
                            acc = 1;
                        }
                    }
                    umma_commit(&bars->acc_full[buf]);
                    umma_commit(&bars->b_empty[st]);
                }
            }
        }
    } else {
        // ======================= loader + epilogue warps ==========================================
        const int q = warp & 3;                                  // TMEM sub-partition of this warp
        const int r4 = (warp - kEpiWarp0) >> 2;                  // 0..3 within the sub-partition
        const int etid = tid - kEpiWarp0 * 32;
        const int rloc = q * 32 + lane;                          // row within the tile == TMEM lane
        const uint32_t a_row_off = (uint32_t)(rloc >> 3) * 1024 + (uint32_t)(rloc & 7) * 16;
        const uint32_t lane_sel = (uint32_t)(q * 32) << 16;
        const bool want_ld = A.ldj_mode != STB_LDJ_NONE;
        const float lo = A.lower, hi = A.upper;
        const float inv_span = 1.f / (hi - lo);
        uint32_t cb = 0;

        for (int it = 0; it < my_tiles; ++it) {
            const long long tile = (long long)blockIdx.x + (long long)it * gridDim.x;
            const long long row0 = tile * kTileRows;
            const int nrows = (int)min((long long)kTileRows, A.rows - row0);
            const uint32_t tpar = it & 1;

            // ---- load the tile: conditioning columns -> bf16x3 A operand, transformed columns -> smem,
            // pass-through columns of the output copied through registers ------------------------------
            {
                const float* xg = A.x + row0 * d;
                const float* gg = BWD ? A.g_out + row0 * d : nullptr;
                float* og = A.y + row0 * d;
                const bool copy_pass = BWD ? (static_cast<const float*>(A.y) != A.g_out)
                                           : (static_cast<const float*>(A.y) != A.x);
                const bool vec = ((d & 3) == 0) && ((reinterpret_cast<uintptr_t>(xg) & 15) == 0) &&
                                 (!BWD || (reinterpret_cast<uintptr_t>(gg) & 15) == 0) &&
                                 ((reinterpret_cast<uintptr_t>(og) & 15) == 0);
                if (vec) {
                    const int d4 = d >> 2, n4 = kTileRows * d4;
                    // four 16-byte loads in flight per thread before the first is consumed (one at a time, the
                    // loop was a chain of exposed global round trips: 21 % of this kernel's stall samples)
                    for (int i0 = etid; i0 < n4; i0 += kEpiThreads * 4) {
                      float4 vb[4], gb[4];
#pragma unroll
                      for (int u4 = 0; u4 < 4; ++u4) {
                        const int i = i0 + u4 * kEpiThreads;
                        const bool live = i < n4 && fast_div(i, hdr->m_d4) < nrows;
                        vb[u4] = live ? __ldg(reinterpret_cast<const float4*>(xg) + i) : make_float4(0.f, 0.f, 0.f, 0.f);
                        gb[u4] = (BWD && live) ? __ldg(reinterpret_cast<const float4*>(gg) + i) : make_float4(0.f, 0.f, 0.f, 0.f);
                      }
#pragma unroll
                      for (int u4 = 0; u4 < 4; ++u4) {
                        const int i = i0 + u4 * kEpiThreads;
                        if (i >= n4) break;
                        const int r = fast_div(i, hdr->m_d4), c = (i - r * d4) << 2;
                        const bool live = r < nrows;
                        const float4 v = vb[u4], gv = gb[u4];
                        const int m0 = hdr->colmap[c], m1 = hdr->colmap[c + 1], m2 = hdr->colmap[c + 2], m3 = hdr->colmap[c + 3];
                        if (m0 >= 0 && (m0 & 3) == 0 && m1 == m0 + 1 && m2 == m0 + 2 && m3 == m0 + 3) {
                            // four consecutive conditioning slots: 8-byte stores into the core-matrix layout
                            a1_put4(abuf, r, m0, v);
                            if (copy_pass && live) reinterpret_cast<float4*>(og)[i] = BWD ? gv : v;
                        } else {
                            const float vv[4] = {v.x, v.y, v.z, v.w};
                            const float gvv[4] = {gv.x, gv.y, gv.z, gv.w};
                            const int mm[4] = {m0, m1, m2, m3};
#pragma unroll
                            for (int u = 0; u < 4; ++u) {
                                if (mm[u] >= 0) {
                                    a1_put(abuf, r, mm[u], vv[u]);
                                    if (copy_pass && live) og[(size_t)r * d + c + u] = BWD ? gvv[u] : vv[u];
                                } else {
                                    const int sl = -mm[u] - 1;
                                    xs[r * kTrStride + sl] = vv[u];
                                    if (BWD) gs[r * kTrStride + sl] = gvv[u];
                                }
                            }
                        }
                      }
                    }
                } else {
                    const int n = kTileRows * d;
                    for (int i = etid; i < n; i += kEpiThreads) {
                        const int r = fast_div(i, hdr->m_d), c = i - r * d;
                        const bool live = r < nrows;
                        const float v = live ? __ldg(xg + i) : 0.f;
                        const float gv = (BWD && live) ? __ldg(gg + i) : 0.f;
                        const int m = hdr->colmap[c];
                        if (m >= 0) {
                            a1_put(abuf, r, m, v);
                            if (copy_pass && live) og[i] = BWD ? gv : v;
                        } else {
                            xs[r * kTrStride - m - 1] = v;
                            if (BWD) gs[r * kTrStride - m - 1] = gv;
                        }
                    }
                }
                // `latent=` columns (coupling.py:64-65): conditioning slots n_cond .. n_cond + n_lat - 1
                const int n_lat = hdr->n_lat;
                for (int i = etid; i < kTileRows * n_lat; i += kEpiThreads) {
                    const int r = i / n_lat, j = i - r * n_lat;
                    a1_put(abuf, r, n_cond + j, (r < nrows) ? __ldg(A.latent + (row0 + r) * n_lat + j) : 0.f);
                }
                // zero the padded conditioning slots [n_cond + n_lat, k1pad) (the buffer is reused for h every tile)
                const int npad = k1pad - n_cond - n_lat;
                const uint32_t m_npad = hdr->m_npad;
                for (int i = etid; i < kTileRows * npad; i += kEpiThreads) {
                    const int r = fast_div(i, m_npad), m = n_cond + n_lat + (i - r * npad);
                    a1_zero(abuf, r, m);
                }
            }
            fence_proxy_async_smem();
            named_bar_sync(1, kEpiThreads);
            if (lane == 0) mbar_arrive(&bars->a1_ready);

            // ---- hidden layer: h = act(acc1 + b1) -> fp16 hi | lo A operand of GEMM2 --------------------
            mbar_wait_sleep(&bars->acc1_full, tpar, 64);
            tc_fence_after();
#pragma unroll 1
            for (int kc = r4; kc < kHid / 8; kc += 4) {
                const int c0 = kc * 8;
                float v[8];
                tmem_ld8(tmem + lane_sel + kColAcc1 + c0, v);
                tmem_ld_wait();
                __align__(16) __half hh[8], hl[8];
                if (act == STB_ACT_TANH) {
#pragma unroll
                    for (int i = 0; i < 8; ++i) v[i] = tanh_fast(v[i] + b1s[c0 + i]);
                } else {
#pragma unroll
                    for (int i = 0; i < 8; ++i) v[i] = sigmoid_act(v[i] + b1s[c0 + i]);          // STB_ACT_SIGMOID
                }
#pragma unroll
                for (int i = 0; i < 8; ++i) split_f16(v[i], hh[i], hl[i]);
                *reinterpret_cast<uint4*>(abuf + a_row_off + kc * 128) = *reinterpret_cast<const uint4*>(hh);
                *reinterpret_cast<uint4*>(abuf + 16384 + a_row_off + kc * 128) = *reinterpret_cast<const uint4*>(hl);
                if (BWD && rloc < nrows) stg256(A.hidden + (size_t)(row0 + rloc) * kHAug + c0, v);
            }
            if (BWD && r4 == 0 && rloc < nrows) {                // augmentation: g_net^T [h | 1] = [gW | gb]
                const float one[8] = {1.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
                stg256(A.hidden + (size_t)(row0 + rloc) * kHAug + kHid, one);
            }
            tc_fence_before();
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) mbar_arrive(&bars->h_ready);

            // ---- chunks out of TMEM: this warp's dim of every second chunk ---------------------------------
            float ld_acc = 0.f;
            float g_ld = 0.f;
            if (BWD && A.g_ldj != nullptr && rloc < nrows) g_ld = __ldg(A.g_ldj + row0 + rloc);
            float* xrow = xs + rloc * kTrStride;
            float* grow = gs + rloc * kTrStride;
#pragma unroll 1
            for (int ji = r4; ji < kG * n_chunks; ji += 4) {
                const uint32_t ccc = cb + (uint32_t)(ji >> 1);
                const uint32_t buf = ccc & 1, buse = ccc >> 1;
                const int g = ji & 1;
                const bool live_dim = ji < n_tr;
                const float xv = live_dim ? xrow[ji] : 0.f;
                const bool inside = live_dim && (xv >= lo) && (xv <= hi);
                const float* bb = b2s + ji * kPPad;
                const float2* bb2 = reinterpret_cast<const float2*>(bb);
                mbar_wait_sleep(&bars->acc_full[buf], buse & 1, 32);
                tc_fence_after();
                const uint32_t col0 = tmem + lane_sel + kColAcc2 + buf * kChunkN + (uint32_t)g * kPPad;
                const bool shift = !((hdr->noshift_mask[ji >> 5] >> (ji & 31)) & 1u);
                float out = xv, ld = 0.f;
                if (KIND == STB_RQS) {
                    float2 t[kBins];
                    tmem_ld16(col0, reinterpret_cast<float*>(t));
                    tmem_ld16(col0 + 16, reinterpret_cast<float*>(t) + 16);
                    tmem_ld_wait();
#pragma unroll
                    for (int i = 0; i < kBins; ++i) t[i] = __ffma2_rn(t[i], f2(s2l), bb2[i]);
                    if (!BWD) {
                        const RqsLoc loc = rqs16_locate<INVERSE, FULL>(t, shift, lo, inv_span, xv, K);
                        float dd[16];
                        tmem_ld16(col0 + 2 * kBins, dd);
                        tmem_ld_wait();
                        tc_fence_before();
                        __syncwarp();
                        if (lane == 0) mbar_arrive(&bars->acc_empty[buf]);
                        if (inside) {
                            float r0, r1;
                            pick_pair16(dd, loc.k, r0, r1);
                            const float u0 = (loc.k == 0) ? STB_RQS_EDGE_CONST : fmaf(r0, s2, bb[2 * kBins + loc.k - 1]);
                            const float u1 = (loc.k == K - 1) ? STB_RQS_EDGE_CONST : fmaf(r1, s2, bb[2 * kBins + loc.k]);
                            rqs16_finish<INVERSE>(loc, u0, u1, lo, hi, want_ld, xv, out, ld, K);
                        }
                        if (A.bins != nullptr && live_dim && rloc < nrows)
                            A.bins[(row0 + rloc) * d + hdr->tr_idx[ji]] = inside ? loc.k : -1;
                    } else {
                        softmax16_num2(t, shift);
                        float2 ee, eo;
                        const BinSearch16 bs = bin_search16<INVERSE>(t, STB_RQS_MIN, (xv - lo) * inv_span, ee, eo);
                        float dd[16];
                        tmem_ld16(col0 + 2 * kBins, dd);
                        tmem_ld_wait();
                        tc_fence_before();
                        __syncwarp();
                        if (lane == 0) mbar_arrive(&bars->acc_empty[buf]);
                        float r0, r1;
                        pick_pair16(dd, bs.k, r0, r1);
                        const int kk = bs.k;
                        const float u0 = (kk == 0) ? STB_RQS_EDGE_CONST : fmaf(r0, s2, bb[2 * kBins + (kk > 0 ? kk - 1 : 0)]);
                        const float u1 = (kk == kBins - 1) ? STB_RQS_EDGE_CONST : fmaf(r1, s2, bb[2 * kBins + (kk < kBins - 1 ? kk : 0)]);
                        const float go = live_dim ? grow[ji] : 0.f;
                        float gx = go, gu0 = 0.f, gu1 = 0.f;
                        if (inside) {
                            rqs16_backward<INVERSE>(t, bs, ee, eo, u0, u1, lo, hi, xv, go, g_ld, gx, gu0, gu1);
                        } else {
#pragma unroll
                            for (int i = 0; i < kBins; ++i) t[i] = f2(0.f);
                        }
                        out = gx;
                        if (live_dim && rloc < nrows) {
                            float* gp = A.g_net + ((size_t)(row0 + rloc) * n_tr + ji) * kPPad;
                            float w[8];
#pragma unroll
                            for (int b8 = 0; b8 < 2; ++b8) {               // widths, then heights
#pragma unroll
                                for (int i = 0; i < 8; ++i) w[i] = t[b8 * 8 + i].x;
                                stg256(gp + b8 * 8, w);
                            }
#pragma unroll
                            for (int b8 = 0; b8 < 2; ++b8) {
#pragma unroll
                                for (int i = 0; i < 8; ++i) w[i] = t[b8 * 8 + i].y;
                                stg256(gp + kBins + b8 * 8, w);
                            }
#pragma unroll
                            for (int b8 = 0; b8 < 2; ++b8) {               // derivative i sits at knot i + 1
#pragma unroll
                                for (int i = 0; i < 8; ++i) {
                                    const int di = b8 * 8 + i;
                                    w[i] = (di == kk - 1) ? gu0 : ((di == kk) ? gu1 : 0.f);
                                    if (di == kBins - 1) w[i] = 0.f;       // padding column
                                }
                                stg256(gp + 2 * kBins + b8 * 8, w);
                            }
                        }
                    }
                } else {
                    const float span = hi - lo;
                    const float u = (xv - lo) / span;
                    float2 t[kBins];
                    tmem_ld16(col0, reinterpret_cast<float*>(t));
                    tmem_ld16(col0 + 16, reinterpret_cast<float*>(t) + 16);
                    tmem_ld_wait();
#pragma unroll
                    for (int i = 0; i < kBins; ++i) t[i] = __ffma2_rn(t[i], f2(s2l), bb2[i]);
                    const CubSel sel = cubic16_locate<INVERSE, FULL>(t, shift, u, K);
                    float dd[8];
                    tmem_ld8(col0 + 2 * kBins, dd);
                    tmem_ld_wait();
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&bars->acc_empty[buf]);
                    if (inside) {
                        const float ul = fmaf(dd[0], s2, bb[2 * kBins]), ur = fmaf(dd[1], s2, bb[2 * kBins + 1]);
                        cubic16_finish<INVERSE>(sel, ul, ur, lo, hi, want_ld, u, out, ld, K);
                    }
                    if (!BWD && A.bins != nullptr && live_dim && rloc < nrows)
                        A.bins[(row0 + rloc) * d + hdr->tr_idx[ji]] = inside ? sel.k : -1;
                }
                if (live_dim) {
                    if (BWD) grow[ji] = out; else xrow[ji] = out;
                }
                ld_acc += ld;
            }
            cb += (uint32_t)n_chunks;

            // ---- per-row log|det J| (+ UnitNormal log-density of the output row) ---------------------------
            if (!BWD && r4 < 3) ld_s[r4 * kTileRows + rloc] = ld_acc;
            named_bar_sync(1, kEpiThreads);
            if (!BWD && r4 == 3 && want_ld && rloc < nrows) {           // fixed summation order: deterministic
                float tot = ld_s[rloc] + ld_s[kTileRows + rloc] + ld_s[2 * kTileRows + rloc] + ld_acc;
                if (A.base_log_prob) {
                    const float* xr = A.x + (row0 + rloc) * d;            // pass-through columns: unchanged by this layer
                    float b = 0.f;
                    for (int c = 0; c < d; ++c) {
                        const int m = hdr->colmap[c];
                        const float v = (m >= 0) ? __ldg(xr + c) : xrow[-m - 1];
                        b += -0.5f * v * v - 0.91893853320467274178f;
                    }
                    tot += b;
                }
                float* dst = A.ldj + row0 + rloc;
                *dst = (A.ldj_mode == STB_LDJ_ADD) ? (*dst + tot) : tot;
            }
            // ---- transformed columns out ---------------------------------------------------------------------
            {
                float* og = A.y + row0 * d;
                const float* src = BWD ? gs : xs;
                for (int i = etid; i < nrows * n_tr; i += kEpiThreads) {
                    const int r = fast_div(i, hdr->m_ntr), sl = i - r * n_tr;
                    og[(size_t)r * d + hdr->tr_idx[sl]] = src[r * kTrStride + sl];
                }
            }
            named_bar_sync(1, kEpiThreads);
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem, kTmemCols);
}

// -----------------------------------------------------------------------------------------------
// training backward with the conditioner's gradient products fused
// -----------------------------------------------------------------------------------------------
// Same recompute as BWD above; the per-element gradient g_net never leaves the SM.  Per chunk
// (2 transformed dims x 48 parameters) the epilogue warps write it, scaled by a per-tile power of two
// and split fp16 hi | lo, into ONE shared K-major buffer G [128 rows x 96], and the issuer runs two more
// groups of UMMAs on it, both with operands that are MN-major VIEWS of buffers the forward needs anyway:
//   g_hidden [128 x 64] += G [128 x 96] . W2chunk [96 x 64]      A = G K-major, B = the ring stage MN-major
//   gW2chunk [96 x 64 | gb2] = G^T [96 x 128] . [h | 1] [128 x 80]  A = G MN-major, B = the h operand MN-major
// g_hidden accumulates in TMEM over the tile's chunks and becomes g_pre = g_hidden * act'(h) [rows, 64];
// the per-(tile, chunk) gW2 partials are added to a [n_chunks * 96, 72] fp32 image in global memory
// (L2-resident, red.global.add.v4.f32) -- summation order over tiles is not deterministic.
// At the tile end the first Linear's products follow (g_w1 != NULL): g_x[cond] = g_out[cond] + g_pre W1[:, cond],
// gW1 += g_pre^T x_cond (bf16x3 operands, MN-major views again), gb1 by warp shuffles; otherwise g_pre is written
// and those three K = 64 products are left to the caller.
namespace train {
constexpr int kTEpiWarp0 = 3;                                     // warp 0 producer, warps 1 / 2 UMMA issuers (F / G)
constexpr int kTThreads = (kTEpiWarp0 + kEpiWarps) * 32;          // 608
constexpr int kHPad = 80;                                         // h operand columns: 64 hidden | 1 | 0 x 15
constexpr uint32_t kHSbo = (kHPad / 8) * 128;                     // 1280: next 8 rows of the h operand
constexpr uint32_t kHLo = kTileRows * kHPad * 2;                  // 20480: lo part
constexpr uint32_t kGSbo = (kChunkN / 8) * 128;                   // 1536: next 8 rows of G
constexpr uint32_t kGLo = kTileRows * kChunkN * 2;                // 24576
constexpr int kWStride = 72;                                      // floats per row of the gW2 image
constexpr uint32_t kSmXs = 0;
constexpr uint32_t kSmA = (kTileRows * kTrStride * 4 + 1023) & ~1023u;
constexpr uint32_t kSmG = kSmA + kABytes;
constexpr uint32_t kSmB = kSmG + 2 * kGLo;
constexpr uint32_t kSmSmall = kSmB + kStages * kChunkBytes;
constexpr uint32_t kSmBar = (kSmSmall + kSmallBytes + 15) & ~15u;
constexpr uint32_t kSmemBytes = kSmBar + 256;
static_assert(kSmemBytes <= 227 * 1024, "shared memory budget");
static_assert(2 * kHLo <= kABytes, "h operand fits the A region");

struct Bars {
    uint64_t setup;
    uint64_t b_full[kStages], b_empty[kStages];
    uint64_t a1_ready, acc1_full, h_ready;
    uint64_t acc_full[2], acc_empty[2];
    uint64_t g_ready, g_empty[2];
    uint64_t w_full[2], w_empty[2];
    uint64_t acch_full;
    uint64_t w1_ready, d_full;
    uint32_t tmem_base;
    uint32_t tile_max;
};
static_assert(sizeof(Bars) <= 256, "barrier block");
constexpr uint32_t kColAcc1 = 0;
constexpr uint32_t kColAcc2 = 64;                // + buf * 96
constexpr uint32_t kColAccH = 256;
constexpr uint32_t kColAccW = 320;               // + wb * 80
constexpr uint32_t kColD1 = 64, kColD2 = 128;    // tile end, over the (idle) chunk accumulators

struct Args {
    const uint8_t* packed;
    const float* x;
    const float* g_out;
    const float* g_ldj;
    float* g_x;
    float* g_pre;            // [rows, 64] (nullable when the first Linear's products run in the kernel)
    float* g_w2;             // [n_chunks * 96, 72], accumulated
    float* g_w1;             // nullable: [64 hidden, 64 conditioning slots], accumulated -> first Linear fused too
    float* g_b1;             // [64], accumulated (with g_w1)
    uint32_t cta_stride;     // deterministic mode: floats between the per-CTA copies of the three images (0: one shared copy)
    uint32_t b1_extra;       // deterministic mode: float offset (from g_b1) of the gb1 slots of sub-partitions 1..3
    float lower, upper;
    long long rows;
    int n_tiles;
};

__device__ __forceinline__ void red_add4(float* p, float a, float b, float c, float d) {
    asm volatile("red.global.add.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}
// 8 scaled gradients -> fp16 hi | lo (saturating), one 16-byte store each
__device__ __forceinline__ void put_g8(uint8_t* dst_hi, const float* v, float sigma) {
    uint4 hh, hl;
    split_f16x2_sat(v[0] * sigma, v[1] * sigma, hh.x, hl.x);
    split_f16x2_sat(v[2] * sigma, v[3] * sigma, hh.y, hl.y);
    split_f16x2_sat(v[4] * sigma, v[5] * sigma, hh.z, hl.z);
    split_f16x2_sat(v[6] * sigma, v[7] * sigma, hh.w, hl.w);
    *reinterpret_cast<uint4*>(dst_hi) = hh;
    *reinterpret_cast<uint4*>(dst_hi + kGLo) = hl;
}

template <int KIND, bool INVERSE>
__global__ void __launch_bounds__(kTThreads, 1) tc_wide_train_kernel(const Args A) {
    extern __shared__ __align__(1024) uint8_t smem[];
    float* xs = reinterpret_cast<float*>(smem + kSmXs);
    uint8_t* abuf = smem + kSmA;
    uint8_t* gbuf = smem + kSmG;
    uint8_t* bst = smem + kSmB;
    const Header* hdr = reinterpret_cast<const Header*>(smem + kSmSmall);
    const float* b1s = reinterpret_cast<const float*>(smem + kSmSmall + kOffB1);
    const float* b2s = reinterpret_cast<const float*>(smem + kSmSmall + kOffB2);
    Bars* bars = reinterpret_cast<Bars*>(smem + kSmBar);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

    if (tid == 0) {
        mbar_init(&bars->setup, 1);
        for (int i = 0; i < kStages; ++i) { mbar_init(&bars->b_full[i], 1); mbar_init(&bars->b_empty[i], 1); }
        mbar_init(&bars->a1_ready, kEpiWarps);
        mbar_init(&bars->acc1_full, 1);
        mbar_init(&bars->h_ready, kEpiWarps);
        for (int b = 0; b < 2; ++b) {
            mbar_init(&bars->acc_full[b], 1); mbar_init(&bars->acc_empty[b], 8);
            mbar_init(&bars->w_full[b], 1); mbar_init(&bars->w_empty[b], 8);
        }
        mbar_init(&bars->g_ready, 8);
        mbar_init(&bars->g_empty[0], 1);
        mbar_init(&bars->g_empty[1], 1);
        mbar_init(&bars->acch_full, 1);
        mbar_init(&bars->w1_ready, kEpiWarps);
        mbar_init(&bars->d_full, 1);
        bars->tile_max = 0;
        fence_mbar_init();
    }
    __shared__ uint32_t tmem_base_s;      // own word: the allocator writes it, keep it away from the mbarrier block
    if (warp == 1) tmem_alloc(&tmem_base_s, kTmemCols);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_base_s;

    if (tid == 0) {
        mbar_arrive_expect_tx(&bars->setup, kSmallBytes);
        bulk_g2s(smem + kSmSmall, A.packed, kSmallBytes, &bars->setup);
    }
    mbar_wait(&bars->setup, 0);

    const int d = hdr->dim, n_tr = hdr->n_tr, n_cond = hdr->n_cond, n_chunks = hdr->n_chunks;
    const int k1pad = hdr->k1pad;
    const int act = hdr->act;
    const float s2 = hdr->s2;
    const float s2l = s2 * 1.4426950408889634f;
    const int my_tiles = (A.n_tiles > (int)blockIdx.x) ? (A.n_tiles - 1 - (int)blockIdx.x) / (int)gridDim.x + 1 : 0;
    const bool full = A.g_w1 != nullptr;                  // the first Linear's gradient products run here too
    const int n_items = n_chunks + (full ? 1 : 0);        // ring items after the leading W1: chunks (+ W1 again)

    if (warp == 0) {
        // ======================= producer =========================================================
        if (lane == 0) {
            uint32_t cc = 0;
            for (int it = 0; it < my_tiles; ++it) {
                for (int c = -1; c < n_items; ++c, ++cc) {
                    const uint32_t st = cc % kStages, use = cc / kStages;
                    mbar_wait_relaxed(&bars->b_empty[st], (use & 1) ^ 1);
                    mbar_arrive_expect_tx(&bars->b_full[st], kChunkBytes);
                    const uint8_t* src = (c < 0 || c == n_chunks) ? A.packed + kOffW1 : A.packed + kOffW2 + (size_t)c * kChunkBytes;
                    bulk_g2s(bst + st * kChunkBytes, src, kChunkBytes, &bars->b_full[st]);
                }
            }
        }
    } else if (warp == 1) {
        // ======================= UMMA issuer F: the forward recompute (GEMM1, GEMM2 chunks) =======
        // Two issuer threads: with one, a wait for the epilogue's gradients (G) held back a recompute GEMM
        // whose operands were ready, and the other way round.
        if (lane == 0) {
            const uint32_t idesc1 = make_idesc(FMT_BF16, 128, kHid);
            const uint32_t idesc2 = make_idesc(FMT_F16, 128, kChunkN);
            const uint32_t a_hi = smem_u32(abuf), a_lo = a_hi + kHLo;
            uint32_t cc = 0, cb = 0;
            for (int it = 0; it < my_tiles; ++it) {
                const uint32_t tpar = it & 1;
                {
                    const uint32_t st = cc % kStages, use = cc / kStages;
                    mbar_wait_relaxed(&bars->b_full[st], use & 1);
                    mbar_wait_relaxed(&bars->a1_ready, tpar);
                    tc_fence_after();
                    const uint32_t a0 = smem_u32(abuf), b0 = smem_u32(bst + st * kChunkBytes);
                    uint32_t acc = 0;
#pragma unroll
                    for (int p = 0; p < 8; ++p) {
                        const int pa = (p == 0 || p == 3 || p == 6) ? 1 : ((p == 1 || p == 4) ? 2 : 0);
                        const int pb = (p == 0 || p == 2) ? 2 : ((p == 1 || p == 3 || p == 5) ? 1 : 0);
                        for (int ks = 0; ks < k1pad / 16; ++ks) {
                            umma_f16(tmem + kColAcc1, make_smem_desc(a0 + pa * kA1Part + ks * 256, 128, 1024),
                                     make_smem_desc(b0 + pb * kW1Part + ks * 256, 128, 1024), idesc1, acc);
                            acc = 1;
                        }
                    }
                    umma_commit(&bars->acc1_full);
                    umma_commit(&bars->b_empty[st]);
                    ++cc;
                }
                for (int c = 0; c < n_chunks; ++c) {
                    const uint32_t ci = cc + (uint32_t)c, st = ci % kStages, use = ci / kStages;
                    mbar_wait_relaxed(&bars->b_full[st], use & 1);
                    const uint32_t n = cb + (uint32_t)c, buf = n & 1, buse = n >> 1;
                    if (c == 0) mbar_wait_relaxed(&bars->h_ready, tpar);
                    mbar_wait_relaxed(&bars->acc_empty[buf], (buse & 1) ^ 1);
                    tc_fence_after();
                    const uint32_t b_hi = smem_u32(bst + st * kChunkBytes), b_lo = b_hi + 12288;
                    const uint32_t dcol = tmem + kColAcc2 + buf * kChunkN;
                    uint32_t acc = 0;
#pragma unroll
                    for (int p = 0; p < 3; ++p) {
                        const uint32_t aa = (p == 0) ? a_lo : a_hi, bb = (p == 1) ? b_lo : b_hi;
#pragma unroll
                        for (int ks = 0; ks < kHid / 16; ++ks) {
                            umma_f16(dcol, make_smem_desc(aa + ks * 256, 128, kHSbo),
                                     make_smem_desc(bb + ks * 256, 128, 1024), idesc2, acc);
                            acc = 1;
                        }
                    }
                    umma_commit(&bars->acc_full[buf]);
                }
                cc += (uint32_t)n_items;
                cb += (uint32_t)n_chunks;
            }
        }
    } else if (warp == 2) {
        // ======================= UMMA issuer G: the gradient products ==============================
        if (lane == 0) {
            const uint32_t idesc_h = make_idesc(FMT_F16, 128, kHid) | kIdescBMajorMN;
            const uint32_t idesc_w = make_idesc(FMT_F16, 128, kHPad) | kIdescAMajorMN | kIdescBMajorMN;
            const uint32_t a_hi = smem_u32(abuf), a_lo = a_hi + kHLo;
            const uint32_t g_hi = smem_u32(gbuf), g_lo = g_hi + kGLo;
            uint32_t cc = 0, cb = 0;
            for (int it = 0; it < my_tiles; ++it) {
                const uint32_t tpar = it & 1;
                const uint32_t cc0 = cc + 1;                    // ring index of chunk 0 of this tile (after the W1 item)
                for (int c = 0; c < n_chunks; ++c) {
                    const uint32_t ci = cc0 + (uint32_t)c, st = ci % kStages;
                    const uint32_t n = cb + (uint32_t)c, wb = n & 1, wuse = n >> 1;
                    mbar_wait_relaxed(&bars->g_ready, n & 1);
                    mbar_wait_relaxed(&bars->w_empty[wb], (wuse & 1) ^ 1);
                    tc_fence_after();
                    const uint32_t b_hi = smem_u32(bst + st * kChunkBytes), b_lo = b_hi + 12288;
                    // g_hidden += G . W2chunk : K = 96 parameters, B = the stage as [K = param][N = hidden]
                    // The tensor core truncates the running accumulator at every step and this sum runs over all
                    // chunks of the tile: the hi*hi products go to one accumulator, the two small correction
                    // passes to another (kColAcc1, free since the tanh pass), so the large sum takes a third of
                    // the steps and the corrections' truncation is far below its resolution.
#pragma unroll
                    for (int p = 0; p < 3; ++p) {
                        const uint32_t aa = (p == 0) ? g_lo : g_hi, bb = (p == 1) ? b_lo : b_hi;
                        const uint32_t dcol = tmem + ((p == 2) ? kColAccH : kColAcc1);
                        uint32_t acc = (c == 0 && p != 1) ? 0u : 1u;
#pragma unroll
                        for (int ks = 0; ks < kChunkN / 16; ++ks) {
                            umma_f16(dcol, make_smem_desc(aa + ks * 256, 128, kGSbo),
                                     make_smem_desc(bb + ks * 2048, 1024, 128), idesc_h, acc);
                            acc = 1;
                        }
                    }
                    // [gW2chunk | gb2] = G^T . [h | 1] : K = 128 rows, both operands MN-major views
                    uint32_t acc = 0;
#pragma unroll
                    for (int p = 0; p < 3; ++p) {
                        const uint32_t aa = (p == 0) ? g_lo : g_hi, bb = (p == 1) ? a_lo : a_hi;
#pragma unroll
                        for (int ks = 0; ks < kTileRows / 16; ++ks) {
                            umma_f16(tmem + kColAccW + wb * kHPad, make_smem_desc(aa + ks * 2 * kGSbo, kGSbo, 128),
                                     make_smem_desc(bb + ks * 2 * kHSbo, kHSbo, 128), idesc_w, acc);
                            acc = 1;
                        }
                    }
                    umma_commit(&bars->w_full[wb]);
                    umma_commit(&bars->g_empty[n & 1]);
                    umma_commit(&bars->b_empty[st]);           // the chunk's ring stage is released here
                }
                umma_commit(&bars->acch_full);
                if (full) {
                    // first Linear: g_x[cond] = g_pre . W1c and gW1c = g_pre^T . x_cond, all operands bf16x3 (exact
                    // splits, fp32 range: no scaling), the 8 leading partial products, smallest first.
                    //   D1 [128 x 64 slots] : A = g_pre K-major (G buffer), B = the W1 image read MN-major
                    //   D2 [64 hid (of 128) x 64 slots] : A = g_pre MN-major, B = the re-split x_cond MN-major
                    const uint32_t ci = cc0 + (uint32_t)n_chunks, st = ci % kStages, use = ci / kStages;
                    mbar_wait_relaxed(&bars->b_full[st], use & 1);
                    mbar_wait_relaxed(&bars->w1_ready, tpar);
                    tc_fence_after();
                    const uint32_t w1 = smem_u32(bst + st * kChunkBytes), xc = smem_u32(abuf);
                    const uint32_t idesc_d1 = make_idesc(FMT_BF16, 128, kHid) | kIdescBMajorMN;
                    const uint32_t idesc_d2 = make_idesc(FMT_BF16, 128, kK1) | kIdescAMajorMN | kIdescBMajorMN;
                    uint32_t acc1 = 0, acc2 = 0;
#pragma unroll
                    for (int p = 0; p < 8; ++p) {
                        const int pa = (p == 0 || p == 3 || p == 6) ? 1 : ((p == 1 || p == 4) ? 2 : 0);
                        const int pb = (p == 0 || p == 2) ? 2 : ((p == 1 || p == 3 || p == 5) ? 1 : 0);
#pragma unroll
                        for (int ks = 0; ks < kHid / 16; ++ks) {
                            umma_f16(tmem + kColD1, make_smem_desc(g_hi + pa * kA1Part + ks * 256, 128, 1024),
                                     make_smem_desc(w1 + pb * kW1Part + ks * 2048, 1024, 128), idesc_d1, acc1);
                            acc1 = 1;
                        }
#pragma unroll
                        for (int ks = 0; ks < kTileRows / 16; ++ks) {
                            umma_f16(tmem + kColD2, make_smem_desc(g_hi + pa * kA1Part + ks * 2048, 1024, 128),
                                     make_smem_desc(xc + pb * kA1Part + ks * 2048, 1024, 128), idesc_d2, acc2);
                            acc2 = 1;
                        }
                    }
                    umma_commit(&bars->d_full);
                    umma_commit(&bars->b_empty[st]);
                }
                cc += 1u + (uint32_t)n_items;
                cb += (uint32_t)n_chunks;
            }
        }
    } else {
        // ======================= loader + epilogue warps ==========================================
        const int q = warp & 3;
        // deterministic mode (A.cta_stride != 0): this CTA accumulates into its OWN copy of the images, every address
        // by one fixed thread, tiles in a fixed order; tcw_reduce_images_kernel then sums the copies in CTA order
        // (the three image pointers are re-derived at their rare uses: the kernel sits at its register ceiling)
#define STB_G_W2P (A.g_w2 + (size_t)blockIdx.x * A.cta_stride)
#define STB_G_W1P (A.g_w1 + (size_t)blockIdx.x * A.cta_stride)
#define STB_G_B1P (A.g_b1 + (size_t)blockIdx.x * A.cta_stride + ((A.cta_stride && q) ? A.b1_extra + (uint32_t)(q - 1) * kHid : 0u))
        const int r4 = (warp - kTEpiWarp0) >> 2;
        const int etid = tid - kTEpiWarp0 * 32;
        const int rloc = q * 32 + lane;
        const uint32_t h_row_off = (uint32_t)(rloc >> 3) * kHSbo + (uint32_t)(rloc & 7) * 16;
        const uint32_t g_row_off = (uint32_t)(rloc >> 3) * kGSbo + (uint32_t)(rloc & 7) * 16;
        const uint32_t lane_sel = (uint32_t)(q * 32) << 16;
        const float lo = A.lower, hi = A.upper;
        const float inv_span = 1.f / (hi - lo);
        uint32_t cb = 0;

        for (int it = 0; it < my_tiles; ++it) {
            const long long tile = (long long)blockIdx.x + (long long)it * gridDim.x;
            const long long row0 = tile * kTileRows;
            const int nrows = (int)min((long long)kTileRows, A.rows - row0);
            const uint32_t tpar = it & 1;
            const bool row_live = rloc < nrows;

            // ---- load the tile (as tc_wide_kernel): conditioning columns -> bf16x3 A operand, transformed
            // columns of x -> smem, pass-through columns of g_out -> g_x; the tile's gradient scale -----------
            float gmax = 0.f;
            {
                const float* xg = A.x + row0 * d;
                const float* gg = A.g_out + row0 * d;
                float* og = A.g_x + row0 * d;
                const bool copy_pass = !full && static_cast<const float*>(A.g_x) != A.g_out;   // full: written at the tile end
                const bool vec = ((d & 3) == 0) && ((reinterpret_cast<uintptr_t>(xg) & 15) == 0) &&
                                 ((reinterpret_cast<uintptr_t>(gg) & 15) == 0) && ((reinterpret_cast<uintptr_t>(og) & 15) == 0);
                if (vec) {
                    const int d4 = d >> 2, n4 = kTileRows * d4;
                    for (int i0 = etid; i0 < n4; i0 += kEpiThreads * 4) {
                      float4 vb[4], gb[4];
#pragma unroll
                      for (int u4 = 0; u4 < 4; ++u4) {
                        const int i = i0 + u4 * kEpiThreads;
                        const bool live = i < n4 && fast_div(i, hdr->m_d4) < nrows;
                        vb[u4] = live ? __ldg(reinterpret_cast<const float4*>(xg) + i) : make_float4(0.f, 0.f, 0.f, 0.f);
                        gb[u4] = live ? __ldg(reinterpret_cast<const float4*>(gg) + i) : make_float4(0.f, 0.f, 0.f, 0.f);
                      }
#pragma unroll
                      for (int u4 = 0; u4 < 4; ++u4) {
                        const int i = i0 + u4 * kEpiThreads;
                        if (i >= n4) break;
                        const int r = fast_div(i, hdr->m_d4), c = (i - r * d4) << 2;
                        const bool live = r < nrows;
                        const float4 v = vb[u4], gv = gb[u4];
                        gmax = fmaxf(gmax, fmaxf(fmaxf(fabsf(gv.x), fabsf(gv.y)), fmaxf(fabsf(gv.z), fabsf(gv.w))));
                        const int m0 = hdr->colmap[c], m1 = hdr->colmap[c + 1], m2 = hdr->colmap[c + 2], m3 = hdr->colmap[c + 3];
                        if (m0 >= 0 && (m0 & 3) == 0 && m1 == m0 + 1 && m2 == m0 + 2 && m3 == m0 + 3) {
                            a1_put4(abuf, r, m0, v);
                            if (copy_pass && live) reinterpret_cast<float4*>(og)[i] = gv;
                        } else {
                            const float vv[4] = {v.x, v.y, v.z, v.w};
                            const float gvv[4] = {gv.x, gv.y, gv.z, gv.w};
                            const int mm[4] = {m0, m1, m2, m3};
#pragma unroll
                            for (int u = 0; u < 4; ++u) {
                                if (mm[u] >= 0) {
                                    a1_put(abuf, r, mm[u], vv[u]);
                                    if (copy_pass && live) og[(size_t)r * d + c + u] = gvv[u];
                                } else {
                                    xs[r * kTrStride - mm[u] - 1] = vv[u];
                                }
                            }
                        }
                      }
                    }
                } else {
                    const int n = kTileRows * d;
                    for (int i = etid; i < n; i += kEpiThreads) {
                        const int r = fast_div(i, hdr->m_d), c = i - r * d;
                        const bool live = r < nrows;
                        const float v = live ? __ldg(xg + i) : 0.f;
                        const float gv = live ? __ldg(gg + i) : 0.f;
                        gmax = fmaxf(gmax, fabsf(gv));
                        const int m = hdr->colmap[c];
                        if (m >= 0) {
                            a1_put(abuf, r, m, v);
                            if (copy_pass && live) og[i] = gv;
                        } else {
                            xs[r * kTrStride - m - 1] = v;
                        }
                    }
                }
                const int npad = k1pad - n_cond;
                const uint32_t m_npad = hdr->m_npad;
                for (int i = etid; i < kTileRows * npad; i += kEpiThreads) {
                    const int r = fast_div(i, m_npad), m = n_cond + (i - r * npad);
                    a1_zero(abuf, r, m);
                }
            }
            float g_ld = 0.f;
            if (A.g_ldj != nullptr && row_live) g_ld = __ldg(A.g_ldj + row0 + rloc);
            gmax = fmaxf(gmax, fabsf(g_ld));
#pragma unroll
            for (int o = 16; o; o >>= 1) gmax = fmaxf(gmax, __shfl_xor_sync(0xffffffffu, gmax, o));
            if (lane == 0) atomicMax(&bars->tile_max, __float_as_uint(gmax));
            fence_proxy_async_smem();
            named_bar_sync(1, kEpiThreads);
            if (lane == 0) mbar_arrive(&bars->a1_ready);
            // per-tile scale: the largest incoming gradient maps to [2^-6, 2^-5) (fp16 head-room for the
            // spline's amplification, 2^-24 absolute resolution of the hi | lo pair below it)
            float sigma = 1.f, inv_sigma = 1.f;
            {
                const uint32_t e = (bars->tile_max >> 23) & 0xffu;
                if (e >= 8u && e <= 240u) {
                    sigma = __uint_as_float((248u - e) << 23);          // 2^(-6 - (e - 127))
                    inv_sigma = __uint_as_float((e + 6u) << 23);
                }
            }

            // ---- hidden layer: h = act(acc1 + b1) -> fp16 hi | lo, 80-column operand [h | 1 | 0] -------------
            mbar_wait_sleep(&bars->acc1_full, tpar, 64);
            tc_fence_after();
#pragma unroll 1
            for (int kc = r4; kc < kHid / 8; kc += 4) {
                const int c0 = kc * 8;
                float v[8];
                tmem_ld8(tmem + lane_sel + kColAcc1 + c0, v);
                tmem_ld_wait();
                __align__(16) __half hh[8], hl[8];
                if (act == STB_ACT_TANH) {
#pragma unroll
                    for (int i = 0; i < 8; ++i) v[i] = tanh_fast(v[i] + b1s[c0 + i]);
                } else {
#pragma unroll
                    for (int i = 0; i < 8; ++i) v[i] = sigmoid_act(v[i] + b1s[c0 + i]);          // STB_ACT_SIGMOID
                }
#pragma unroll
                for (int i = 0; i < 8; ++i) split_f16(v[i], hh[i], hl[i]);
                *reinterpret_cast<uint4*>(abuf + h_row_off + kc * 128) = *reinterpret_cast<const uint4*>(hh);
                *reinterpret_cast<uint4*>(abuf + kHLo + h_row_off + kc * 128) = *reinterpret_cast<const uint4*>(hl);
            }
            if (r4 < 2) {                                       // columns 64..79: 1, 0, ... (hi), 0 (lo)
                const uint32_t one = row_live ? 0x3c00u : 0u;   // rows beyond the batch contribute nothing to gb2
                *reinterpret_cast<uint4*>(abuf + h_row_off + (8 + r4) * 128) = make_uint4(r4 == 0 ? one : 0u, 0u, 0u, 0u);
                *reinterpret_cast<uint4*>(abuf + kHLo + h_row_off + (8 + r4) * 128) = make_uint4(0u, 0u, 0u, 0u);
            }
            tc_fence_before();
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) mbar_arrive(&bars->h_ready);

            // ---- chunks: parameters out of TMEM, element gradient in registers, G into shared memory ---------
            float* xrow = xs + rloc * kTrStride;
            auto flush_w = [&](int c) {
                // this group's gW2 partial of chunk c: TMEM lane = packed parameter column, 65 columns
                const uint32_t n = cb + (uint32_t)c, wb = n & 1, wuse = n >> 1;
                mbar_wait_sleep(&bars->w_full[wb], wuse & 1, 64);
                tc_fence_after();
                const int g = r4 & 1;
                if (q < 3) {
                    float* dst = STB_G_W2P + ((size_t)c * kChunkN + rloc) * kWStride + g * 32;
                    const uint32_t col = tmem + lane_sel + kColAccW + wb * kHPad + (uint32_t)g * 32;
                    float v[16];
#pragma unroll
                    for (int hh2 = 0; hh2 < 2; ++hh2) {
                        tmem_ld16(col + hh2 * 16, v);
                        tmem_ld_wait();
#pragma unroll
                        for (int i = 0; i < 16; i += 4) {
                            red_add4(dst + hh2 * 16 + i, v[i] * inv_sigma, v[i + 1] * inv_sigma, v[i + 2] * inv_sigma, v[i + 3] * inv_sigma);
                        }
                    }
                    if (g == 1) {
                        float w8[8];
                        tmem_ld8(tmem + lane_sel + kColAccW + wb * kHPad + kHid, w8);
                        tmem_ld_wait();
                        atomicAdd(STB_G_W2P + ((size_t)c * kChunkN + rloc) * kWStride + kHid, w8[0] * inv_sigma);
                    }
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&bars->w_empty[wb]);
            };
            int prev = -1;
#pragma unroll 1
            for (int ji = r4; ji < kG * n_chunks; ji += 4) {
                const int c = ji >> 1;
                const uint32_t n = cb + (uint32_t)c;
                const uint32_t buf = n & 1, buse = n >> 1;
                const int g = ji & 1;
                const bool live_dim = ji < n_tr;
                const float xv = live_dim ? xrow[ji] : 0.f;
                const bool inside = live_dim && row_live && (xv >= lo) && (xv <= hi);
                const float go = (live_dim && row_live) ? __ldg(A.g_out + (size_t)(row0 + rloc) * d + hdr->tr_idx[ji]) : 0.f;
                const float* bb = b2s + ji * kPPad;
                const float2* bb2 = reinterpret_cast<const float2*>(bb);
                mbar_wait_sleep(&bars->acc_full[buf], buse & 1, 32);
                tc_fence_after();
                const uint32_t col0 = tmem + lane_sel + kColAcc2 + buf * kChunkN + (uint32_t)g * kPPad;
                const bool shift = !((hdr->noshift_mask[ji >> 5] >> (ji & 31)) & 1u);
                float2 t[kBins];
                tmem_ld16(col0, reinterpret_cast<float*>(t));
                tmem_ld16(col0 + 16, reinterpret_cast<float*>(t) + 16);
                tmem_ld_wait();
#pragma unroll
                for (int i = 0; i < kBins; ++i) t[i] = __ffma2_rn(t[i], f2(s2l), bb2[i]);
                softmax16_num2(t, shift);
                float2 ee, eo;
                float gx = go, gu0 = 0.f, gu1 = 0.f;
                int kk;
                if (KIND == STB_RQS) {
                    const BinSearch16 bs = bin_search16<INVERSE>(t, STB_RQS_MIN, (xv - lo) * inv_span, ee, eo);
                    float dd[16];
                    tmem_ld16(col0 + 2 * kBins, dd);
                    tmem_ld_wait();
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&bars->acc_empty[buf]);
                    float r0, r1;
                    pick_pair16(dd, bs.k, r0, r1);
                    kk = bs.k;
                    const float u0 = (kk == 0) ? STB_RQS_EDGE_CONST : fmaf(r0, s2, bb[2 * kBins + (kk > 0 ? kk - 1 : 0)]);
                    const float u1 = (kk == kBins - 1) ? STB_RQS_EDGE_CONST : fmaf(r1, s2, bb[2 * kBins + (kk < kBins - 1 ? kk : 0)]);
                    if (inside) {
                        rqs16_backward<INVERSE>(t, bs, ee, eo, u0, u1, lo, hi, xv, go, g_ld, gx, gu0, gu1);
                    } else {
#pragma unroll
                        for (int i = 0; i < kBins; ++i) t[i] = f2(0.f);
                    }
                } else {
                    const float u = (xv - lo) / (hi - lo);
                    const BinSearch16 bs = bin_search16<INVERSE>(t, STB_CUB_MIN, u, ee, eo);
                    float dd[8];
                    tmem_ld8(col0 + 2 * kBins, dd);
                    tmem_ld_wait();
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&bars->acc_empty[buf]);
                    kk = bs.k;
                    const float ul = fmaf(dd[0], s2, bb[2 * kBins]), ur = fmaf(dd[1], s2, bb[2 * kBins + 1]);
                    if (inside) {
                        cubic16_backward<INVERSE>(t, bs, ee, eo, ul, ur, lo, hi, u, go, g_ld, gx, gu0, gu1);
                    } else {
#pragma unroll
                        for (int i = 0; i < kBins; ++i) t[i] = f2(0.f);
                    }
                }
                if (live_dim) xrow[ji] = gx;                       // x of this element is dead: reuse for g_x
                if (prev >= 0) flush_w(prev);
                // G is one buffer: chunk n may be written once the products of chunk n - 1 have retired.  Two
                // barriers alternate so that a warp (which handles every second chunk) waits on consecutive
                // phases of ONE barrier: with a single barrier the phase it skips makes parity ambiguous.
                if (n >= 1) mbar_wait_sleep(&bars->g_empty[(n - 1) & 1], ((n - 1) >> 1) & 1, 64);
                {
                    uint8_t* gdst = gbuf + g_row_off + (uint32_t)(g * (kPPad / 8)) * 128;
                    float w[8];
#pragma unroll
                    for (int b8 = 0; b8 < 4; ++b8) {               // packed column order: (w_i, h_i) interleaved
#pragma unroll
                        for (int i = 0; i < 4; ++i) { w[2 * i] = t[b8 * 4 + i].x; w[2 * i + 1] = t[b8 * 4 + i].y; }
                        put_g8(gdst + b8 * 128, w, sigma);
                    }
                    // derivative columns 32..47: zero except at the two knots of bin k
                    const uint4 z4 = make_uint4(0u, 0u, 0u, 0u);
                    *reinterpret_cast<uint4*>(gdst + 4 * 128) = z4;
                    *reinterpret_cast<uint4*>(gdst + 5 * 128) = z4;
                    *reinterpret_cast<uint4*>(gdst + kGLo + 4 * 128) = z4;
                    *reinterpret_cast<uint4*>(gdst + kGLo + 5 * 128) = z4;
                    uint32_t dh, dl;
                    split_f16x2_sat(gu0 * sigma, gu1 * sigma, dh, dl);
                    if (KIND == STB_RQS) {
                        if (kk > 0) {                               // derivative kk - 1 (knot kk)
                            uint8_t* pd = gdst + (4 + ((kk - 1) >> 3)) * 128 + ((kk - 1) & 7) * 2;
                            *reinterpret_cast<uint16_t*>(pd) = (uint16_t)(dh & 0xffffu);
                            *reinterpret_cast<uint16_t*>(pd + kGLo) = (uint16_t)(dl & 0xffffu);
                        }
                        if (kk < kBins - 1) {                       // derivative kk (knot kk + 1)
                            uint8_t* pd = gdst + (4 + (kk >> 3)) * 128 + (kk & 7) * 2;
                            *reinterpret_cast<uint16_t*>(pd) = (uint16_t)(dh >> 16);
                            *reinterpret_cast<uint16_t*>(pd + kGLo) = (uint16_t)(dl >> 16);
                        }
                    } else {                                        // cubic: columns 32, 33 = the end derivatives
                        *reinterpret_cast<uint32_t*>(gdst + 4 * 128) = dh;
                        *reinterpret_cast<uint32_t*>(gdst + kGLo + 4 * 128) = dl;
                    }
                }
                fence_proxy_async_smem();
                __syncwarp();
                if (lane == 0) mbar_arrive(&bars->g_ready);
                prev = c;
            }
            if (prev >= 0) flush_w(prev);
            cb += (uint32_t)n_chunks;

            // ---- g_pre = g_hidden * act'(h) ----------------------------------------------------------------------
            mbar_wait_sleep(&bars->acch_full, tpar, 64);
            tc_fence_after();
            {
                const float unscale = s2 * inv_sigma;
#pragma unroll 1
                for (int kc = r4; kc < kHid / 8; kc += 4) {
                    float v[8], vc[8];
                    tmem_ld8(tmem + lane_sel + kColAccH + kc * 8, v);
                    tmem_ld8(tmem + lane_sel + kColAcc1 + kc * 8, vc);
                    tmem_ld_wait();
#pragma unroll
                    for (int i = 0; i < 8; ++i) v[i] += vc[i];
                    const uint4 hh = *reinterpret_cast<const uint4*>(abuf + h_row_off + kc * 128);
                    const uint4 hl = *reinterpret_cast<const uint4*>(abuf + kHLo + h_row_off + kc * 128);
                    const __half* ph = reinterpret_cast<const __half*>(&hh);
                    const __half* pl = reinterpret_cast<const __half*>(&hl);
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        const float h = __half2float(ph[i]) + __half2float(pl[i]);
                        const float da = (act == STB_ACT_TANH) ? (1.f - h * h)
                                       : ((act == STB_ACT_SIGMOID) ? h * (1.f - h) : ((h > 0.f) ? 1.f : 0.f));
                        v[i] = v[i] * unscale * da;
                    }
                    if (row_live && A.g_pre != nullptr) stg256(A.g_pre + (size_t)(row0 + rloc) * kHid + kc * 8, v);
                    if (full) {
                        // bf16x3 parts of g_pre, K-major [128 x 64] in the (now idle) G buffer
                        __align__(16) __nv_bfloat16 q0[8], q1[8], q2[8];
#pragma unroll
                        for (int i = 0; i < 8; ++i) split_bf16x3(v[i], q0[i], q1[i], q2[i]);
                        uint8_t* dst = gbuf + (uint32_t)(rloc >> 3) * 1024 + (uint32_t)(rloc & 7) * 16 + kc * 128;
                        *reinterpret_cast<uint4*>(dst) = *reinterpret_cast<const uint4*>(q0);
                        *reinterpret_cast<uint4*>(dst + kA1Part) = *reinterpret_cast<const uint4*>(q1);
                        *reinterpret_cast<uint4*>(dst + 2 * kA1Part) = *reinterpret_cast<const uint4*>(q2);
                        // gb1 += column sums over the warp's 32 rows
#pragma unroll
                        for (int i = 0; i < 8; ++i) {
                            float sum = v[i];
#pragma unroll
                            for (int o = 16; o; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
                            if (lane == i) atomicAdd(STB_G_B1P + kc * 8 + i, sum);
                        }
                    }
                }
            }
            tc_fence_before();
            named_bar_sync(1, kEpiThreads);
            if (full) {
                // ---- conditioning columns again: x_cond as bf16x3 (its buffer held h meanwhile) --------------------
                {
                    const float* xg = A.x + row0 * d;
                    const int n = kTileRows * d;
                    for (int i = etid; i < n; i += kEpiThreads) {
                        const int r = fast_div(i, hdr->m_d), c = i - r * d;
                        const int m = hdr->colmap[c];
                        if (m >= 0) {
                            const float v = (r < nrows) ? __ldg(xg + i) : 0.f;
                            a1_put(abuf, r, m, v);
                        }
                    }
                    const int npad = kK1 - n_cond;               // all 64 slots are read as N
                    const uint32_t m_npad = hdr->m_npad64;
                    for (int i = etid; i < kTileRows * npad; i += kEpiThreads) {
                        const int r = fast_div(i, m_npad), m = n_cond + (i - r * npad);
                        a1_zero(abuf, r, m);
                    }
                }
                fence_proxy_async_smem();
                __syncwarp();
                if (lane == 0) mbar_arrive(&bars->w1_ready);
                mbar_wait_sleep(&bars->d_full, tpar, 64);
                tc_fence_after();
                {
                    float v[16];
                    // g_x[cond] = g_out[cond] + g_pre . W1c : thread = row, 16 conditioning slots per warp
                    tmem_ld16(tmem + lane_sel + kColD1 + r4 * 16, v);
                    tmem_ld_wait();
                    if (row_live) {
                        const float* gr = A.g_out + (size_t)(row0 + rloc) * d;
                        float* xr = A.g_x + (size_t)(row0 + rloc) * d;
                        // all 16 loads first: load-then-store per element is a chain of exposed round trips (g_x may
                        // alias g_out, so the compiler keeps the order)
                        float go16[16];
#pragma unroll
                        for (int i = 0; i < 16; ++i) {
                            const int m = r4 * 16 + i;
                            go16[i] = (m < n_cond) ? __ldg(gr + hdr->cond_idx[m]) : 0.f;
                        }
#pragma unroll
                        for (int i = 0; i < 16; ++i) {
                            const int m = r4 * 16 + i;
                            if (m < n_cond) xr[hdr->cond_idx[m]] = go16[i] + v[i];
                        }
                    }
                    // gW1c[hid][slot] += D2 : TMEM lane = hidden unit (64 valid), 16 slots per warp
                    tmem_ld16(tmem + lane_sel + kColD2 + r4 * 16, v);
                    tmem_ld_wait();
                    if (q < 2) {
                        float* dst = STB_G_W1P + (size_t)rloc * kK1 + r4 * 16;
#pragma unroll
                        for (int i = 0; i < 16; i += 4) red_add4(dst + i, v[i], v[i + 1], v[i + 2], v[i + 3]);
                    }
                }
                tc_fence_before();
            }
            // ---- transformed columns of g_x out ----------------------------------------------------------------
            {
                float* og = A.g_x + row0 * d;
                for (int i = etid; i < nrows * n_tr; i += kEpiThreads) {
                    const int r = fast_div(i, hdr->m_ntr), sl = i - r * n_tr;
                    og[(size_t)r * d + hdr->tr_idx[sl]] = xs[r * kTrStride + sl];
                }
                if (etid == 0) bars->tile_max = 0;
            }
            named_bar_sync(1, kEpiThreads);
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem, kTmemCols);
}
}  // namespace train

// -----------------------------------------------------------------------------------------------
// packing
// -----------------------------------------------------------------------------------------------
// the image's layout for spline64_pack_kernel (tc_pack.cuh), plus this file's header fields: the division magics and
// the column -> slot map
struct PackLayout {
    using Hdr = Header;
    static constexpr uint32_t kMagic = tcw::kMagic, kOffB1 = tcw::kOffB1, kOffW1 = tcw::kOffW1;
    static constexpr int kK1 = tcw::kK1, kMaxTr = tcw::kMaxTr;
    static __device__ void header_extra(Header* hdr, const SplinePackArgs& a) {
        const int n_cond = a.m.n_cond;
        hdr->k1pad = (n_cond + a.n_lat + 15) & ~15;
        if (hdr->k1pad == 0) hdr->k1pad = 16;
        hdr->m_d = div_magic(a.dim); hdr->m_d4 = div_magic(max(a.dim >> 2, 1)); hdr->m_ntr = div_magic(a.m.n_tr);
        hdr->m_npad = div_magic(max(hdr->k1pad - n_cond - a.n_lat, 1));
        hdr->m_npad64 = div_magic(max(kK1 - n_cond, 1));
        for (int j = 0; j < kMaxDim; ++j) hdr->colmap[j] = 0;
        for (int i = 0; i < n_cond; ++i) hdr->colmap[a.m.cond_idx[i]] = (int16_t)i;
        for (int i = 0; i < a.m.n_tr; ++i) hdr->colmap[a.m.tr_idx[i]] = (int16_t)(-i - 1);
    }
};

// the shared spline gate, then this file's conditioner: MLP[64]
static_assert(kMaxTr == kK1, "spline_gate bounds the transformed dims by GEMM1's K");
static bool admit(const stb_layer* L, MaskSplit& m) {
    return spline_gate(L, kMaxDim, kK1, m) && L->net.n_linear == 2 && L->net.dims[1] == kHid;
}

}  // namespace tcw

bool tcw_layer_supported(const stb_layer* L) {
    tcw::MaskSplit m;
    return tcw::admit(L, m);
}

uint64_t tcw_packed_bytes(const stb_layer*) { return tcw::kPackedBytes; }

int tcw_pack_layer(const stb_layer* L, void* out, cudaStream_t stream) {
    using namespace tcw;
    SplinePackArgs a;
    if (!admit(L, a.m)) return set_error(STB_ENOTSUP, "layer has no wide tensor-core path");
    a.out = static_cast<uint8_t*>(out);
    a.n_chunks = (a.m.n_tr + kG - 1) / kG;
    a.n_lat = L->latent_dim; a.n_bins = L->n_bins;
    a.kind = L->kind; a.dim = L->dim; a.P = spline_params_per_dim(L->kind, L->n_bins);
    a.act = L->net.activation;
    a.W1 = L->net.W[0]; a.b1 = L->net.b[0]; a.W2 = L->net.W[1]; a.b2 = L->net.b[1];
    const BoundArgs b = spline_bound_args(a.m, a.W2, a.b2, kHid, a.P, a.n_bins, a.act,
                                          a.out + offsetof(Header, noshift_mask));
    return pack_image(out, sizeof(Header), stream, "tcw_pack", [&] {
        pack_pass(spline64_maxabs_kernel<PackLayout>, 64, 256, stream, a);
        pack_pass(spline64_pack_kernel<PackLayout>, 296, 256, stream, a);
        pack_pass(tc_bound_kernel, (kMaxTr + 7) / 8, 256, stream, b);
    });
}

int tcw_layer_apply(const stb_layer* L, const void* image, int direction, const float* x, const float* latent, float* y,
                    float* ldj, int ldj_mode, int base_log_prob, int64_t rows, cudaStream_t stream, int32_t* bins) {
    using namespace tcw;
    Args A = {};
    A.bins = bins;
    A.latent = L->latent_dim > 0 ? latent : nullptr;
    A.packed = static_cast<const uint8_t*>(image);
    A.x = x; A.y = y; A.ldj = ldj;
    A.ldj_mode = ldj ? ldj_mode : STB_LDJ_NONE;
    A.base_log_prob = base_log_prob;
    A.lower = L->lower; A.upper = L->upper;
    A.rows = rows;
    const long long tiles = (rows + kTileRows - 1) / kTileRows;
    if (tiles > 0x7fffffffLL) return set_error(STB_EINVAL, "too many rows");
    A.n_tiles = (int)tiles;
    void (*kern)(Args) = pick_variant(L->kind, direction == STB_INVERSE, L->n_bins == kBins,
                                      [](auto K, auto I, auto F) { return tc_wide_kernel<K, I, false, F>; });
    return launch_persistent(kern, A, tiles, 1, kThreads, kSmemBytes, stream, "tc_wide_kernel");
}

// quadratic and cubic (fused variant); `latent=` layers train through the element-wise kernels + autograd
bool tcw_backward_supported(const stb_layer* L) { return tcw_layer_supported(L) && L->latent_dim == 0 && L->n_bins == tcw::kBins; }

int tcw_layer_backward(const stb_layer* L, const void* image, int direction, const float* x, const float* g_out,
                       const float* g_ldj, float* g_x, float* g_net, float* hidden, int64_t rows,
                       cudaStream_t stream) {
    using namespace tcw;
    if (L->kind != STB_RQS) return set_error(STB_ENOTSUP, "tensor-core backward is built for the quadratic spline");
    Args A = {};
    A.packed = static_cast<const uint8_t*>(image);
    A.x = x; A.y = g_x; A.ldj = nullptr;
    A.ldj_mode = STB_LDJ_NONE;
    A.lower = L->lower; A.upper = L->upper;
    A.rows = rows;
    A.g_out = g_out; A.g_ldj = g_ldj; A.g_net = g_net; A.hidden = hidden;
    const long long tiles = (rows + kTileRows - 1) / kTileRows;
    if (tiles > 0x7fffffffLL) return set_error(STB_EINVAL, "too many rows");
    A.n_tiles = (int)tiles;
    void (*kern)(Args) = (direction == STB_INVERSE) ? tc_wide_kernel<STB_RQS, true, true> : tc_wide_kernel<STB_RQS, false, true>;
    return launch_persistent(kern, A, tiles, 1, kThreads, kSmemBytes, stream, "tc_wide_kernel (backward)");
}


// STRIBOR_B200_DETERMINISTIC=1: bit-reproducible parameter gradients.  The default adds every tile's partial
// products to ONE L2-resident image with red.global.add (summation order over tiles varies run to run); in this mode
// each CTA owns a copy of the images (single writer per address, tiles in a fixed order) and a second kernel adds
// the copies in CTA order.
static bool train_deterministic() {
    static const bool on = [] { const char* e = getenv("STRIBOR_B200_DETERMINISTIC"); return e && e[0] == '1'; }();
    return on;
}
namespace tcw { namespace train {
constexpr uint32_t kImgFloats = (uint32_t)kMaxChunks * kChunkN * kWStride + kHid * kK1 + kHid;      // gW2 | gW1 | gb1
constexpr uint32_t kCtaStride = kImgFloats + 3 * kHid;                                               // + gb1 slots of q = 1..3
constexpr int kDetMaxCtas = 160;

// image 0 (+)= images 1 .. n_cta-1, then the four gb1 slots collapse into the first: fixed order, one thread per element
__global__ void tcw_reduce_images_kernel(float* base, int n_cta) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= kCtaStride) return;
    float acc = base[i];
    for (int c = 1; c < n_cta; ++c) acc += base[(size_t)c * kCtaStride + i];
    base[i] = acc;
}
// gb1 [64] sits at the end of the image, the slots of sub-partitions 1..3 right behind it
__global__ void tcw_collapse_gb1_kernel(float* base) {
    const uint32_t i = threadIdx.x;
    if (i >= kHid) return;
    float* b1 = base + kImgFloats - kHid;
    b1[i] = ((b1[i] + base[kImgFloats + i]) + base[kImgFloats + kHid + i]) + base[kImgFloats + 2 * kHid + i];
}
}}

uint64_t tcw_train_workspace_floats(const stb_layer* L, int64_t rows) {
    (void)L;
    const uint64_t img = train_deterministic() ? (uint64_t)tcw::train::kDetMaxCtas * tcw::train::kCtaStride
                                               : (uint64_t)tcw::train::kImgFloats;
    return (uint64_t)rows * tcw::kHAug + img;
}

// Fused: g_x; gW2 image = workspace[rows * 72 : +3072 * 72] (accumulated).  first_linear != 0: the first Linear's
// products run in the kernel too -- g_x is complete, gW1c [64 x 64 slots] and gb1 [64] follow the image
// (accumulated); else g_pre = workspace[0 : rows * 64] is written and those products are left to the caller.
int tcw_layer_backward_fused(const stb_layer* L, const void* image, int direction, const float* x, const float* g_out,
                             const float* g_ldj, float* g_x, float* workspace, int first_linear, int64_t rows,
                             cudaStream_t stream) {
    using namespace tcw;
    const int act = L->net.activation;
    if (act != STB_ACT_TANH && act != STB_ACT_SIGMOID && act != STB_ACT_RELU)
        return set_error(STB_ENOTSUP, "fused conditioner backward: Tanh / Sigmoid / ReLU hidden activation only");
    train::Args A = {};
    A.packed = static_cast<const uint8_t*>(image);
    A.x = x; A.g_out = g_out; A.g_ldj = g_ldj; A.g_x = g_x;
    A.g_w2 = workspace + (size_t)rows * kHAug;
    if (first_linear) {
        A.g_pre = nullptr;
        A.g_w1 = A.g_w2 + (size_t)kMaxChunks * kChunkN * train::kWStride;
        A.g_b1 = A.g_w1 + kHid * kK1;
    } else {
        A.g_pre = workspace;
    }
    A.lower = L->lower; A.upper = L->upper;
    A.rows = rows;
    const long long tiles = (rows + kTileRows - 1) / kTileRows;
    if (tiles > 0x7fffffffLL) return set_error(STB_EINVAL, "too many rows");
    A.n_tiles = (int)tiles;
    void (*kern)(train::Args) = pick_variant(L->kind, direction == STB_INVERSE,
                                             [](auto K, auto I) { return train::tc_wide_train_kernel<K, I>; });
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)train::kSmemBytes);
    if (e != cudaSuccess) return set_error(STB_ECUDA, "cudaFuncSetAttribute: %s", cudaGetErrorString(e));
    int grid = (int)min((long long)sm_count(), tiles);
    const bool det = train_deterministic();
    if (det) {
        grid = min(grid, train::kDetMaxCtas);
        A.cta_stride = train::kCtaStride;
        A.b1_extra = kHid;                       // from g_b1 (the last 64 floats of an image) to the slots behind it
    }
    kern<<<grid, train::kTThreads, train::kSmemBytes, stream>>>(A);
    count_launch();
    if (det) {
        train::tcw_reduce_images_kernel<<<(train::kCtaStride + 255) / 256, 256, 0, stream>>>(A.g_w2, grid);
        count_launch();
        if (first_linear) {
            train::tcw_collapse_gb1_kernel<<<1, 64, 0, stream>>>(A.g_w2);
            count_launch();
        }
    }
    e = cudaGetLastError();
    if (e != cudaSuccess) return set_error(STB_ECUDA, "tc_wide_train_kernel launch: %s", cudaGetErrorString(e));
    return STB_OK;
}

}  // namespace stb
