// Tensor-core spline coupling with a WIDE conditioner (tcgen05 + TMEM-resident activations).
//
// Scope: st.Coupling(st.Spline(dim <= 64, 2 <= n_bins <= 16, 'quadratic' | 'cubic', latent_net = MLP(dim (+ latent), [H] or
// [H, H], dim * P)), mask) with H in {64 (two hidden layers only), 128, 192, 256}, Tanh / Sigmoid, conditioning + latent
// columns <= 32 -- the secondary shape of BASELINE.json configs[2] (SURVEY.md 8d: MLP[256,256], 7.34 MFLOP per sample),
// which round 1 left on the CUDA-core kernel.  MLP[64] stays on tc_layer.cu / tc_wide.cu.
//
// With K = H the last Linear no longer fits the layout of tc_layer.cu (a 256-wide fp16 hi|lo A operand is 128 KB of
// shared memory per 128 rows).  Here the hidden activations never leave the tensor-core side:
//   GEMM1  [128 x 32] x [32 x H]    A = gathered conditioning columns, three bf16 parts in shared memory, 8 partial
//                                   products into ONE accumulator, smallest first -> TMEM columns [0, H)
//   act    16 epilogue warps (TMEM sub-partition q x column group g): tcgen05.ld 16 columns, activation + fp16 hi|lo
//          split on packed pairs, tcgen05.st of the 8 + 8 packed columns back INTO the columns just consumed
//   GEMM2' [128 x H] x [H x H]      (two hidden layers) A = h1 from TMEM, weights streamed in 16-wide K blocks ->
//                                   TMEM [256, 256 + H); second activation in place again
//   chunks TWO transformed dims at a time: [128 x H] x [H x 96], A = the last hidden layer from TMEM, the chunk's
//          packed last-Linear rows as a lo item and a hi item (one ring stage each), passes hi*lo, lo*hi, hi*hi -> one of
//          two 96-column accumulator buffers (buffer b <-> issuer b); epilogue group g (4 warps = the tile's 128 rows)
//          takes dims g, g + 4, ...: thread = row pulls its 48 parameters and evaluates the spline in registers
//          (tc_spline16.cuh, the same code as the MLP[64] kernels)
// One persistent CTA per SM, 19 warps (producer, two issuers, 16 epilogue), tile = 128 rows, 3-stage cp.async.bulk ring.
//
// Reference semantics restated here: flows/coupling.py:53-95, flows/spline.py:76-105, net/mlp.py:46-58,
// util/rational_quadratic_spline.py, util/cubic_spline.py, flow.py:42-47.
#include "common.cuh"
#include "stb_math.cuh"
#include "tc_common.cuh"
#include "tc_pack.cuh"
#include "tc_spline16.cuh"

namespace stb {
using namespace tc;

namespace tch {
using namespace sp16;

constexpr int kRows = 128;
constexpr int kK1 = 32;
constexpr int kPPad = 48;
constexpr int kMaxDim = 64;
constexpr int kMaxTr = 32;
constexpr int kMaxH = 256;
constexpr int kXsStride = kMaxDim + 1;
constexpr int kStages = 3;
constexpr int kNBuf = 2;                 // 96-column chunk accumulators (two transformed dims): buffer b belongs to issuer b and to epilogue groups 2b, 2b + 1
constexpr int kChunkN = 2 * kPPad;
constexpr int kEpiWarp0 = 2;
constexpr int kEpiWarps = 16;
constexpr int kIssuers = 2;                              // UMMA issuer threads of the chunk phase (dims ji % 2)
constexpr int kIssuerB = kEpiWarp0 + kEpiWarps;          // issuer 1: warp 18 (issuer 0 = warp 1)
constexpr int kThreads = (kEpiWarp0 + kEpiWarps + kIssuers - 1) * 32;
constexpr int kEpiThreads = kEpiWarps * 32;
constexpr uint32_t kMagic = 0x53544834u;

struct Header {                          // 1024 bytes
    uint32_t magic;
    int32_t kind, dim, n_cond, n_tr, H, n_hidden, P, act;
    float s_mid, s_out;                  // power-of-two scales of the packed second-hidden / last Linear
    uint32_t max_mid, max_out;           // scratch (max |W| bits)
    uint32_t noshift_mask;
    int32_t cond_idx[kK1];
    int32_t tr_idx[kMaxTr];
    int32_t n_lat;                       // `latent=` columns (coupling.py:64-65): GEMM1 columns n_cond .. n_cond + n_lat - 1
    int32_t n_bins;                      // 2 .. 16 real bins in the 16-bin packed layout (padded bins: weight 0, bias -inf)
    int32_t pad[256 - 16 - kK1 - kMaxTr];
};
static_assert(sizeof(Header) == 1024, "header layout");
constexpr uint32_t kOffB1 = 1024, kOffB2 = kOffB1 + kMaxH * 4, kOffB3 = kOffB2 + kMaxH * 4;     // b3: float [32][48]
constexpr uint32_t kSmallBytes = kOffB3 + kMaxTr * kPPad * 4;                                    // 9216
constexpr uint32_t kOffW = kSmallBytes;

__host__ __device__ inline uint32_t w1_block(int H) { return (uint32_t)H * 32; }      // [H x 16] bf16
__host__ __device__ inline uint32_t w2_block(int H) { return (uint32_t)H * 64; }      // [H x 16] fp16 hi | lo
__host__ __device__ inline uint32_t w3_block() { return kPPad * 64; }                 // [48 x 16] fp16 hi | lo = 3072
__host__ __device__ inline uint32_t stage_bytes(int H) { return (uint32_t)H * 192; }  // = 6 W1 blocks = 3 W2 blocks = one dim of W3
__host__ __device__ inline uint32_t off_w2(int H) { return kOffW + 6 * w1_block(H); }
__host__ __device__ inline uint32_t off_w3(int H, int n_hidden) {
    return off_w2(H) + (n_hidden == 2 ? (uint32_t)(H / 16) * w2_block(H) : 0u);
}
__host__ __device__ inline uint32_t packed_bytes(int H, int n_hidden) {
    return off_w3(H, n_hidden) + (uint32_t)kMaxTr * stage_bytes(H);
}

// shared memory map
constexpr uint32_t kSmXs = 0;                                       // float [128][65]
constexpr uint32_t kSmA1 = (kRows * kXsStride * 4 + 127) & ~127u;   // 3 x 8 KB
constexpr uint32_t kA1Part = kRows * kK1 * 2;
constexpr uint32_t kSmSmall = kSmA1 + 3 * kA1Part;
constexpr uint32_t kSmLd = kSmSmall + kSmallBytes;                  // float [4][128]
constexpr uint32_t kSmBar = kSmLd + 4 * kRows * 4;
constexpr uint32_t kSmRing = (kSmBar + 256 + 127) & ~127u;
__host__ __device__ inline uint32_t smem_bytes(int H) { return kSmRing + kStages * stage_bytes(H); }

struct Bars {
    uint64_t setup;
    uint64_t b_full[kStages], b_empty[kStages];
    uint64_t a1_ready, acc1_full, h1_ready, acc2_full, h2_ready;
    uint64_t acc_full[kNBuf], acc_empty[kNBuf];
};
static_assert(sizeof(Bars) <= 256, "barrier block");

struct Args {
    const uint8_t* packed;
    const float* x;
    const float* latent;     // [rows, lat_stride] or NULL
    int lat_stride;
    float* y;
    float* ldj;
    int32_t* bins;
    int ldj_mode, base_log_prob;
    float lower, upper;
    long long rows;
    int n_tiles;
};

// two hidden units: activation of (acc * sc + bias), fp16 hi | lo parts packed for the TMEM A operand
template <bool TANH>
__device__ __forceinline__ void act_split2(float2 v, float2 sc, float2 bias, uint32_t& hi, uint32_t& lo) {
    const float2 pre = __ffma2_rn(v, sc, bias);
    float2 h;
    if (TANH) { h.x = tanh_fast(pre.x); h.y = tanh_fast(pre.y); }
    else { h.x = sigmoid_act(pre.x); h.y = sigmoid_act(pre.y); }
    asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(hi) : "f"(h.y), "f"(h.x));
    const float2 hf = __half22float2(*reinterpret_cast<const __half2*>(&hi));
    const float2 res = __ffma2_rn(hf, make_float2(-1.f, -1.f), h);
    asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(lo) : "f"(res.y), "f"(res.x));
}

// hidden layer in place: this warp's columns [c_begin, c_end) of the accumulator at `acc` become h (hi at +0, lo at +8
// of every 16-column block)
__device__ __forceinline__ void activate_in_place(uint32_t acc, int c_begin, int c_end, float sc, const float* bias, int act) {
    for (int c0 = c_begin; c0 < c_end; c0 += 16) {
        float v[16];
        tmem_ld16(acc + c0, v);
        tmem_ld_wait();
        uint32_t hh[8], hl[8];
        const float2* b2p = reinterpret_cast<const float2*>(bias + c0);
        if (act == STB_ACT_TANH) {
#pragma unroll
            for (int i = 0; i < 8; ++i) act_split2<true>(make_float2(v[2 * i], v[2 * i + 1]), make_float2(sc, sc), b2p[i], hh[i], hl[i]);
        } else {
#pragma unroll
            for (int i = 0; i < 8; ++i) act_split2<false>(make_float2(v[2 * i], v[2 * i + 1]), make_float2(sc, sc), b2p[i], hh[i], hl[i]);
        }
        tmem_st8(acc + c0, hh);
        tmem_st8(acc + c0 + 8, hl);
    }
    tmem_st_wait();
}

// FULL = false: 2 .. 15 real bins in the padded 16-bin layout (tc_spline16.cuh)
template <int KIND, bool INVERSE, bool FULL = true>
__global__ void __launch_bounds__(kThreads, 1) tc_hw_spline_kernel(const Args A) {
    extern __shared__ __align__(1024) uint8_t smem[];
    __shared__ uint32_t tmem_base_s;
    float* xs = reinterpret_cast<float*>(smem + kSmXs);
    uint8_t* a1buf = smem + kSmA1;
    const Header* hdr = reinterpret_cast<const Header*>(smem + kSmSmall);
    const float* b1s = reinterpret_cast<const float*>(smem + kSmSmall + kOffB1);
    const float* b2h = reinterpret_cast<const float*>(smem + kSmSmall + kOffB2);
    const float* b3s = reinterpret_cast<const float*>(smem + kSmSmall + kOffB3);
    float* ld_s = reinterpret_cast<float*>(smem + kSmLd);
    Bars* bars = reinterpret_cast<Bars*>(smem + kSmBar);
    uint8_t* ring = smem + kSmRing;

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

    if (tid == 0) {
        mbar_init(&bars->setup, 1);
        for (int i = 0; i < kStages; ++i) { mbar_init(&bars->b_full[i], 1); mbar_init(&bars->b_empty[i], 1); }
        mbar_init(&bars->a1_ready, kEpiWarps);
        mbar_init(&bars->acc1_full, 1);
        mbar_init(&bars->h1_ready, kEpiWarps);
        mbar_init(&bars->acc2_full, 1);
        mbar_init(&bars->h2_ready, kEpiWarps);
        for (int b = 0; b < kNBuf; ++b) { mbar_init(&bars->acc_full[b], 1); mbar_init(&bars->acc_empty[b], 8); }
        fence_mbar_init();
    }
    if (warp == 1) tmem_alloc(&tmem_base_s, 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_base_s;
    if (tid == 0) {
        mbar_arrive_expect_tx(&bars->setup, kSmallBytes);
        bulk_g2s(smem + kSmSmall, A.packed, kSmallBytes, &bars->setup);
    }
    mbar_wait(&bars->setup, 0);

    const int d = hdr->dim, n_tr = hdr->n_tr, n_cond = hdr->n_cond, H = hdr->H, n_hidden = hdr->n_hidden, act = hdr->act;
    const int kb_h = H / 16;
    const uint32_t stage = stage_bytes(H);
    const uint32_t w1b = w1_block(H), w2b = w2_block(H);
    const int n_items2 = (n_hidden == 2) ? (kb_h + 2) / 3 : 0;              // W2' items of up to 3 K blocks
    const uint32_t col_h_last = (n_hidden == 2) ? 256u : 0u;                // A operand of the chunk GEMMs
    const uint32_t col_chunk = (n_hidden == 2) ? 0u : (uint32_t)H;          // two 96-column accumulators
    const int n_chunks = (n_tr + 1) / 2;
    const int my_tiles = (A.n_tiles > (int)blockIdx.x) ? (A.n_tiles - 1 - (int)blockIdx.x) / (int)gridDim.x + 1 : 0;

    // ---- one chunk = TWO transformed dims: [128 x H] x [H x 96] into accumulator buffer `buf`, A = the last hidden layer
    // in TMEM.  The chunk UMMAs cost a fixed ~38 clocks each whatever N (measured: N = 16 and N = 48 take the same
    // time), so two dims per UMMA halve the chunk phase's tensor time.  A chunk's weights travel as two ring
    // items -- the fp16 lo parts, then the hi parts, each [96 x H] K-major in K blocks of 16 -- and the three passes
    // go hi*lo (item 0, released), then lo*hi and hi*hi (item 1): corrections first, the accumulator truncates.
    // Every mbarrier of the chunk phase is a PRIVATE channel, so that a waiter's successive waits are successive phases
    // whatever the relative speed of the agents (a parity wait cannot tell "two phases behind" from "done"): accumulator
    // buffer b is written by issuer b only and read by epilogue groups 2b, 2b + 1 only; a ring stage is refilled only
    // after the issuer that consumed its previous item has released it.
    auto issue_chunk = [&](uint32_t rc, uint32_t buf, uint32_t buse) {
        const uint32_t idesc3 = make_idesc(FMT_F16, 128, kChunkN);
        const uint32_t dcol = tmem + col_chunk + buf * kChunkN;
        const uint32_t ad0 = tmem + col_h_last;
        uint32_t acc = 0;
#pragma unroll 1
        for (int item = 0; item < 2; ++item, ++rc) {
            const uint32_t st = rc % kStages, use = rc / kStages;
            mbar_wait_relaxed(&bars->b_full[st], use & 1);
            if (item == 0) mbar_wait_relaxed(&bars->acc_empty[buf], (buse & 1) ^ 1);
            tc_fence_after();
            const uint64_t bd0 = make_smem_desc(smem_u32(ring + st * stage), 128, 256);
#pragma unroll 1
            for (int p = (item == 0 ? 0 : 1); p < (item == 0 ? 1 : 3); ++p) {       // p: 0 hi*lo, 1 lo*hi, 2 hi*hi
                // descriptors advance by constants: 3072 B (>> 4 in the descriptor's address field) and 16 TMEM columns
                uint64_t bd = bd0;
                uint32_t ad = ad0 + ((p == 1) ? 8u : 0u);
#pragma unroll 4
                for (int kb = 0; kb < kb_h; ++kb) {
                    umma_f16_ts(dcol, ad, bd, idesc3, acc);
                    acc = 1;
                    bd += (uint64_t)(w3_block() >> 4);
                    ad += 16u;
                }
            }
            if (item == 1) umma_commit(&bars->acc_full[buf]);
            umma_commit(&bars->b_empty[st]);
        }
    };

    if (warp == 0) {
        // ======================= producer: one ring item = W1 | 3 K blocks of W2' | one dim of W3 ===================
        if (lane == 0) {
            uint32_t rc = 0;
            auto put = [&](const uint8_t* src, uint32_t bytes) {
                const uint32_t st = rc % kStages, use = rc / kStages;
                mbar_wait_relaxed(&bars->b_empty[st], (use & 1) ^ 1);
                mbar_arrive_expect_tx(&bars->b_full[st], bytes);
                bulk_g2s(ring + st * stage, src, bytes, &bars->b_full[st]);
                ++rc;
            };
            for (int it = 0; it < my_tiles; ++it) {
                if (it + 1 < my_tiles) {
                    const long long nrow0 = ((long long)blockIdx.x + (long long)(it + 1) * gridDim.x) * kRows;
                    const long long nb = min((long long)kRows, A.rows - nrow0) * d * 4;
                    const char* src = reinterpret_cast<const char*>(A.x + nrow0 * d);
                    if (nb >= 16 && ((reinterpret_cast<uintptr_t>(src) & 15) == 0))
                        asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(src), "r"((uint32_t)(nb & ~15LL)) : "memory");
                }
                put(A.packed + kOffW, 6 * w1b);
                for (int i2 = 0; i2 < n_items2; ++i2) {
                    const int nb = min(3, kb_h - 3 * i2);
                    put(A.packed + off_w2(H) + (uint32_t)(3 * i2) * w2b, (uint32_t)nb * w2b);
                }
                for (int i3 = 0; i3 < 2 * n_chunks; ++i3) put(A.packed + off_w3(H, n_hidden) + (uint32_t)i3 * stage, stage);
            }
        }
    } else if (warp == 1) {
        // ======================= UMMA issuer ==========================================================================
        if (lane == 0) {
            const uint32_t idesc1 = make_idesc(FMT_BF16, 128, H);
            const uint32_t idesc2 = make_idesc(FMT_F16, 128, H);
            const uint32_t a0 = smem_u32(a1buf);
            uint32_t rc = 0, tp = 0;
            uint32_t nuse[2] = {0, 0};             // uses so far of this issuer's buffers 0 and 2
            for (int it = 0; it < my_tiles; ++it, tp ^= 1) {
                {   // ---- GEMM1: 8 bf16 partial products, smallest first, one accumulator -----------------------------
                    const uint32_t st = rc % kStages, use = rc / kStages;
                    mbar_wait_relaxed(&bars->b_full[st], use & 1);
                    mbar_wait_relaxed(&bars->a1_ready, tp);
                    tc_fence_after();
                    const uint32_t b0 = smem_u32(ring + st * stage);
                    uint32_t acc = 0;
#pragma unroll
                    for (int p = 0; p < 8; ++p) {
                        // (pa,pb): (1,2) (2,1) (0,2) (1,1) (2,0) (0,1) (1,0) (0,0)
                        const int pa = (p == 0 || p == 3 || p == 6) ? 1 : ((p == 1 || p == 4) ? 2 : 0);
                        const int pb = (p == 0 || p == 2) ? 2 : ((p == 1 || p == 3 || p == 5) ? 1 : 0);
#pragma unroll
                        for (int ks = 0; ks < 2; ++ks) {
                            // packed W1 blocks are ordered (pb = 2, 1, 0) x (kb = 0, 1)
                            umma_f16(tmem, make_smem_desc(a0 + pa * kA1Part + ks * 256, 128, 512),
                                     make_smem_desc(b0 + (uint32_t)((2 - pb) * 2 + ks) * w1b, 128, 256), idesc1, acc);
                            acc = 1;
                        }
                    }
                    umma_commit(&bars->acc1_full);
                    umma_commit(&bars->b_empty[st]);
                    ++rc;
                }
                if (n_hidden == 2) {   // ---- GEMM2': A = h1 from TMEM, per K block lo*hi, hi*lo, hi*hi ---------------------
                    mbar_wait_relaxed(&bars->h1_ready, tp);
                    uint32_t acc = 0;
                    for (int i2 = 0; i2 < n_items2; ++i2, ++rc) {
                        const uint32_t st = rc % kStages, use = rc / kStages;
                        mbar_wait_relaxed(&bars->b_full[st], use & 1);
                        tc_fence_after();
                        const int nb = min(3, kb_h - 3 * i2);
                        for (int j = 0; j < nb; ++j) {
                            const int kb = 3 * i2 + j;
                            const uint32_t bb = smem_u32(ring + st * stage) + (uint32_t)j * w2b;
                            const uint64_t b_hi = make_smem_desc(bb, 128, 256), b_lo = make_smem_desc(bb + (uint32_t)H * 32, 128, 256);
                            const uint32_t a_hi = tmem + (uint32_t)kb * 16, a_lo = a_hi + 8;
                            umma_f16_ts(tmem + 256, a_lo, b_hi, idesc2, acc); acc = 1;
                            umma_f16_ts(tmem + 256, a_hi, b_lo, idesc2, 1);
                            umma_f16_ts(tmem + 256, a_hi, b_hi, idesc2, 1);
                        }
                        umma_commit(&bars->b_empty[st]);
                    }
                    umma_commit(&bars->acc2_full);
                }
                mbar_wait_relaxed(n_hidden == 2 ? &bars->h2_ready : &bars->h1_ready, tp);
                for (int c = 0; c < n_chunks; ++c, rc += 2)
                    if (!(c & 1)) { issue_chunk(rc, 0u, nuse[0]); ++nuse[0]; }
            }
        }
    } else if (warp >= kIssuerB) {
        // ======================= second UMMA issuer: the odd chunks (buffer 1) ==========================================
        // One thread spends ~8 issue slots (elect loop + descriptor arithmetic on the uniform datapath) per UMMA and a dim
        // is 3 H / 16 of them (48 at H = 256): with one issuer that thread, not the tensor pipe, paced the chunk phase
        // (2.8e7 samples/s with one issuer, 4.7e7 with two at MLP[256,256]; a third changes nothing).
        if (lane == 0) {
            uint32_t rc = 0, tp = 0;
            uint32_t nuse[2] = {0, 0};
            for (int it = 0; it < my_tiles; ++it, tp ^= 1) {
                rc += 1u + (uint32_t)n_items2;
                mbar_wait_relaxed(n_hidden == 2 ? &bars->h2_ready : &bars->h1_ready, tp);
                for (int c = 0; c < n_chunks; ++c, rc += 2)
                    if (c & 1) { issue_chunk(rc, 1u, nuse[0]); ++nuse[0]; }
            }
        }
    } else {
        // ======================= epilogue warps ========================================================================
        const int q = warp & 3;
        const int g = (warp - kEpiWarp0) >> 2;                  // epilogue group 0..3 (one warp per TMEM sub-partition each)
        const int etid = tid - kEpiWarp0 * 32;
        const int row = q * 32 + lane;
        float* xrow = xs + row * kXsStride;
        const uint32_t lane_sel = (uint32_t)(q * 32) << 16;
        const bool want_ld = A.ldj_mode != STB_LDJ_NONE;
        const float lo = A.lower, hi = A.upper;
        const float inv_span = 1.f / (hi - lo);
        const float s2 = hdr->s_out, s2l = s2 * 1.4426950408889634f;
        const float s_mid = hdr->s_mid;
        const int K = FULL ? kBins : hdr->n_bins;
        const uint32_t noshift_mask = hdr->noshift_mask;
        const int dshift = ((d & (d - 1)) == 0) ? (31 - __clz(d)) : -1;
        uint32_t buse = 0, tp = 0;                  // uses so far of this group's accumulator buffer (buffer g)

        for (int it = 0; it < my_tiles; ++it, tp ^= 1) {
            const long long row0 = ((long long)blockIdx.x + (long long)it * gridDim.x) * kRows;
            const int nrows = (int)min((long long)kRows, A.rows - row0);
            {   // ---- stage the x tile ------------------------------------------------------------------------------------
                const float* xg = A.x + row0 * d;
                const int n = nrows * d;
                if ((d & 3) == 0 && ((reinterpret_cast<uintptr_t>(xg) & 15) == 0)) {
                    const int n4 = (kRows * d) >> 2;
                    for (int i = etid; i < n4; i += kEpiThreads) {
                        const float4 v = (i * 4 < n) ? __ldg(reinterpret_cast<const float4*>(xg) + i) : make_float4(0.f, 0.f, 0.f, 0.f);
                        const int r = (dshift >= 0) ? ((i * 4) >> dshift) : (i * 4) / d, c = (i * 4) - r * d;
                        float* dst = xs + r * kXsStride + c;
                        dst[0] = v.x; dst[1] = v.y; dst[2] = v.z; dst[3] = v.w;
                    }
                } else {
                    for (int i = etid; i < kRows * d; i += kEpiThreads) {
                        const int r = i / d, c = i - r * d;
                        xs[r * kXsStride + c] = (i < n) ? __ldg(xg + i) : 0.f;
                    }
                }
            }
            named_bar_sync(1, kEpiThreads);
            // ---- A1: 8 of the 32 conditioning columns of this row (column group g), three bf16 parts ---------------------
            {
                const uint32_t off = (uint32_t)(row >> 3) * 512 + (uint32_t)(row & 7) * 16 + (uint32_t)g * 128;
                __align__(16) __nv_bfloat16 q0[8], q1[8], q2[8];
#pragma unroll
                for (int u = 0; u < 8; ++u) {
                    const int k = g * 8 + u;
                    float v = 0.f;
                    if (k < n_cond) v = xrow[hdr->cond_idx[k]];
                    else if (k < n_cond + hdr->n_lat && row < nrows) v = __ldg(A.latent + (row0 + row) * A.lat_stride + (k - n_cond));
                    split_bf16x3(v, q0[u], q1[u], q2[u]);
                }
                *reinterpret_cast<uint4*>(a1buf + off) = *reinterpret_cast<const uint4*>(q0);
                *reinterpret_cast<uint4*>(a1buf + kA1Part + off) = *reinterpret_cast<const uint4*>(q1);
                *reinterpret_cast<uint4*>(a1buf + 2 * kA1Part + off) = *reinterpret_cast<const uint4*>(q2);
                tc_fence_before();
                fence_proxy_async_smem();
                __syncwarp();
                if (lane == 0) mbar_arrive(&bars->a1_ready);
            }
            // ---- hidden layers in place: this warp's quarter of the columns ------------------------------------------------
            const int cq = H / 4;
            mbar_wait_sleep(&bars->acc1_full, tp, 64);
            tc_fence_after();
            activate_in_place(tmem + lane_sel, g * cq, (g + 1) * cq, 1.f, b1s, act);
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&bars->h1_ready);
            if (n_hidden == 2) {
                mbar_wait_sleep(&bars->acc2_full, tp, 64);
                tc_fence_after();
                activate_in_place(tmem + lane_sel + 256, g * cq, (g + 1) * cq, s_mid, b2h, act);
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&bars->h2_ready);
            }
            // ---- chunks: dims g, g + 4, ... of this group's 128 rows -----------------------------------------------------------
            float ld_acc = 0.f;
#pragma unroll 1
            for (int ji = g; ji < 2 * n_chunks; ji += 4, ++buse) {
                const uint32_t buf = (uint32_t)(g >> 1);              // chunk ji >> 1 alternates between the two buffers
                if (ji >= n_tr) {                                     // odd number of dims: the last chunk's padding half
                    mbar_wait_sleep(&bars->acc_full[buf], buse & 1, 32);
                    tc_fence_after();
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&bars->acc_empty[buf]);
                    continue;
                }
                const int j = hdr->tr_idx[ji];
                const float xv = xrow[j];
                const bool inside = (xv >= lo) && (xv <= hi);
                const float* bb = b3s + ji * kPPad;
                const float2* bb2 = reinterpret_cast<const float2*>(bb);
                mbar_wait_sleep(&bars->acc_full[buf], buse & 1, 32);
                tc_fence_after();
                const uint32_t col0 = tmem + lane_sel + col_chunk + buf * kChunkN + (uint32_t)(g & 1) * kPPad;
                const bool shift = !((noshift_mask >> (ji & 31)) & 1u);
                float out = xv, ld = 0.f;
                int kbin = -1;
                if (KIND == STB_RQS) {
                    RqsLoc loc;
                    {
                        float2 t[kBins];
                        tmem_ld16(col0, reinterpret_cast<float*>(t));
                        tmem_ld16(col0 + 16, reinterpret_cast<float*>(t) + 16);
                        tmem_ld_wait();
#pragma unroll
                        for (int i = 0; i < kBins; ++i) t[i] = __ffma2_rn(t[i], f2(s2l), bb2[i]);
                        loc = rqs16_locate<INVERSE, FULL>(t, shift, lo, inv_span, xv, K);
                    }
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
                        kbin = loc.k;
                    }
                } else {
                    const float span = hi - lo;
                    const float u = (xv - lo) / span;
                    CubSel sel;
                    {
                        float2 t[kBins];
                        tmem_ld16(col0, reinterpret_cast<float*>(t));
                        tmem_ld16(col0 + 16, reinterpret_cast<float*>(t) + 16);
                        tmem_ld_wait();
#pragma unroll
                        for (int i = 0; i < kBins; ++i) t[i] = __ffma2_rn(t[i], f2(s2l), bb2[i]);
                        sel = cubic16_locate<INVERSE, FULL>(t, shift, u, K);
                    }
                    float dd[8];
                    tmem_ld8(col0 + 2 * kBins, dd);
                    tmem_ld_wait();
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&bars->acc_empty[buf]);
                    if (inside) {
                        const float ul = fmaf(dd[0], s2, bb[2 * kBins]), ur = fmaf(dd[1], s2, bb[2 * kBins + 1]);
                        cubic16_finish<INVERSE>(sel, ul, ur, lo, hi, want_ld, u, out, ld, K);
                        kbin = sel.k;
                    }
                }
                xrow[j] = out;
                if (A.bins != nullptr && row < nrows) A.bins[(row0 + row) * d + j] = kbin;
                ld_acc += ld;
            }
            // ---- per-row log|det J| over the four groups (+ UnitNormal log-density of the output row) -------------------------
            ld_s[g * kRows + row] = ld_acc;
            named_bar_sync(1, kEpiThreads);
            if (g == 0 && want_ld && row < nrows) {
                float tot = (ld_s[row] + ld_s[kRows + row]) + (ld_s[2 * kRows + row] + ld_s[3 * kRows + row]);
                if (A.base_log_prob) {
                    float b = 0.f;
                    for (int c = 0; c < d; ++c) { const float v = xrow[c]; b += -0.5f * v * v - 0.91893853320467274178f; }
                    tot += b;
                }
                float* dst = A.ldj + row0 + row;
                *dst = (A.ldj_mode == STB_LDJ_ADD) ? (*dst + tot) : tot;
            }
            if (A.y != nullptr) {
                float* yg = A.y + row0 * d;
                const int n = nrows * d;
                if ((d & 3) == 0 && ((reinterpret_cast<uintptr_t>(yg) & 15) == 0)) {
                    const int n4 = n >> 2;
                    for (int i = etid; i < n4; i += kEpiThreads) {
                        const int r = (dshift >= 0) ? ((i * 4) >> dshift) : (i * 4) / d, c = (i * 4) - r * d;
                        const float* src = xs + r * kXsStride + c;
                        reinterpret_cast<float4*>(yg)[i] = make_float4(src[0], src[1], src[2], src[3]);
                    }
                } else {
                    for (int i = etid; i < n; i += kEpiThreads) {
                        const int r = i / d, c = i - r * d;
                        yg[i] = xs[r * kXsStride + c];
                    }
                }
            }
            named_bar_sync(1, kEpiThreads);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem, 512);
}

// -----------------------------------------------------------------------------------------------
// packing
// -----------------------------------------------------------------------------------------------
struct PackArgs {
    const float *W1, *b1, *W2, *b2, *W3, *b3;
    uint8_t* out;
    int kind, dim, H, n_hidden, P, act, n_lat, n_bins;
    MaskSplit m;
};

__global__ void tch_maxabs_kernel(const PackArgs a) {
    Header* hdr = reinterpret_cast<Header*>(a.out);
    float m2 = 0.f, m3 = 0.f;
    const int gtid = blockIdx.x * blockDim.x + threadIdx.x, gsz = gridDim.x * blockDim.x;
    if (a.n_hidden == 2)
        for (int i = gtid; i < a.H * a.H; i += gsz) m2 = fmaxf(m2, fabsf(a.W2[i]));
    const int total = a.m.n_tr * a.P * a.H;
    for (int i = gtid; i < total; i += gsz) {
        const int k = i % a.H, rp = i / a.H, p = rp % a.P, ji = rp / a.P;
        m3 = fmaxf(m3, fabsf(a.W3[((size_t)a.m.tr_idx[ji] * a.P + p) * a.H + k]));
    }
    warp_max_to(&hdr->max_mid, m2);
    warp_max_to(&hdr->max_out, m3);
}

__global__ void tch_pack_kernel(const PackArgs a) {
    Header* hdr = reinterpret_cast<Header*>(a.out);
    const float s_mid = pow2_scale(__uint_as_float(hdr->max_mid)), s_out = pow2_scale(__uint_as_float(hdr->max_out));
    const int gtid = blockIdx.x * blockDim.x + threadIdx.x, gsz = gridDim.x * blockDim.x;
    const int H = a.H;
    if (gtid == 0) {
        hdr->magic = kMagic; hdr->kind = a.kind; hdr->dim = a.dim; hdr->n_cond = a.m.n_cond; hdr->n_tr = a.m.n_tr; hdr->H = H;
        hdr->n_hidden = a.n_hidden; hdr->P = a.P; hdr->act = a.act; hdr->s_mid = s_mid; hdr->s_out = s_out; hdr->n_lat = a.n_lat; hdr->n_bins = a.n_bins;
        for (int i = 0; i < kK1; ++i) hdr->cond_idx[i] = a.m.cond_idx[i];
        for (int i = 0; i < kMaxTr; ++i) hdr->tr_idx[i] = a.m.tr_idx[i];
    }
    float* b1 = reinterpret_cast<float*>(a.out + kOffB1);
    float* b2 = reinterpret_cast<float*>(a.out + kOffB2);
    for (int i = gtid; i < kMaxH; i += gsz) {
        b1[i] = (i < H) ? a.b1[i] : 0.f;
        b2[i] = (i < H && a.n_hidden == 2) ? a.b2[i] : 0.f;
    }
    fill_spline_bias(reinterpret_cast<float*>(a.out + kOffB3), kMaxTr, a.b3, a.m, a.P, a.n_bins, gtid, gsz);
    for (int i = gtid; i < H * kK1; i += gsz) {
        const int n = i / kK1, k = i % kK1;
        store_w1_blocks(a.out + kOffW, H, n, k, first_linear_w(a.W1, n, k, a.dim + a.n_lat, a.dim, a.m, -1, a.m.n_cond, a.n_lat));
    }
    if (a.n_hidden == 2) {
        const float inv = 1.f / s_mid;
        for (int i = gtid; i < H * H; i += gsz) store_hilo_blocks(a.out + off_w2(H), H, i / H, i % H, a.W2[i] * inv);
    }
    {   // last Linear: per chunk of two transformed dims a lo item and a hi item
        uint8_t* w3 = a.out + off_w3(H, a.n_hidden);
        const float inv = 1.f / s_out;
        const int per_dim = kPPad * H;
        for (int i = gtid; i < kMaxTr * per_dim; i += gsz) {
            const int ji = i / per_dim, rem = i % per_dim, n = rem / H, k = rem % H;
            const int p = param_of_col(n, a.n_bins, a.P);
            float v = 0.f;
            if (ji < a.m.n_tr && p >= 0) v = a.W3[((size_t)a.m.tr_idx[ji] * a.P + p) * H + k] * inv;
            __half hi, lo;
            split_f16(v, hi, lo);
            // chunk c = ji / 2 (two dims, 96 rows): item 2c holds the lo parts, item 2c + 1 the hi parts, each as H / 16
            // blocks [96 x 16] (3072 B)
            const int n2 = (ji & 1) * kPPad + n;
            uint8_t* blk = w3 + (size_t)(ji & ~1) * stage_bytes(H) + (size_t)(k >> 4) * w3_block();
            *reinterpret_cast<__half*>(blk + blk_off(n2, k & 15)) = lo;
            *reinterpret_cast<__half*>(blk + stage_bytes(H) + blk_off(n2, k & 15)) = hi;
        }
    }
}

// the shared spline gate, then this file's conditioner: MLP[H] or MLP[H, H], H a multiple of 64 up to 256, not MLP[64]
// (tc_layer.cu / tc_wide.cu)
static_assert(kMaxTr == kK1, "spline_gate bounds the transformed dims by GEMM1's K");
static bool admit(const stb_layer* L, MaskSplit& m) {
    if (!spline_gate(L, kMaxDim, kK1, m)) return false;
    const stb_mlp& N = L->net;
    const int H = N.dims[1];
    if (H < 64 || H > kMaxH || (H % 64) != 0) return false;
    if (N.n_linear == 2 && H == 64) return false;
    return N.n_linear == 2 || N.dims[2] == H;
}

}  // namespace tch

bool tch_layer_supported(const stb_layer* L) {
    tch::MaskSplit m;
    return tch::admit(L, m);
}

uint64_t tch_packed_bytes(const stb_layer* L) { return tch::packed_bytes(L->net.dims[1], L->net.n_linear - 1); }

int tch_pack_layer(const stb_layer* L, void* out, cudaStream_t stream) {
    using namespace tch;
    PackArgs a;
    if (!admit(L, a.m)) return set_error(STB_ENOTSUP, "layer has no wide-conditioner tensor-core path");
    const stb_mlp& N = L->net;
    a.out = static_cast<uint8_t*>(out);
    a.kind = L->kind; a.dim = L->dim; a.H = N.dims[1]; a.n_hidden = N.n_linear - 1; a.act = N.activation;
    a.n_lat = L->latent_dim; a.n_bins = L->n_bins; a.P = spline_params_per_dim(L->kind, L->n_bins);
    a.W1 = N.W[0]; a.b1 = N.b[0];
    a.W2 = a.n_hidden == 2 ? N.W[1] : nullptr; a.b2 = a.n_hidden == 2 ? N.b[1] : nullptr;
    a.W3 = N.W[N.n_linear - 1]; a.b3 = N.b[N.n_linear - 1];
    const BoundArgs b = spline_bound_args(a.m, a.W3, a.b3, a.H, a.P, a.n_bins, a.act,
                                          a.out + offsetof(Header, noshift_mask));
    return pack_image(out, sizeof(Header), stream, "tch_pack", [&] {
        pack_pass(tch_maxabs_kernel, 128, 256, stream, a);
        pack_pass(tch_pack_kernel, 592, 256, stream, a);
        pack_pass(tc_bound_kernel, 1, kMaxTr * 32, stream, b);
    });
}

int tch_layer_apply(const stb_layer* L, int direction, const float* x, const float* latent, float* y, float* ldj,
                    int ldj_mode, int base_log_prob, int64_t rows, cudaStream_t stream, int32_t* bins) {
    using namespace tch;
    const int H = L->net.dims[1];
    if (L->packed_bytes < packed_bytes(H, L->net.n_linear - 1)) return set_error(STB_EINVAL, "packed image too small");
    Args A = {};
    A.latent = L->latent_dim > 0 ? latent : nullptr;
    A.lat_stride = L->latent_dim;
    A.packed = static_cast<const uint8_t*>(L->packed);
    A.x = x; A.y = y; A.ldj = ldj; A.bins = bins;
    A.ldj_mode = ldj ? ldj_mode : STB_LDJ_NONE;
    A.base_log_prob = base_log_prob;
    A.lower = L->lower; A.upper = L->upper;
    A.rows = rows;
    const long long tiles = (rows + kRows - 1) / kRows;
    if (tiles > 0x7fffffffLL) return set_error(STB_EINVAL, "too many rows");
    A.n_tiles = (int)tiles;
    void (*kern)(Args) = pick_variant(L->kind, direction == STB_INVERSE, L->n_bins == kBins,
                                      [](auto K, auto I, auto F) { return tc_hw_spline_kernel<K, I, F>; });
    // one CTA per SM, each streaming its own weights: clusters of CTAs sharing one weight stream measured slower
    // (DESIGN.md 4.1f)
    return launch_persistent(kern, A, tiles, 1, kThreads, smem_bytes(H), stream, "tc_hw_spline_kernel");
}

}  // namespace stb
