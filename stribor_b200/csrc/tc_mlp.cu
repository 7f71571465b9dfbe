// Tensor-core fused AFFINE coupling layer with a wide conditioner (tcgen05 + TMEM + bulk copies).
//
// Scope: st.Coupling(st.Affine(dim <= 64, latent_net = MLP(dim (+ latent), [H] or [H, H], 2 dim)), mask),
// H in {64, 128, 192, 256}, conditioning + latent (+ t) columns <= 32 -- BASELINE.json configs[1] (MLP[256,256]) -- and
// st.ContinuousAffineCoupling(MLP(dim (+1), [H] or [H, H], 2 dim), TimeLinear(2 dim), mask)
// (configs[3], flows/coupling.py:188-213: the time column joins the conditioning columns, the
// affine parameters are multiplied by scale * t in the epilogue).  Here the
// conditioner IS the work (2 * (32 H + H^2 + 64 H) flop per row-layer against 520 B), so the layout
// is a plain chain of GEMMs with the activations kept on chip:
//
//   tile = 128 rows, persistent CTA per SM, 18 warps
//   warp 0       producer: streams the packed weights in 16-wide K blocks ([N x 16] K-major,
//                <= 16 KB) L2 -> smem through a 3-stage cp.async.bulk / mbarrier ring
//   warp 1       UMMA issuer.  Every GEMM accumulates into TWO TMEM accumulators: the full-magnitude
//                hi*hi products go to `main`, all correction products (lo*hi, hi*lo; for the bf16x3
//                first layer everything but x0*W0) to `corr`, because the tensor core truncates
//                the running accumulator at every step (profiles/r01_tc_accuracy.txt); the epilogue
//                adds the two in fp32.
//   warps 2-17   four per TMEM sub-partition q, each owning a quarter of the columns: stage x,
//                mask gather + exact bf16x3 split (A operand of layer 1), tanh + fp16 hi|lo split of
//                each hidden layer's accumulator back into the A operand of the next GEMM, and the
//                affine transform + log|det J| from the last accumulator.
//
// Kernels in this file: tc_mlp_affine_kernel<NCG> (the layout above; NCG = 2: small conditioners, two CTAs per SM),
// tc_mlp_pipe_kernel (H >= 128: single accumulators, activations resident in TMEM, the next GEMM issued wave by wave
// behind the activation pass, the next tile prepared inside the current one's GEMM drains), tc_mlp_chain_kernel<V> and
// tc_mlp_chain4_kernel (a whole affine / continuous-affine flow in one launch, weights resident in shared memory).
//
// Reference semantics: flows/coupling.py:53-95, flows/affine.py:59-109, net/mlp.py:46-58.
#include "common.cuh"
#include "stb_math.cuh"
#include "tc_common.cuh"
#include "tc_pack.cuh"

namespace stb {
using namespace tc;

namespace tcm {

constexpr int kRows = 128;
constexpr int kK1 = 32;
constexpr int kMaxTr = 32;
constexpr int kNOut = 64;                  // [log_scale(32) | shift(32)] of the transformed dims
constexpr int kMaxDim = 64;
constexpr int kMaxH = 256;
constexpr int kStages = 3;
constexpr int kEpiWarp0 = 2;
constexpr uint32_t kSlotBytes = 16384;     // one K block: [<=256 x 16] fp16 hi | lo
constexpr uint32_t kMagic = 0x53544d31u;

struct Header {                            // 1024 bytes
    uint32_t magic;
    int32_t dim, n_cond, n_tr, H, n_hidden, act;
    float s_mid, s_out;                    // power-of-two scales of the packed 2nd / last Linear
    uint32_t max_mid, max_out;             // scratch (max |W| bits)
    int32_t cond_idx[kK1];
    int32_t tr_idx[kMaxTr];
    int32_t cont, time_col;                // continuous-affine: scale by the time embedding; A1 column holding t (-1: none)
    float ts_ls[kMaxTr], ts_sh[kMaxTr];    // TimeLinear.scale of the transformed dims (log-scale half | shift half)
    int32_t lat0, n_lat;                   // `latent=` input (coupling.py:64-65): A1 columns lat0 .. lat0 + n_lat - 1
    int32_t pad[256 - 15 - kK1 - 3 * kMaxTr];
};
static_assert(sizeof(Header) == 1024, "header layout");
// packed image: header | b1[256] | b2[256] | b3[64] | pad to 4096 | W blocks (see pack kernel)
constexpr uint32_t kOffB1 = 1024, kOffB2 = kOffB1 + kMaxH * 4, kOffB3 = kOffB2 + kMaxH * 4;
constexpr uint32_t kSmallBytes = kOffB3 + kNOut * 4;                 // 3328
constexpr uint32_t kOffW = 4096;

__host__ __device__ inline uint32_t w1_block_bytes(int H) { return (uint32_t)H * 32; }        // one bf16 part
__host__ __device__ inline uint32_t w2_block_bytes(int H) { return (uint32_t)H * 64; }        // hi | lo
__host__ __device__ inline uint32_t w3_block_bytes() { return kNOut * 64; }
__host__ __device__ inline uint32_t packed_bytes(int H, int n_hidden) {
    return kOffW + 6 * w1_block_bytes(H) + (n_hidden == 2 ? (H / 16) * w2_block_bytes(H) : 0) + (H / 16) * w3_block_bytes();
}

// Two configurations of the same kernel (NCG = epilogue warps per TMEM sub-partition = column groups):
//   NCG = 4  16 epilogue warps, one CTA per SM, dim <= 64, H <= 256, 512 TMEM columns
//   NCG = 2   8 epilogue warps, TWO CTAs per SM (dim <= 32, H = 64, weights resident, 256 TMEM columns):
//             small conditioners (configs[3]) are latency-bound per tile -- a second CTA's phases fill the
//             other's waits
template <int NCG>
struct Cfg {
    static constexpr int kEpiThreads = NCG * 4 * 32;
    // NCG = 2: padded to 12 warps -- the register file is allocated for the block rounded up to a multiple of
    // 4 warps, and two CTAs per SM need <= 80 registers per thread at that size (ptxas derives it from here)
    static constexpr int kThreads = (NCG == 4) ? kEpiThreads + 64 : 384;
    static constexpr int kXs = (NCG == 4) ? kMaxDim + 1 : 33;               // row stride of the x tile
    static constexpr uint32_t kColCorr = (NCG == 4) ? 256u : 128u;
    static constexpr uint32_t kTmemCols = (NCG == 4) ? 512u : 256u;
    // shared memory map (A operand size depends on H)
    static constexpr uint32_t kSmXs = 0;                                     // float [128][kXs]
    static constexpr uint32_t kSmRing = (kSmXs + kRows * kXs * 4 + 127) & ~127u;   // 3 x 16 KB
    static constexpr uint32_t kSmSmall = kSmRing + kStages * kSlotBytes;     // header + biases
    static constexpr uint32_t kSmLd = kSmSmall + 3584;                       // float [4][128] log-det partials
    static constexpr uint32_t kSmT = kSmLd + 4 * kRows * 4;                  // float [128] time input
    static constexpr uint32_t kSmBar = kSmT + kRows * 4;
    static constexpr uint32_t kSmA = kSmBar + 256;                           // A operand: 128 x H fp16 hi | lo (>= 24 KB)
    static_assert(kSmRing % 16 == 0 && kSmSmall % 16 == 0 && kSmA % 16 == 0, "alignment");
    static constexpr uint32_t smem_bytes(int H) { return kSmA + (uint32_t)kRows * H * 4; }
};

struct Bars {
    uint64_t setup;
    uint64_t full[kStages], empty[kStages];
    uint64_t a_ready, acc_ready;
    uint32_t tmem_base;
};

constexpr uint32_t kColMain = 0;

struct Args {
    const uint8_t* packed;
    const float* x;
    const float* latent;                   // [rows, lat_stride] or NULL
    int lat_stride;
    const float* t;
    float* y;
    float* ldj;
    int ldj_mode, base_log_prob, inverse;
    long long rows;
    int n_tiles;
};

// exp(v) for the affine scale: 2^p on MUFU.EX2 with p = v log2(e), and the rounding error of that product put back
// as a first-order correction (e ln 2) -- ~3e-7 relative like expf, 5 instructions instead of ~18
__device__ __forceinline__ float exp_fast(float v) {
    const float p = v * 1.4426950408889634f;
    const float e = fmaf(v, 1.4426950408889634f, -p) + v * 1.925963033500011e-08f;     // low part of log2(e) included
    const float r = ex2_approx(p);
    return fmaf(r, e * 0.6931471805599453f, r);
}

// Hidden layer of the conditioner for TWO units at a time on Blackwell's packed fp32 pipe (FADD2 / FMUL2 / FFMA2):
// h = tanh((main + corr) * sc + bias) with the arithmetic of tanh_fast (tc_spline16.cuh), then the fp16 hi | lo split, each
// part as one packed conversion.  Half the issue slots of the scalar form -- the activation passes were 45 % of
// the chain kernel's clocks and ~40 % of the MLP[256,256] kernel's stall samples.
__device__ __forceinline__ void tanh_split2(float2 vm, float2 vc, float2 sc, float2 bias, uint32_t& hi, uint32_t& lo) {
    const float2 pre = __ffma2_rn(__fadd2_rn(vm, vc), sc, bias);
    // tanh|v| = 2 / (1 + t) - 1, t = exp(-2|v|) in (0, 1]: 1 / (1 + t) by MUFU.RCP + one Newton step (~1 ulp of a
    // value in [0.5, 1)), so the absolute error of the result is ~1.5e-7 -- what the consumer (a contraction with
    // O(0.1) weights) sees; 6 issue slots per unit instead of 9.5 for the quotient form
    const float2 p = __fmul2_rn(pre, make_float2(2.885390081777927f, 2.885390081777927f));
    float2 t;
    t.x = ex2_approx(-fabsf(p.x));                            // the -|.| folds into the MUFU operand
    t.y = ex2_approx(-fabsf(p.y));
    const float2 one = make_float2(1.f, 1.f), mone = make_float2(-1.f, -1.f);
    const float2 den = __fadd2_rn(t, one);                    // 1 + t
    const float2 nden = __ffma2_rn(t, mone, mone);            // -(1 + t)
    float2 r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r.x) : "f"(den.x));
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r.y) : "f"(den.y));
    const float2 r1 = __ffma2_rn(__ffma2_rn(nden, r, one), r, r);         // r (2 - den r)
    const float2 th = __ffma2_rn(r1, make_float2(2.f, 2.f), mone);
    const float2 h = make_float2(copysignf(th.x, pre.x), copysignf(th.y, pre.y));
    asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(hi) : "f"(h.y), "f"(h.x));
    const float2 hf = __half22float2(*reinterpret_cast<const __half2*>(&hi));
    const float2 res = __ffma2_rn(hf, mone, h);               // h - hi: exact
    asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(lo) : "f"(res.y), "f"(res.x));
}

// the same for Sigmoid (the only other activation that reaches this kernel, see tcm_layer_supported)
__device__ __forceinline__ void sigmoid_split2(float2 vm, float2 vc, float2 sc, float2 bias, uint32_t& hi, uint32_t& lo) {
    const float2 pre = __ffma2_rn(__fadd2_rn(vm, vc), sc, bias);
    float2 e;
    e.x = ex2_approx(-1.4426950408889634f * fmaxf(pre.x, -80.f));
    e.y = ex2_approx(-1.4426950408889634f * fmaxf(pre.y, -80.f));
    const float2 one = make_float2(1.f, 1.f), mone = make_float2(-1.f, -1.f);
    const float2 den = __fadd2_rn(e, one);
    const float2 nden = __ffma2_rn(e, mone, mone);
    float2 r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r.x) : "f"(den.x));
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r.y) : "f"(den.y));
    const float2 h = __ffma2_rn(__ffma2_rn(r, nden, one), r, r);        // 1 / den with one residual correction
    asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(hi) : "f"(h.y), "f"(h.x));
    const float2 hf = __half22float2(*reinterpret_cast<const __half2*>(&hi));
    const float2 res = __ffma2_rn(hf, mone, h);
    asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(lo) : "f"(res.y), "f"(res.x));
}

template <int NCG>
__global__ void __launch_bounds__(Cfg<NCG>::kThreads, (NCG == 4) ? 1 : 2) tc_mlp_affine_kernel(const Args A) {
    using C = Cfg<NCG>;
    constexpr int kEpiThreads = C::kEpiThreads;
    constexpr int kXsStride = C::kXs;
    constexpr uint32_t kColCorr = C::kColCorr, kTmemCols = C::kTmemCols;
    constexpr uint32_t kSmSmall = C::kSmSmall;
    extern __shared__ __align__(1024) uint8_t smem[];
    float* xs = reinterpret_cast<float*>(smem + C::kSmXs);
    uint8_t* ring = smem + C::kSmRing;
    const Header* hdr = reinterpret_cast<const Header*>(smem + kSmSmall);
    const float* b1s = reinterpret_cast<const float*>(smem + kSmSmall + kOffB1);
    const float* b2s = reinterpret_cast<const float*>(smem + kSmSmall + kOffB2);
    const float* b3s = reinterpret_cast<const float*>(smem + kSmSmall + kOffB3);
    float* ld_s = reinterpret_cast<float*>(smem + C::kSmLd);
    float* t_s = reinterpret_cast<float*>(smem + C::kSmT);
    Bars* bars = reinterpret_cast<Bars*>(smem + C::kSmBar);
    uint8_t* abuf = smem + C::kSmA;

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

    if (tid == 0) {
        mbar_init(&bars->setup, 1);
        for (int i = 0; i < kStages; ++i) { mbar_init(&bars->full[i], 1); mbar_init(&bars->empty[i], 1); }
        mbar_init(&bars->a_ready, NCG * 4);
        mbar_init(&bars->acc_ready, 1);
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

    const int d = hdr->dim, n_tr = hdr->n_tr, n_cond = hdr->n_cond, H = hdr->H, n_hidden = hdr->n_hidden;
    const int act = hdr->act;
    const int kb_h = H / 16;                                   // K blocks of a GEMM whose K is H
    const uint32_t a_part = (uint32_t)kRows * kK1 * 2;         // 8192: one bf16 part of A1
    const uint32_t a_lo = (uint32_t)kRows * H * 2;             // byte offset of the lo half of the A operand
    const uint32_t a_sbo = (uint32_t)(H / 8) * 128;
    const int dshift = ((d & (d - 1)) == 0) ? (31 - __clz(d)) : -1;
    const int my_tiles = (A.n_tiles > (int)blockIdx.x) ? (A.n_tiles - 1 - (int)blockIdx.x) / (int)gridDim.x + 1 : 0;
    const int blocks_per_tile = 6 + (n_hidden == 2 ? kb_h : 0) + kb_h;
    const uint32_t w1b = w1_block_bytes(H), w2b = w2_block_bytes(H), w3b = w3_block_bytes();

    // Small conditioners (all weight blocks together <= the ring, e.g. MLP[64] of configs[3]): the blocks are
    // loaded ONCE and stay resident -- streaming them per 128-row tile was several times the tile's own bytes.
    const uint32_t w_total = 6 * w1b + (n_hidden == 2 ? kb_h * w2b : 0) + kb_h * w3b;
    const bool resident = w_total <= kStages * kSlotBytes;

    if (warp == 0) {
        // ======================= producer =========================================================
        if (lane == 0 && resident) {
            if (my_tiles > 0) {
                mbar_arrive_expect_tx(&bars->full[0], w_total);
                bulk_g2s(ring, A.packed + kOffW, w_total, &bars->full[0]);
            }
            for (int it = 0; it + 1 < my_tiles; ++it) {
                const long long nrow0 = ((long long)blockIdx.x + (long long)(it + 1) * gridDim.x) * kRows;
                const long long nb = min((long long)kRows, A.rows - nrow0) * d * 4;
                const char* src = reinterpret_cast<const char*>(A.x + nrow0 * d);
                if (nb >= 16 && ((reinterpret_cast<uintptr_t>(src) & 15) == 0))
                    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(src), "r"((uint32_t)(nb & ~15LL)) : "memory");
            }
        } else if (lane == 0) {
            uint32_t cc = 0;
            for (int it = 0; it < my_tiles; ++it) {
                if (it + 1 < my_tiles) {
                    const long long nrow0 = ((long long)blockIdx.x + (long long)(it + 1) * gridDim.x) * kRows;
                    const long long nb = min((long long)kRows, A.rows - nrow0) * d * 4;
                    const char* src = reinterpret_cast<const char*>(A.x + nrow0 * d);
                    if (nb >= 16 && ((reinterpret_cast<uintptr_t>(src) & 15) == 0))
                        asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(src), "r"((uint32_t)(nb & ~15LL)) : "memory");
                }
                const uint8_t* src = A.packed + kOffW;
                for (int b = 0; b < blocks_per_tile; ++b, ++cc) {
                    const uint32_t bytes = (b < 6) ? w1b : ((n_hidden == 2 && b < 6 + kb_h) ? w2b : w3b);
                    const uint32_t st = cc % kStages, use = cc / kStages;
                    mbar_wait_relaxed(&bars->empty[st], (use & 1) ^ 1);
                    mbar_arrive_expect_tx(&bars->full[st], bytes);
                    bulk_g2s(ring + st * kSlotBytes, src, bytes, &bars->full[st]);
                    src += bytes;
                }
            }
        }
    } else if (warp == 1) {
        // ======================= UMMA issuer ======================================================
        if (lane == 0) {
            const uint32_t idesc1 = make_idesc(FMT_BF16, 128, H);
            const uint32_t idesc2 = make_idesc(FMT_F16, 128, H);
            const uint32_t idesc3 = make_idesc(FMT_F16, 128, kNOut);
            const uint32_t a0 = smem_u32(abuf);
            const uint32_t dmain = tmem + kColMain, dcorr = tmem + kColCorr;
            uint32_t cc = 0, ause = 0;
            if (resident && my_tiles > 0) { mbar_wait(&bars->full[0], 0); tc_fence_after(); }
            for (int it = 0; it < my_tiles; ++it) {
                // ---- layer 1: bf16x3 x bf16x3, blocks ordered (pb = 2, 1, 0) x (kb = 0, 1) -------------
                mbar_wait(&bars->a_ready, ause & 1); ++ause;
                tc_fence_after();
                uint32_t acc_m = 0, acc_c = 0;
                uint32_t roff = 0;                          // resident: byte offset of the block in the image
                for (int b = 0; b < 6; ++b, ++cc) {
                    const int pb = 2 - b / 2, kb = b & 1;
                    const uint32_t st = cc % kStages, use = cc / kStages;
                    if (!resident) { mbar_wait(&bars->full[st], use & 1); tc_fence_after(); }
                    const uint64_t bd = make_smem_desc(smem_u32(ring) + (resident ? roff : st * kSlotBytes), 128, 256);
                    roff += w1b;
                    for (int pa = 2; pa >= 0; --pa) {
                        if (pa == 2 && pb == 2) continue;
                        const uint64_t ad = make_smem_desc(a0 + pa * a_part + kb * 256, 128, 512);
                        if (pa == 0 && pb == 0) { umma_f16(dmain, ad, bd, idesc1, acc_m); acc_m = 1; }
                        else { umma_f16(dcorr, ad, bd, idesc1, acc_c); acc_c = 1; }
                    }
                    if (!resident) umma_commit(&bars->empty[st]);
                }
                umma_commit(&bars->acc_ready);
                // ---- hidden -> hidden (optional) and hidden -> output: fp16 hi | lo -------------------
                for (int layer = (n_hidden == 2 ? 0 : 1); layer < 2; ++layer) {
                    mbar_wait(&bars->a_ready, ause & 1); ++ause;
                    tc_fence_after();
                    const bool last = (layer == 1);
                    const uint32_t idesc = last ? idesc3 : idesc2;
                    const uint32_t lo_off = last ? kNOut * 32 : (uint32_t)H * 32;     // lo half inside a block
                    acc_m = acc_c = 0;
                    for (int kb = 0; kb < kb_h; ++kb, ++cc) {
                        const uint32_t st = cc % kStages, use = cc / kStages;
                        if (!resident) { mbar_wait(&bars->full[st], use & 1); tc_fence_after(); }
                        const uint32_t bb = smem_u32(ring) + (resident ? roff : st * kSlotBytes);
                        roff += last ? w3b : w2b;
                        const uint64_t b_hi = make_smem_desc(bb, 128, 256), b_lo = make_smem_desc(bb + lo_off, 128, 256);
                        const uint64_t a_hi = make_smem_desc(a0 + kb * 256, 128, a_sbo);
                        const uint64_t a_l = make_smem_desc(a0 + a_lo + kb * 256, 128, a_sbo);
                        umma_f16(dcorr, a_l, b_hi, idesc, acc_c); acc_c = 1;
                        umma_f16(dcorr, a_hi, b_lo, idesc, 1);
                        umma_f16(dmain, a_hi, b_hi, idesc, acc_m); acc_m = 1;
                        if (!resident) umma_commit(&bars->empty[st]);
                    }
                    umma_commit(&bars->acc_ready);
                }
            }
        }
    } else if (warp < kEpiWarp0 + NCG * 4) {
        // ======================= epilogue warps ====================================================
        const int q = warp & 3;
        const int cg = (warp - ((q >= kEpiWarp0) ? q : q + 4)) >> 2;      // column group 0..NCG-1
        const int etid = tid - kEpiWarp0 * 32;
        const int row = q * 32 + lane;
        float* xrow = xs + row * kXsStride;
        const uint32_t lane_sel = (uint32_t)(q * 32) << 16;
        const bool want_ld = A.ldj_mode != STB_LDJ_NONE;
        const bool inverse = A.inverse != 0;
        const float s_mid = hdr->s_mid, s_out = hdr->s_out;
        uint32_t acc_use = 0;

        for (int it = 0; it < my_tiles; ++it) {
            const long long row0 = ((long long)blockIdx.x + (long long)it * gridDim.x) * kRows;
            const int nrows = (int)min((long long)kRows, A.rows - row0);
            // ---- stage x -----------------------------------------------------------------------------
            {
                const float* xg = A.x + row0 * d;
                const int n = nrows * d;
                if ((d & 3) == 0 && ((reinterpret_cast<uintptr_t>(xg) & 15) == 0)) {
                    // 16-byte loads, four in flight per thread before the first store (the scalar loop was a
                    // chain of ~16 exposed global round trips per tile: 12.6 % of the kernel's stall samples)
                    const int n4 = (kRows * d) >> 2;
                    for (int i0 = etid; i0 < n4; i0 += kEpiThreads * 4) {
                        float4 v[4];
#pragma unroll
                        for (int u = 0; u < 4; ++u) {
                            const int i = i0 + u * kEpiThreads;
                            v[u] = (i < n4 && i * 4 < n) ? __ldg(reinterpret_cast<const float4*>(xg) + i)
                                                         : make_float4(0.f, 0.f, 0.f, 0.f);
                        }
#pragma unroll
                        for (int u = 0; u < 4; ++u) {
                            const int i = i0 + u * kEpiThreads;
                            if (i < n4) {
                                const int r = (dshift >= 0) ? ((i * 4) >> dshift) : (i * 4) / d, c = (i * 4) - r * d;
                                float* dst = xs + r * kXsStride + c;
                                dst[0] = v[u].x; dst[1] = v[u].y; dst[2] = v[u].z; dst[3] = v[u].w;
                            }
                        }
                    }
                } else {
                    for (int i = etid; i < kRows * d; i += kEpiThreads) {
                        const int r = (dshift >= 0) ? (i >> dshift) : i / d, c = i - r * d;
                        xs[r * kXsStride + c] = (i < n) ? __ldg(xg + i) : 0.f;
                    }
                }
                if (etid < kRows) t_s[etid] = (A.t != nullptr && etid < nrows) ? __ldg(A.t + row0 + etid) : 0.f;
            }
            named_bar_sync(1, kEpiThreads);
            // ---- A1: 8 of the 32 conditioning columns of this row, three bf16 parts ---------------------
            {
#pragma unroll 1
                for (int kc = cg; kc < kK1 / 8; kc += NCG) {
                    const uint32_t off = (uint32_t)(row >> 3) * 512 + (uint32_t)(row & 7) * 16 + kc * 128;
                    __align__(16) __nv_bfloat16 q0[8], q1[8], q2[8];
#pragma unroll
                    for (int u = 0; u < 8; ++u) {
                        const int k = kc * 8 + u;
                        float v = (k < n_cond) ? xrow[hdr->cond_idx[k]] : ((k == hdr->time_col) ? t_s[row] : 0.f);
                        if (k >= hdr->lat0 && k < hdr->lat0 + hdr->n_lat && row < nrows)
                            v = __ldg(A.latent + (row0 + row) * A.lat_stride + (k - hdr->lat0));
                        split_bf16x3(v, q0[u], q1[u], q2[u]);
                    }
                    *reinterpret_cast<uint4*>(abuf + off) = *reinterpret_cast<const uint4*>(q0);
                    *reinterpret_cast<uint4*>(abuf + a_part + off) = *reinterpret_cast<const uint4*>(q1);
                    *reinterpret_cast<uint4*>(abuf + 2 * a_part + off) = *reinterpret_cast<const uint4*>(q2);
                }
                fence_proxy_async_smem();
                __syncwarp();
                if (lane == 0) mbar_arrive(&bars->a_ready);
            }
            // ---- hidden layers: h = act((main + corr) * s + b) -> fp16 hi | lo A operand -----------------
            for (int layer = 0; layer < n_hidden; ++layer) {
                mbar_wait_sleep(&bars->acc_ready, acc_use & 1, 64); ++acc_use;
                tc_fence_after();
                const float sc = (layer == 0) ? 1.f : s_mid;
                const float* bias = (layer == 0) ? b1s : b2s;
                const int cols = H / NCG;                        // this warp's share of the hidden units
                const uint32_t a_row = (uint32_t)(row >> 3) * a_sbo + (uint32_t)(row & 7) * 16;
                for (int cb = 0; cb < cols; cb += 16) {
                    const int c0 = cg * cols + cb;
                    float vm[16], vc[16];
                    tmem_ld16(tmem + lane_sel + kColMain + c0, vm);
                    tmem_ld16(tmem + lane_sel + kColCorr + c0, vc);
                    tmem_ld_wait();
                    __align__(16) __half hh[16], hl[16];
                    if (act == STB_ACT_TANH) {
                        const float2* b2p = reinterpret_cast<const float2*>(bias + c0);
#pragma unroll
                        for (int i = 0; i < 8; ++i)
                            tanh_split2(make_float2(vm[2 * i], vm[2 * i + 1]), make_float2(vc[2 * i], vc[2 * i + 1]),
                                        make_float2(sc, sc), b2p[i], reinterpret_cast<uint32_t*>(hh)[i],
                                        reinterpret_cast<uint32_t*>(hl)[i]);
                    } else {                                   // STB_ACT_SIGMOID
                        const float2* b2p = reinterpret_cast<const float2*>(bias + c0);
#pragma unroll
                        for (int i = 0; i < 8; ++i)
                            sigmoid_split2(make_float2(vm[2 * i], vm[2 * i + 1]), make_float2(vc[2 * i], vc[2 * i + 1]),
                                           make_float2(sc, sc), b2p[i], reinterpret_cast<uint32_t*>(hh)[i],
                                           reinterpret_cast<uint32_t*>(hl)[i]);
                    }
#pragma unroll
                    for (int half8 = 0; half8 < 2; ++half8) {
                        const int kc = (c0 >> 3) + half8;
                        *reinterpret_cast<uint4*>(abuf + a_row + kc * 128) = *reinterpret_cast<const uint4*>(hh + half8 * 8);
                        *reinterpret_cast<uint4*>(abuf + a_lo + a_row + kc * 128) = *reinterpret_cast<const uint4*>(hl + half8 * 8);
                    }
                }
                tc_fence_before();
                fence_proxy_async_smem();
                __syncwarp();
                if (lane == 0) mbar_arrive(&bars->a_ready);
            }
            // ---- output layer: [log_scale | shift] of this warp's 8 transformed dims ---------------------
            mbar_wait_sleep(&bars->acc_ready, acc_use & 1, 64); ++acc_use;
            tc_fence_after();
            float ld_acc = 0.f;
#pragma unroll 1
            for (int og = cg; og < kMaxTr / 8; og += NCG) {
                float lm[8], lc[8], sm[8], sc_[8];
                tmem_ld8(tmem + lane_sel + kColMain + og * 8, lm);
                tmem_ld8(tmem + lane_sel + kColCorr + og * 8, lc);
                tmem_ld8(tmem + lane_sel + kColMain + kMaxTr + og * 8, sm);
                tmem_ld8(tmem + lane_sel + kColCorr + kMaxTr + og * 8, sc_);
                tmem_ld_wait();
#pragma unroll
                for (int u = 0; u < 8; ++u) {
                    const int ji = og * 8 + u;
                    if (ji < n_tr) {
                        const int j = hdr->tr_idx[ji];
                        float ls = fmaf(lm[u] + lc[u], s_out, b3s[ji]);
                        float sh = fmaf(sm[u] + sc_[u], s_out, b3s[kMaxTr + ji]);
                        if (hdr->cont) {                       // coupling.py:199-205
                            const float tv = t_s[row];
                            ls *= hdr->ts_ls[ji] * tv;
                            sh *= hdr->ts_sh[ji] * tv;
                        }
                        const float xv = xrow[j];
                        if (inverse) { xrow[j] = (xv - sh) * exp_fast(-ls); ld_acc -= ls; }
                        else { xrow[j] = xv * exp_fast(ls) + sh; ld_acc += ls; }
                    }
                }
            }
            tc_fence_before();
            ld_s[cg * kRows + row] = ld_acc;
            named_bar_sync(1, kEpiThreads);
            if (cg == 0 && want_ld && row < nrows) {
                float tot = (NCG == 4) ? (ld_s[row] + ld_s[kRows + row]) + (ld_s[2 * kRows + row] + ld_s[3 * kRows + row])
                                       : ld_s[row] + ld_s[kRows + row];
                if (A.base_log_prob) {
                    float b = 0.f;
                    for (int c = 0; c < d; ++c) { const float v = xrow[c]; b += -0.5f * v * v - 0.91893853320467274178f; }
                    tot += b;
                }
                float* dst = A.ldj + row0 + row;
                *dst = (A.ldj_mode == STB_LDJ_ADD) ? (*dst + tot) : tot;
            }
            {
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
                        const int r = (dshift >= 0) ? (i >> dshift) : i / d, c = i - r * d;
                        yg[i] = xs[r * kXsStride + c];
                    }
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
// Wide conditioners, pipelined: tc_mlp_pipe_kernel
// -----------------------------------------------------------------------------------------------
// Same layer as tc_mlp_affine_kernel<4> (BASELINE.json configs[1]: MLP[256,256]) restructured so that the tensor pipe and
// the activation passes overlap.  In that kernel every GEMM waits for the whole previous activation pass and every
// activation pass for the whole GEMM (40 k clocks per 128-row tile for 9.7 k clocks of tensor work) because TMEM is full
// (main + corr accumulators of a 256-wide layer) and the next A operand lives in 128 KB of shared memory.  Here:
//   * every GEMM uses ONE accumulator (per K block: lo*hi, hi*lo, then hi*hi -- the order tc_hwide.cu's hidden GEMM
//     uses), so layer l's accumulator [0, H) and layer l+1's [256, 256 + H) coexist;
//   * the hidden activations go back INTO the accumulator columns just consumed (tcgen05.st) and are read from TMEM as
//     the next GEMM's A operand: no shared-memory A buffer, no proxy fence;
//   * a warp (TMEM sub-partition q, column quarter g) activates its columns 16 at a time; after every such WAVE j the
//     issuer is told (wave barrier, 16 arrivals) and runs the next GEMM over the four K blocks {g H/64 + j} that just
//     became available, while the warps are already on wave j + 1 (one barrier per K block -- 4 arrivals -- measured
//     10 % slower: the issuer's extra waits sit on the critical path);
//   * the epilogue warps prepare tile i + 1 inside tile i's waits: its rows are staged (second xs buffer) while GEMM2's
//     last K blocks drain, its A1 operand is split while GEMM3's drain, and its GEMM1 runs under tile i's affine
//     output / store phase (the issuer only waits until the output accumulator has been read: d3_read).
// Weights stream one 16-wide K block per ring item (<= 16 KB), in the order the issuer consumes them.
constexpr int kPipeStages = 6;
constexpr int kPipeThreads = (2 + 16) * 32;

struct PipeBars {
    uint64_t setup;
    uint64_t full[kPipeStages], empty[kPipeStages];
    uint64_t a1_ready, acc1_full, acc2_full, acc3_full, d3_read;
    uint64_t wave1[4], wave2[4];
};
static_assert(sizeof(PipeBars) <= 256, "barrier block");

constexpr uint32_t kPipeXsBytes = (kRows * (kMaxDim + 1) * 4 + 127) & ~127u; // float [128][65], one per tile in flight
constexpr uint32_t kPipeSmXs = 0;
constexpr uint32_t kPipeSmA1 = 2 * kPipeXsBytes;                             // 3 x 8 KB (bf16x3 of [128 x 32])
constexpr uint32_t kPipeSmSmall = kPipeSmA1 + 3 * kRows * kK1 * 2;
constexpr uint32_t kPipeSmLd = kPipeSmSmall + 3584;                          // float [4][128]
constexpr uint32_t kPipeSmT = kPipeSmLd + 4 * kRows * 4;                     // float [2][128]
constexpr uint32_t kPipeSmBar = kPipeSmT + 2 * kRows * 4;
constexpr uint32_t kPipeSmRing = (kPipeSmBar + 256 + 127) & ~127u;
__host__ __device__ inline uint32_t pipe_slot_bytes(int H) { return (uint32_t)H * 64; }
__host__ __device__ inline uint32_t pipe_smem_bytes(int H) { return kPipeSmRing + kPipeStages * pipe_slot_bytes(H); }

// this warp's 16 columns starting at c0 of the accumulator at `acc` -> h (fp16 hi at +0, lo at +8), in place
__device__ __forceinline__ void pipe_activate16(uint32_t acc, int c0, float sc, const float* bias, int act) {
    float v[16];
    tmem_ld16(acc + c0, v);
    tmem_ld_wait();
    uint32_t hh[8], hl[8];
    const float2* b2p = reinterpret_cast<const float2*>(bias + c0);
    const float2 z = make_float2(0.f, 0.f);
    if (act == STB_ACT_TANH) {
#pragma unroll
        for (int i = 0; i < 8; ++i) tanh_split2(make_float2(v[2 * i], v[2 * i + 1]), z, make_float2(sc, sc), b2p[i], hh[i], hl[i]);
    } else {
#pragma unroll
        for (int i = 0; i < 8; ++i) sigmoid_split2(make_float2(v[2 * i], v[2 * i + 1]), z, make_float2(sc, sc), b2p[i], hh[i], hl[i]);
    }
    tmem_st8(acc + c0, hh);
    tmem_st8(acc + c0 + 8, hl);
    tmem_st_wait();
}

__global__ void __launch_bounds__(kPipeThreads, 1) tc_mlp_pipe_kernel(const Args A) {
    constexpr int kXsStride = kMaxDim + 1;
    constexpr int kEpiThreads = 16 * 32;
    extern __shared__ __align__(1024) uint8_t smem[];
    __shared__ uint32_t tmem_base_s;
    float* xs = reinterpret_cast<float*>(smem + kPipeSmXs);
    uint8_t* a1buf = smem + kPipeSmA1;
    const Header* hdr = reinterpret_cast<const Header*>(smem + kPipeSmSmall);
    const float* b1s = reinterpret_cast<const float*>(smem + kPipeSmSmall + kOffB1);
    const float* b2s = reinterpret_cast<const float*>(smem + kPipeSmSmall + kOffB2);
    const float* b3s = reinterpret_cast<const float*>(smem + kPipeSmSmall + kOffB3);
    float* ld_s = reinterpret_cast<float*>(smem + kPipeSmLd);
    float* t_s = reinterpret_cast<float*>(smem + kPipeSmT);
    PipeBars* bars = reinterpret_cast<PipeBars*>(smem + kPipeSmBar);
    uint8_t* ring = smem + kPipeSmRing;

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    if (tid == 0) {
        mbar_init(&bars->setup, 1);
        for (int i = 0; i < kPipeStages; ++i) { mbar_init(&bars->full[i], 1); mbar_init(&bars->empty[i], 1); }
        mbar_init(&bars->a1_ready, 16);
        mbar_init(&bars->acc1_full, 1);
        mbar_init(&bars->acc2_full, 1);
        mbar_init(&bars->acc3_full, 1);
        mbar_init(&bars->d3_read, 16);
        for (int j = 0; j < 4; ++j) { mbar_init(&bars->wave1[j], 16); mbar_init(&bars->wave2[j], 16); }
        fence_mbar_init();
    }
    if (warp == 1) tmem_alloc(&tmem_base_s, 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_base_s;
    if (tid == 0) {
        mbar_arrive_expect_tx(&bars->setup, kSmallBytes);
        bulk_g2s(smem + kPipeSmSmall, A.packed, kSmallBytes, &bars->setup);
    }
    mbar_wait(&bars->setup, 0);

    const int d = hdr->dim, n_tr = hdr->n_tr, n_cond = hdr->n_cond, H = hdr->H, n_hidden = hdr->n_hidden, act = hdr->act;
    const int cq = H / 4;                        // columns of a column quarter
    const int nw = cq / 16;                      // waves = K blocks per quarter
    const uint32_t slot = pipe_slot_bytes(H);
    const uint32_t w1b = w1_block_bytes(H), w2b = w2_block_bytes(H), w3b = w3_block_bytes();
    const uint32_t col_d3 = (n_hidden == 2) ? 0u : 256u;          // output accumulator: over the dead h1, or beside it
    const int my_tiles = (A.n_tiles > (int)blockIdx.x) ? (A.n_tiles - 1 - (int)blockIdx.x) / (int)gridDim.x + 1 : 0;
    const uint8_t* img_w2 = A.packed + kOffW + 6 * w1b;
    const uint8_t* img_w3 = img_w2 + (n_hidden == 2 ? (uint32_t)(H / 16) * w2b : 0u);

    if (warp == 0) {
        // ======================= producer: one K block per ring item, in consumption order =======================
        if (lane == 0) {
            uint32_t rc = 0;
            auto put = [&](const uint8_t* src, uint32_t bytes) {
                const uint32_t st = rc % kPipeStages, use = rc / kPipeStages;
                mbar_wait_relaxed(&bars->empty[st], (use & 1) ^ 1);
                mbar_arrive_expect_tx(&bars->full[st], bytes);
                bulk_g2s(ring + st * slot, src, bytes, &bars->full[st]);
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
                for (int b = 0; b < 6; ++b) put(A.packed + kOffW + (uint32_t)b * w1b, w1b);
                if (n_hidden == 2)
                    for (int j = 0; j < nw; ++j)
                        for (int g = 0; g < 4; ++g) put(img_w2 + (uint32_t)(g * nw + j) * w2b, w2b);
                for (int j = 0; j < nw; ++j)
                    for (int g = 0; g < 4; ++g) put(img_w3 + (uint32_t)(g * nw + j) * w3b, w3b);
            }
        }
    } else if (warp == 1) {
        // ======================= UMMA issuer ===========================================================================
        if (lane == 0) {
            const uint32_t idesc1 = make_idesc(FMT_BF16, 128, H);
            const uint32_t idesc2 = make_idesc(FMT_F16, 128, H);
            const uint32_t idesc3 = make_idesc(FMT_F16, 128, kNOut);
            const uint32_t a0 = smem_u32(a1buf);
            constexpr uint32_t a_part = (uint32_t)kRows * kK1 * 2;
            uint32_t rc = 0, tp = 0;
            for (int it = 0; it < my_tiles; ++it, tp ^= 1) {
                // ---- layer 1: bf16x3 x bf16x3 into one accumulator, blocks (pb = 2, 1, 0) x (kb = 0, 1) as they arrive ----
                mbar_wait_relaxed(&bars->a1_ready, tp);
                if (it > 0) mbar_wait_relaxed(&bars->d3_read, tp ^ 1);      // tile it-1's output accumulator has been read
                tc_fence_after();
                uint32_t acc = 0;
                for (int b = 0; b < 6; ++b, ++rc) {
                    const int pb = 2 - b / 2, kb = b & 1;
                    const uint32_t st = rc % kPipeStages, use = rc / kPipeStages;
                    mbar_wait_relaxed(&bars->full[st], use & 1);
                    tc_fence_after();
                    const uint64_t bd = make_smem_desc(smem_u32(ring + st * slot), 128, 256);
                    for (int pa = 2; pa >= 0; --pa) {
                        if (pa == 2 && pb == 2) continue;
                        umma_f16(tmem, make_smem_desc(a0 + pa * a_part + kb * 256, 128, 512), bd, idesc1, acc);
                        acc = 1;
                    }
                    umma_commit(&bars->empty[st]);
                }
                umma_commit(&bars->acc1_full);
                // ---- hidden -> hidden (optional) and hidden -> output, four K blocks per activation wave --------------------
                for (int layer = (n_hidden == 2 ? 0 : 1); layer < 2; ++layer) {
                    const bool last = (layer == 1);
                    const uint32_t a_base = tmem + ((last && n_hidden == 2) ? 256u : 0u);      // h1 at [0, H), h2 at [256, 256 + H)
                    const uint32_t dcol = last ? tmem + col_d3 : tmem + 256u;
                    const uint32_t idesc = last ? idesc3 : idesc2;
                    const uint32_t lo_off = last ? kNOut * 32 : (uint32_t)H * 32;
                    uint64_t* wave = (last && n_hidden == 2) ? bars->wave2 : bars->wave1;
                    acc = 0;
                    for (int j = 0; j < nw; ++j) {
                        mbar_wait_relaxed(&wave[j], tp);
                        for (int g = 0; g < 4; ++g, ++rc) {
                            const int kb = g * nw + j;
                            const uint32_t st = rc % kPipeStages, use = rc / kPipeStages;
                            mbar_wait_relaxed(&bars->full[st], use & 1);
                            tc_fence_after();
                            const uint32_t bb = smem_u32(ring + st * slot);
                            const uint64_t b_hi = make_smem_desc(bb, 128, 256), b_lo = make_smem_desc(bb + lo_off, 128, 256);
                            const uint32_t a_hi = a_base + (uint32_t)kb * 16, a_lo = a_hi + 8;
                            umma_f16_ts(dcol, a_lo, b_hi, idesc, acc); acc = 1;
                            umma_f16_ts(dcol, a_hi, b_lo, idesc, 1);
                            umma_f16_ts(dcol, a_hi, b_hi, idesc, 1);
                            umma_commit(&bars->empty[st]);
                        }
                    }
                    umma_commit(last ? &bars->acc3_full : &bars->acc2_full);
                }
            }
        }
    } else {
        // ======================= epilogue warps ===========================================================================
        const int q = warp & 3;
        const int g = (warp - 2) >> 2;
        const int etid = tid - 64;
        const int row = q * 32 + lane;
        const uint32_t lane_sel = (uint32_t)(q * 32) << 16;
        const bool want_ld = A.ldj_mode != STB_LDJ_NONE;
        const bool inverse = A.inverse != 0;
        const float s_mid = hdr->s_mid, s_out = hdr->s_out;
        const int dshift = ((d & (d - 1)) == 0) ? (31 - __clz(d)) : -1;
        uint32_t tp = 0;

        // rows of tile `it` -> xs buffer it & 1 (zero rows past the end), t likewise
        auto stage_x = [&](int it) {
            const long long row0 = ((long long)blockIdx.x + (long long)it * gridDim.x) * kRows;
            const int nrows = (int)min((long long)kRows, A.rows - row0);
            float* xb = xs + (it & 1) * (kPipeXsBytes / 4);
            const float* xg = A.x + row0 * d;
            const int n = nrows * d;
            if ((d & 3) == 0 && ((reinterpret_cast<uintptr_t>(xg) & 15) == 0)) {
                const int n4 = (kRows * d) >> 2;
                for (int i = etid; i < n4; i += kEpiThreads) {
                    const float4 v = (i * 4 < n) ? __ldg(reinterpret_cast<const float4*>(xg) + i) : make_float4(0.f, 0.f, 0.f, 0.f);
                    const int r = (dshift >= 0) ? ((i * 4) >> dshift) : (i * 4) / d, c = (i * 4) - r * d;
                    float* dst = xb + r * kXsStride + c;
                    dst[0] = v.x; dst[1] = v.y; dst[2] = v.z; dst[3] = v.w;
                }
            } else {
                for (int i = etid; i < kRows * d; i += kEpiThreads) {
                    const int r = i / d, c = i - r * d;
                    xb[r * kXsStride + c] = (i < n) ? __ldg(xg + i) : 0.f;
                }
            }
            if (etid < kRows) t_s[(it & 1) * kRows + etid] = (A.t != nullptr && etid < nrows) ? __ldg(A.t + row0 + etid) : 0.f;
            named_bar_sync(1, kEpiThreads);
        };
        // A1 of tile `it`: 8 of the 32 conditioning columns of this row (column group g), three bf16 parts
        auto split_a1 = [&](int it) {
            const float* xr = xs + (it & 1) * (kPipeXsBytes / 4) + row * kXsStride;
            const uint32_t off = (uint32_t)(row >> 3) * 512 + (uint32_t)(row & 7) * 16 + (uint32_t)g * 128;
            constexpr uint32_t a_part = (uint32_t)kRows * kK1 * 2;
            __align__(16) __nv_bfloat16 q0[8], q1[8], q2[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const int k = g * 8 + u;
                float v = (k < n_cond) ? xr[hdr->cond_idx[k]] : ((k == hdr->time_col) ? t_s[(it & 1) * kRows + row] : 0.f);
                if (k >= hdr->lat0 && k < hdr->lat0 + hdr->n_lat) {
                    const long long grow = ((long long)blockIdx.x + (long long)it * gridDim.x) * kRows + row;
                    if (grow < A.rows) v = __ldg(A.latent + grow * A.lat_stride + (k - hdr->lat0));
                }
                split_bf16x3(v, q0[u], q1[u], q2[u]);
            }
            *reinterpret_cast<uint4*>(a1buf + off) = *reinterpret_cast<const uint4*>(q0);
            *reinterpret_cast<uint4*>(a1buf + a_part + off) = *reinterpret_cast<const uint4*>(q1);
            *reinterpret_cast<uint4*>(a1buf + 2 * a_part + off) = *reinterpret_cast<const uint4*>(q2);
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) mbar_arrive(&bars->a1_ready);
        };

        if (my_tiles > 0) {
            stage_x(0);
            split_a1(0);       // the A1 buffer is free: nothing has been issued yet
        }
        for (int it = 0; it < my_tiles; ++it, tp ^= 1) {
            const long long row0 = ((long long)blockIdx.x + (long long)it * gridDim.x) * kRows;
            const int nrows = (int)min((long long)kRows, A.rows - row0);
            float* xrow = xs + (it & 1) * (kPipeXsBytes / 4) + row * kXsStride;
            const bool more = it + 1 < my_tiles;
            // ---- hidden layer 1 in place, wave by wave: the next GEMM runs behind ---------------------------------------------
            mbar_wait_sleep(&bars->acc1_full, tp, 32);       // GEMM1(it) done: the A1 buffer is free as well
            tc_fence_after();
            for (int j = 0; j < nw; ++j) {
                pipe_activate16(tmem + lane_sel, g * cq + 16 * j, 1.f, b1s, act);
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&bars->wave1[j]);
            }
            if (more) stage_x(it + 1);                       // while the next GEMM's last K blocks drain
            if (n_hidden == 2) {
                mbar_wait_sleep(&bars->acc2_full, tp, 32);
                tc_fence_after();
                for (int j = 0; j < nw; ++j) {
                    pipe_activate16(tmem + lane_sel + 256, g * cq + 16 * j, s_mid, b2s, act);
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&bars->wave2[j]);
                }
            }
            if (more) split_a1(it + 1);                      // the A1 buffer is free since acc1_full; GEMM3's last blocks drain
            // ---- output layer: [log_scale | shift] of this warp's 8 transformed dims (one accumulator) ------------------
            mbar_wait_sleep(&bars->acc3_full, tp, 32);
            tc_fence_after();
            float ld_acc = 0.f;
            {
                float lm[8], sm[8];
                if (g * 8 < n_tr) {
                    tmem_ld8(tmem + lane_sel + col_d3 + g * 8, lm);
                    tmem_ld8(tmem + lane_sel + col_d3 + kMaxTr + g * 8, sm);
                    tmem_ld_wait();
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&bars->d3_read);   // GEMM1 of the next tile may overwrite the accumulator
                if (g * 8 < n_tr) {
#pragma unroll
                    for (int u = 0; u < 8; ++u) {
                        const int ji = g * 8 + u;
                        if (ji < n_tr) {
                            const int j = hdr->tr_idx[ji];
                            float ls = fmaf(lm[u], s_out, b3s[ji]);
                            float sh = fmaf(sm[u], s_out, b3s[kMaxTr + ji]);
                            if (hdr->cont) {                       // coupling.py:199-205
                                const float tv = t_s[(it & 1) * kRows + row];
                                ls *= hdr->ts_ls[ji] * tv;
                                sh *= hdr->ts_sh[ji] * tv;
                            }
                            const float xv = xrow[j];
                            if (inverse) { xrow[j] = (xv - sh) * exp_fast(-ls); ld_acc -= ls; }
                            else { xrow[j] = xv * exp_fast(ls) + sh; ld_acc += ls; }
                        }
                    }
                }
            }
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
                const float* xb = xs + (it & 1) * (kPipeXsBytes / 4);
                float* yg = A.y + row0 * d;
                const int n = nrows * d;
                if ((d & 3) == 0 && ((reinterpret_cast<uintptr_t>(yg) & 15) == 0)) {
                    const int n4 = n >> 2;
                    for (int i = etid; i < n4; i += kEpiThreads) {
                        const int r = (dshift >= 0) ? ((i * 4) >> dshift) : (i * 4) / d, c = (i * 4) - r * d;
                        const float* src = xb + r * kXsStride + c;
                        reinterpret_cast<float4*>(yg)[i] = make_float4(src[0], src[1], src[2], src[3]);
                    }
                } else {
                    for (int i = etid; i < n; i += kEpiThreads) {
                        const int r = i / d, c = i - r * d;
                        yg[i] = xb[r * kXsStride + c];
                    }
                }
            }
            named_bar_sync(1, kEpiThreads);      // ld_s, and this xs buffer (staged again two tiles on), are free
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem, 512);
}

// -----------------------------------------------------------------------------------------------
// CHAIN: every layer of an affine / continuous-affine flow in ONE launch (flow.py:104-107, 118-125 and
// NeuralFlow.forward, flow.py:172-184, inside the kernel)
// -----------------------------------------------------------------------------------------------
// Small conditioners only (H = 64, dim <= 32 -- BASELINE.json configs[3]): the weight blocks of ALL chained
// layers (28 KB each for MLP[k -> 64 -> 2 dim]) are loaded once per CTA and stay in shared memory, a 128-row
// tile is read once, every layer is applied to it in place, and it is written once: 132 B of DRAM traffic per
// row for the whole flow instead of per layer.  Such a tile is latency-bound (five dependent phases per layer:
// A1 split -> GEMM1 -> activation -> GEMM2 -> affine), so one CTA runs V independent "virtual CTAs" -- each
// with its own tile, barriers, A-operand buffer, issuer warp, eight epilogue warps and 128 TMEM columns --
// that share the resident weights and fill each other's waits (the per-layer kernel gets the same effect from
// two CTAs per SM, which cannot share the weights).

constexpr int kMaxChainM = 8;
constexpr int kVcThreads = 384;            // per virtual CTA: producer, issuer, 8 epilogue warps, 2 idle (register budget)
constexpr int kChainNCG = 2;
constexpr uint32_t kSmallSlot = 3584;      // header | biases of one layer
constexpr uint32_t kVcCols = 128;          // TMEM columns of one virtual CTA: main [0, 64) | corr [64, 128)

struct ChainArgs {
    const uint8_t* packed[kMaxChainM];
    uint32_t w_off[kMaxChainM], w_bytes[kMaxChainM];
    int n_layers, dim, xs_stride;
    uint32_t sm_w, sm_vc, vc_bytes;        // shared-memory map: resident weights, first virtual CTA, its size
    const float* x;
    const float* t;
    float* y;
    float* ldj;
    int ldj_mode, base_log_prob, inverse;
    long long rows;
    int n_tiles;
    int permuted;                          // permutations between the layers, folded into the index lists
    ChainPerm perm;
};

struct VcBars {
    uint64_t a_ready, acc_ready;
};

template <int V>
__global__ void __launch_bounds__(V * kVcThreads, 1) tc_mlp_chain_kernel(const ChainArgs A) {
    constexpr int NCG = kChainNCG;
    constexpr int kEpiThreads = NCG * 4 * 32;
    extern __shared__ __align__(1024) uint8_t smem[];
    __shared__ uint64_t w_full;
    __shared__ uint32_t tmem_base_s;

    const int tid = threadIdx.x;
    const int vc = tid / kVcThreads, vtid = tid - vc * kVcThreads;
    const int warp = vtid >> 5, lane = vtid & 31;
    const int d = A.dim, L = A.n_layers, xs_stride = A.xs_stride;

    uint8_t* vbase = smem + A.sm_vc + (uint32_t)vc * A.vc_bytes;
    float* xs = reinterpret_cast<float*>(vbase);
    const uint32_t xs_bytes = ((uint32_t)kRows * xs_stride * 4 + 127) & ~127u;
    float* ld_s = reinterpret_cast<float*>(vbase + xs_bytes);                  // [2][128]
    float* t_s = ld_s + NCG * kRows;                                            // [128]
    VcBars* bars = reinterpret_cast<VcBars*>(t_s + kRows);
    uint8_t* abuf = vbase + xs_bytes + NCG * kRows * 4 + kRows * 4 + 128;

    if (tid == 0) {
        mbar_init(&w_full, 1);
        fence_mbar_init();
    }
    if (vtid == 0) {
        mbar_init(&bars->a_ready, NCG * 4);
        mbar_init(&bars->acc_ready, 1);
        fence_mbar_init();
    }
    if (tid < 32) tmem_alloc(&tmem_base_s, 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_base_s + (uint32_t)vc * kVcCols;
    if (tid == 0) {                               // headers, biases and weight blocks of every layer: once per CTA
        uint32_t total = 0;
        for (int l = 0; l < L; ++l) total += kSmallBytes + A.w_bytes[l];
        mbar_arrive_expect_tx(&w_full, total);
        for (int l = 0; l < L; ++l) {
            bulk_g2s(smem + (uint32_t)l * kSmallSlot, A.packed[l], kSmallBytes, &w_full);
            bulk_g2s(smem + A.sm_w + A.w_off[l], A.packed[l] + kOffW, A.w_bytes[l], &w_full);
        }
    }
    mbar_wait(&w_full, 0);
    if (A.permuted) {                             // logical -> physical tile columns, once: the headers stay resident
        __syncthreads();
        for (int i = tid; i < L * (kK1 + kMaxTr); i += V * kVcThreads) {
            const int l = i / (kK1 + kMaxTr), k = i - l * (kK1 + kMaxTr);
            Header* h = reinterpret_cast<Header*>(smem + (uint32_t)l * kSmallSlot);
            if (k < kK1) h->cond_idx[k] = A.perm.phys[l][h->cond_idx[k]];
            else h->tr_idx[k - kK1] = A.perm.phys[l][h->tr_idx[k - kK1]];
        }
        __syncthreads();
    }

    constexpr int H = 64;
    constexpr int kb_h = H / 16;
    constexpr uint32_t a_part = (uint32_t)kRows * kK1 * 2;
    constexpr uint32_t a_lo = (uint32_t)kRows * H * 2;
    constexpr uint32_t a_sbo = (uint32_t)(H / 8) * 128;
    constexpr uint32_t w1b = (uint32_t)H * 32, w2b = (uint32_t)H * 64, w3b = kNOut * 64;
    const int dshift = ((d & (d - 1)) == 0) ? (31 - __clz(d)) : -1;
    const int n_vcta = (int)gridDim.x * V, my_vcta = (int)blockIdx.x * V + vc;
    const int my_tiles = (A.n_tiles > my_vcta) ? (A.n_tiles - 1 - my_vcta) / n_vcta + 1 : 0;

    if (warp == 0) {
        // ---- L2 prefetch of this virtual CTA's next tiles -------------------------------------------
        if (lane == 0)
            for (int it = 1; it < my_tiles; ++it) {
                const long long nrow0 = ((long long)my_vcta + (long long)it * n_vcta) * kRows;
                const long long nb = min((long long)kRows, A.rows - nrow0) * d * 4;
                const char* src = reinterpret_cast<const char*>(A.x + nrow0 * d);
                if (nb >= 16 && ((reinterpret_cast<uintptr_t>(src) & 15) == 0))
                    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(src), "r"((uint32_t)(nb & ~15LL)) : "memory");
                if (it >= 4) break;                     // a few tiles ahead is enough; the rest follows the loads
            }
    } else if (warp == 1) {
        // ---- UMMA issuer of this virtual CTA -----------------------------------------------------------
        if (lane == 0) {
            const uint32_t idesc1 = make_idesc(FMT_BF16, 128, H);
            const uint32_t idesc2 = make_idesc(FMT_F16, 128, H);
            const uint32_t idesc3 = make_idesc(FMT_F16, 128, kNOut);
            const uint32_t a0 = smem_u32(abuf);
            const uint32_t dmain = tmem, dcorr = tmem + H;
            uint32_t ause = 0;
            tc_fence_after();
            for (int it = 0; it < my_tiles; ++it)
            for (int l = 0; l < L; ++l) {
                const Header* hdr = reinterpret_cast<const Header*>(smem + (uint32_t)l * kSmallSlot);
                const int n_hidden = hdr->n_hidden;
                const int k1b = (hdr->n_cond + (hdr->time_col >= 0 ? 1 : 0) <= 16) ? 1 : 2;   // K blocks of layer 1 in use
                uint32_t roff = smem_u32(smem + A.sm_w + A.w_off[l]);
                mbar_wait(&bars->a_ready, ause & 1); ++ause;
                tc_fence_after();
                uint32_t acc_m = 0, acc_c = 0;
                for (int b = 0; b < 6; ++b, roff += w1b) {
                    const int pb = 2 - b / 2, kb = b & 1;
                    if (kb >= k1b) continue;                      // all-zero K block (<= 16 conditioning inputs)
                    const uint64_t bd = make_smem_desc(roff, 128, 256);
                    for (int pa = 2; pa >= 0; --pa) {
                        if (pa == 2 && pb == 2) continue;
                        const uint64_t ad = make_smem_desc(a0 + pa * a_part + kb * 256, 128, 512);
                        if (pa == 0 && pb == 0) { umma_f16(dmain, ad, bd, idesc1, acc_m); acc_m = 1; }
                        else { umma_f16(dcorr, ad, bd, idesc1, acc_c); acc_c = 1; }
                    }
                }
                umma_commit(&bars->acc_ready);
                for (int layer = (n_hidden == 2 ? 0 : 1); layer < 2; ++layer) {
                    mbar_wait(&bars->a_ready, ause & 1); ++ause;
                    tc_fence_after();
                    const bool last = (layer == 1);
                    const uint32_t idesc = last ? idesc3 : idesc2;
                    const uint32_t lo_off = last ? kNOut * 32 : (uint32_t)H * 32;
                    acc_m = acc_c = 0;
                    for (int kb = 0; kb < kb_h; ++kb) {
                        const uint64_t b_hi = make_smem_desc(roff, 128, 256), b_lo = make_smem_desc(roff + lo_off, 128, 256);
                        roff += last ? w3b : w2b;
                        const uint64_t a_hi = make_smem_desc(a0 + kb * 256, 128, a_sbo);
                        const uint64_t a_l = make_smem_desc(a0 + a_lo + kb * 256, 128, a_sbo);
                        umma_f16(dcorr, a_l, b_hi, idesc, acc_c); acc_c = 1;
                        umma_f16(dcorr, a_hi, b_lo, idesc, 1);
                        umma_f16(dmain, a_hi, b_hi, idesc, acc_m); acc_m = 1;
                    }
                    umma_commit(&bars->acc_ready);
                }
            }
        }
    } else if (warp < kEpiWarp0 + NCG * 4) {
        // ---- epilogue warps of this virtual CTA ------------------------------------------------------------
        const int q = warp & 3;
        const int cg = (warp - ((q >= kEpiWarp0) ? q : q + 4)) >> 2;
        const int etid = vtid - kEpiWarp0 * 32;
        const int row = q * 32 + lane;
        float* xrow = xs + row * xs_stride;
        const uint32_t lane_sel = (uint32_t)(q * 32) << 16;
        const bool want_ld = A.ldj_mode != STB_LDJ_NONE;
        const bool inverse = A.inverse != 0;
        const int bar_id = 1 + vc;
        uint32_t acc_use = 0;

        for (int it = 0; it < my_tiles; ++it) {
            const long long row0 = ((long long)my_vcta + (long long)it * n_vcta) * kRows;
            const int nrows = (int)min((long long)kRows, A.rows - row0);
            {   // ---- stage x (once per flow) ---------------------------------------------------------------
                const float* xg = A.x + row0 * d;
                const int n = nrows * d;
                if ((d & 3) == 0 && ((reinterpret_cast<uintptr_t>(xg) & 15) == 0)) {
                    const int n4 = (kRows * d) >> 2;
                    for (int i0 = etid; i0 < n4; i0 += kEpiThreads * 4) {
                        float4 v[4];
#pragma unroll
                        for (int u = 0; u < 4; ++u) {
                            const int i = i0 + u * kEpiThreads;
                            v[u] = (i < n4 && i * 4 < n) ? __ldg(reinterpret_cast<const float4*>(xg) + i)
                                                         : make_float4(0.f, 0.f, 0.f, 0.f);
                        }
#pragma unroll
                        for (int u = 0; u < 4; ++u) {
                            const int i = i0 + u * kEpiThreads;
                            if (i < n4) {
                                const int r = (dshift >= 0) ? ((i * 4) >> dshift) : (i * 4) / d, c = (i * 4) - r * d;
                                float* dst = xs + r * xs_stride + c;
                                dst[0] = v[u].x; dst[1] = v[u].y; dst[2] = v[u].z; dst[3] = v[u].w;
                            }
                        }
                    }
                } else {
                    for (int i = etid; i < kRows * d; i += kEpiThreads) {
                        const int r = (dshift >= 0) ? (i >> dshift) : i / d, c = i - r * d;
                        xs[r * xs_stride + c] = (i < n) ? __ldg(xg + i) : 0.f;
                    }
                }
                if (etid < kRows) t_s[etid] = (A.t != nullptr && etid < nrows) ? __ldg(A.t + row0 + etid) : 0.f;
            }
            named_bar_sync(bar_id, kEpiThreads);
            float ld_acc = 0.f;
#pragma unroll 1
            for (int l = 0; l < L; ++l) {
                const uint8_t* small = smem + (uint32_t)l * kSmallSlot;
                const Header* hdr = reinterpret_cast<const Header*>(small);
                const float* b1s = reinterpret_cast<const float*>(small + kOffB1);
                const float* b2s = reinterpret_cast<const float*>(small + kOffB2);
                const float* b3s = reinterpret_cast<const float*>(small + kOffB3);
                const int n_tr = hdr->n_tr, n_cond = hdr->n_cond, n_hidden = hdr->n_hidden, act = hdr->act;
                const int time_col = hdr->time_col;
                const int k1b = (n_cond + (time_col >= 0 ? 1 : 0) <= 16) ? 1 : 2;
                // ---- A1: this row's conditioning columns (+ t) as three bf16 parts ------------------------
#pragma unroll 1
                for (int kc = cg; kc < 2 * k1b; kc += NCG) {
                    const uint32_t off = (uint32_t)(row >> 3) * 512 + (uint32_t)(row & 7) * 16 + kc * 128;
                    __align__(16) __nv_bfloat16 q0[8], q1[8], q2[8];
#pragma unroll
                    for (int u = 0; u < 8; ++u) {
                        const int k = kc * 8 + u;
                        const float v = (k < n_cond) ? xrow[hdr->cond_idx[k]] : ((k == time_col) ? t_s[row] : 0.f);
                        split_bf16x3(v, q0[u], q1[u], q2[u]);
                    }
                    *reinterpret_cast<uint4*>(abuf + off) = *reinterpret_cast<const uint4*>(q0);
                    *reinterpret_cast<uint4*>(abuf + a_part + off) = *reinterpret_cast<const uint4*>(q1);
                    *reinterpret_cast<uint4*>(abuf + 2 * a_part + off) = *reinterpret_cast<const uint4*>(q2);
                }
                fence_proxy_async_smem();
                __syncwarp();
                if (lane == 0) mbar_arrive(&bars->a_ready);
                // ---- hidden layers ------------------------------------------------------------------------
                for (int layer = 0; layer < n_hidden; ++layer) {
                    mbar_wait_sleep(&bars->acc_ready, acc_use & 1, 32); ++acc_use;
                    tc_fence_after();
                    const float sc = (layer == 0) ? 1.f : hdr->s_mid;
                    const float* bias = (layer == 0) ? b1s : b2s;
                    constexpr int cols = H / NCG;
                    const uint32_t a_row = (uint32_t)(row >> 3) * a_sbo + (uint32_t)(row & 7) * 16;
#pragma unroll 1
                    for (int cb = 0; cb < cols; cb += 16) {
                        const int c0 = cg * cols + cb;
                        float vm[16], vc_[16];
                        tmem_ld16(tmem + lane_sel + c0, vm);
                        tmem_ld16(tmem + lane_sel + H + c0, vc_);
                        tmem_ld_wait();
                        __align__(16) __half hh[16], hl[16];
                        if (act == STB_ACT_TANH) {
                            const float2* b2p = reinterpret_cast<const float2*>(bias + c0);
#pragma unroll
                            for (int i = 0; i < 8; ++i)
                                tanh_split2(make_float2(vm[2 * i], vm[2 * i + 1]), make_float2(vc_[2 * i], vc_[2 * i + 1]),
                                            make_float2(sc, sc), b2p[i], reinterpret_cast<uint32_t*>(hh)[i],
                                            reinterpret_cast<uint32_t*>(hl)[i]);
                        } else {                               // STB_ACT_SIGMOID
                            const float2* b2p = reinterpret_cast<const float2*>(bias + c0);
#pragma unroll
                            for (int i = 0; i < 8; ++i)
                                sigmoid_split2(make_float2(vm[2 * i], vm[2 * i + 1]), make_float2(vc_[2 * i], vc_[2 * i + 1]),
                                               make_float2(sc, sc), b2p[i], reinterpret_cast<uint32_t*>(hh)[i],
                                               reinterpret_cast<uint32_t*>(hl)[i]);
                        }
#pragma unroll
                        for (int half8 = 0; half8 < 2; ++half8) {
                            const int kc = (c0 >> 3) + half8;
                            *reinterpret_cast<uint4*>(abuf + a_row + kc * 128) = *reinterpret_cast<const uint4*>(hh + half8 * 8);
                            *reinterpret_cast<uint4*>(abuf + a_lo + a_row + kc * 128) = *reinterpret_cast<const uint4*>(hl + half8 * 8);
                        }
                    }
                    tc_fence_before();
                    fence_proxy_async_smem();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&bars->a_ready);
                }
                // ---- output layer: affine transform of this warp's transformed dims ---------------------------
                mbar_wait_sleep(&bars->acc_ready, acc_use & 1, 32); ++acc_use;
                tc_fence_after();
                const float s_out = hdr->s_out;
                const bool cont = hdr->cont != 0;
                const float tv = t_s[row];
#pragma unroll 1
                for (int og = cg; og * 8 < n_tr; og += NCG) {
                    float lm[8], lc[8], sm_[8], sc_[8];
                    tmem_ld8(tmem + lane_sel + og * 8, lm);
                    tmem_ld8(tmem + lane_sel + H + og * 8, lc);
                    tmem_ld8(tmem + lane_sel + kMaxTr + og * 8, sm_);
                    tmem_ld8(tmem + lane_sel + H + kMaxTr + og * 8, sc_);
                    tmem_ld_wait();
#pragma unroll
                    for (int u = 0; u < 8; ++u) {
                        const int ji = og * 8 + u;
                        if (ji < n_tr) {
                            const int j = hdr->tr_idx[ji];
                            float ls = fmaf(lm[u] + lc[u], s_out, b3s[ji]);
                            float sh = fmaf(sm_[u] + sc_[u], s_out, b3s[kMaxTr + ji]);
                            if (cont) {                        // coupling.py:199-205
                                ls *= hdr->ts_ls[ji] * tv;
                                sh *= hdr->ts_sh[ji] * tv;
                            }
                            const float xv = xrow[j];
                            if (inverse) { xrow[j] = (xv - sh) * exp_fast(-ls); ld_acc -= ls; }
                            else { xrow[j] = xv * exp_fast(ls) + sh; ld_acc += ls; }
                        }
                    }
                }
                tc_fence_before();
                // the next layer gathers columns other warps have just written (and reuses the accumulators)
                named_bar_sync(bar_id, kEpiThreads);
            }   // layers

            ld_s[cg * kRows + row] = ld_acc;
            named_bar_sync(bar_id, kEpiThreads);
            if (cg == 0 && want_ld && row < nrows) {
                float tot = ld_s[row] + ld_s[kRows + row];
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
                if (A.permuted) {
                    for (int i = etid; i < n; i += kEpiThreads) {
                        const int r = (dshift >= 0) ? (i >> dshift) : i / d, c = i - r * d;
                        yg[i] = xs[r * xs_stride + A.perm.out_phys[c]];
                    }
                } else if ((d & 3) == 0 && ((reinterpret_cast<uintptr_t>(yg) & 15) == 0)) {
                    const int n4 = n >> 2;
                    for (int i = etid; i < n4; i += kEpiThreads) {
                        const int r = (dshift >= 0) ? ((i * 4) >> dshift) : (i * 4) / d, c = (i * 4) - r * d;
                        const float* src = xs + r * xs_stride + c;
                        reinterpret_cast<float4*>(yg)[i] = make_float4(src[0], src[1], src[2], src[3]);
                    }
                } else {
                    for (int i = etid; i < n; i += kEpiThreads) {
                        const int r = (dshift >= 0) ? (i >> dshift) : i / d, c = i - r * d;
                        yg[i] = xs[r * xs_stride + c];
                    }
                }
            }
            named_bar_sync(bar_id, kEpiThreads);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (tid < 32) tmem_dealloc(tmem_base_s, 512);
}

// -----------------------------------------------------------------------------------------------
// packing
// -----------------------------------------------------------------------------------------------
struct PackArgs {
    const float *W1, *b1, *W2, *b2, *W3, *b3, *time_scale;
    uint8_t* out;
    int dim, H, n_hidden, act, in_dim, cont, time_col, lat0, n_lat;
    MaskSplit m;
};

__device__ __forceinline__ int out_row_affine(const PackArgs& a, int n) {     // packed output column -> Linear row
    const int p = n / kMaxTr, ji = n % kMaxTr;
    return (ji < a.m.n_tr) ? p * a.dim + a.m.tr_idx[ji] : -1;
}

__global__ void tcm_maxabs_kernel(const PackArgs a) {
    Header* hdr = reinterpret_cast<Header*>(a.out);
    float m2 = 0.f, m3 = 0.f;
    const int gtid = blockIdx.x * blockDim.x + threadIdx.x, gsz = gridDim.x * blockDim.x;
    if (a.n_hidden == 2)
        for (int i = gtid; i < a.H * a.H; i += gsz) m2 = fmaxf(m2, fabsf(a.W2[i]));
    for (int i = gtid; i < kNOut * a.H; i += gsz) {
        const int r = out_row_affine(a, i / a.H);
        if (r >= 0) m3 = fmaxf(m3, fabsf(a.W3[(size_t)r * a.H + i % a.H]));
    }
    warp_max_to(&hdr->max_mid, m2);
    warp_max_to(&hdr->max_out, m3);
}

__global__ void tcm_pack_kernel(const PackArgs a) {
    Header* hdr = reinterpret_cast<Header*>(a.out);
    const float s_mid = pow2_scale(__uint_as_float(hdr->max_mid)), s_out = pow2_scale(__uint_as_float(hdr->max_out));
    const int gtid = blockIdx.x * blockDim.x + threadIdx.x, gsz = gridDim.x * blockDim.x;
    const int H = a.H;
    if (gtid == 0) {
        hdr->magic = kMagic; hdr->dim = a.dim; hdr->n_cond = a.m.n_cond; hdr->n_tr = a.m.n_tr; hdr->H = H;
        hdr->n_hidden = a.n_hidden; hdr->act = a.act; hdr->s_mid = s_mid; hdr->s_out = s_out;
        for (int i = 0; i < kK1; ++i) hdr->cond_idx[i] = a.m.cond_idx[i];
        for (int i = 0; i < kMaxTr; ++i) hdr->tr_idx[i] = a.m.tr_idx[i];
        hdr->cont = a.cont; hdr->time_col = a.time_col; hdr->lat0 = a.lat0; hdr->n_lat = a.n_lat;
        for (int i = 0; i < kMaxTr; ++i) {
            hdr->ts_ls[i] = (a.cont && i < a.m.n_tr) ? a.time_scale[a.m.tr_idx[i]] : 0.f;
            hdr->ts_sh[i] = (a.cont && i < a.m.n_tr) ? a.time_scale[a.dim + a.m.tr_idx[i]] : 0.f;
        }
    }
    float* b1 = reinterpret_cast<float*>(a.out + kOffB1);
    float* b2 = reinterpret_cast<float*>(a.out + kOffB2);
    float* b3 = reinterpret_cast<float*>(a.out + kOffB3);
    for (int i = gtid; i < kMaxH; i += gsz) {
        b1[i] = (i < H) ? a.b1[i] : 0.f;
        b2[i] = (i < H && a.n_hidden == 2) ? a.b2[i] : 0.f;
    }
    for (int i = gtid; i < kNOut; i += gsz) {
        const int r = out_row_affine(a, i);
        b3[i] = (r >= 0) ? a.b3[r] : 0.f;
    }
    uint8_t* w = a.out + kOffW;
    for (int i = gtid; i < H * kK1; i += gsz) {
        const int n = i / kK1, k = i % kK1;
        store_w1_blocks(w, H, n, k, first_linear_w(a.W1, n, k, a.in_dim, a.dim, a.m, a.time_col, a.lat0, a.n_lat));
    }
    w += 6 * w1_block_bytes(H);
    if (a.n_hidden == 2) {
        const float inv = 1.f / s_mid;
        for (int i = gtid; i < H * H; i += gsz) store_hilo_blocks(w, H, i / H, i % H, a.W2[i] * inv);
        w += (size_t)(H / 16) * w2_block_bytes(H);
    }
    const float inv = 1.f / s_out;
    for (int i = gtid; i < kNOut * H; i += gsz) {
        const int n = i / H, k = i % H;
        const int r = out_row_affine(a, n);
        store_hilo_blocks(w, kNOut, n, k, r >= 0 ? a.W3[(size_t)r * H + k] * inv : 0.f);
    }
}

// the mask split, then the GEMM1 slots: [conditioning columns | t (continuous-affine) | latent] within K = 32
static bool fill_pack_args(const stb_layer* L, PackArgs& a) {
    if (!split_mask(L, kK1, kMaxTr, a.m)) return false;
    const stb_mlp& N = L->net;
    a.in_dim = N.dims[0];
    a.cont = L->kind == STB_CONT_AFFINE;
    a.time_col = -1;
    if (L->time_input) {
        if (a.m.n_cond >= kK1) return false;
        a.time_col = a.m.n_cond;                                // first free A1 column
    }
    a.n_lat = L->latent_dim;
    a.lat0 = a.m.n_cond + (a.time_col >= 0 ? 1 : 0);
    if (a.lat0 + a.n_lat > kK1) return false;
    if (a.in_dim != L->dim + a.n_lat + (a.time_col >= 0 ? 1 : 0)) return false;
    a.time_scale = L->time_scale;
    a.dim = L->dim; a.H = N.dims[1]; a.n_hidden = N.n_linear - 1; a.act = N.activation;
    a.W1 = N.W[0]; a.b1 = N.b[0];
    a.W2 = a.n_hidden == 2 ? N.W[1] : nullptr; a.b2 = a.n_hidden == 2 ? N.b[1] : nullptr;
    a.W3 = N.W[N.n_linear - 1]; a.b3 = N.b[N.n_linear - 1];
    return true;
}

}  // namespace tcm

bool tcm_layer_supported(const stb_layer* L) {
    using namespace tcm;
    if (L->kind != STB_AFFINE && L->kind != STB_CONT_AFFINE) return false;
    if (!L->cond_x || L->zero_cond || L->latent_dim < 0) return false;
    if (L->kind == STB_AFFINE && L->time_input) return false;
    if (L->row_out || L->dim < 2 || L->dim > kMaxDim) return false;
    const stb_mlp& N = L->net;
    if ((N.n_linear != 2 && N.n_linear != 3) || N.final_activation != STB_ACT_NONE) return false;
    const int H = N.dims[1];
    if (H < 64 || H > kMaxH || (H % 64) != 0) return false;
    if (N.n_linear == 3 && N.dims[2] != H) return false;
    if (!tc_epilogue_ok(L)) return false;
    PackArgs a;
    return fill_pack_args(L, a);
}

uint64_t tcm_packed_bytes(const stb_layer* L) { return tcm::packed_bytes(L->net.dims[1], L->net.n_linear - 1); }

int tcm_pack_layer(const stb_layer* L, void* out, cudaStream_t stream) {
    using namespace tcm;
    PackArgs a;
    if (!fill_pack_args(L, a)) return set_error(STB_ENOTSUP, "layer has no tensor-core path");
    a.out = static_cast<uint8_t*>(out);
    return pack_image(out, kOffW, stream, "tcm_pack", [&] {
        pack_pass(tcm_maxabs_kernel, 64, 256, stream, a);
        pack_pass(tcm_pack_kernel, 296, 256, stream, a);
    });
}

int tcm_layer_apply(const stb_layer* L, int direction, const float* x, const float* latent, const float* t, float* y,
                    float* ldj, int ldj_mode, int base_log_prob, int64_t rows, cudaStream_t stream) {
    using namespace tcm;
    const int H = L->net.dims[1];
    if (L->packed_bytes < packed_bytes(H, L->net.n_linear - 1)) return set_error(STB_EINVAL, "packed image too small");
    Args A;
    A.latent = L->latent_dim > 0 ? latent : nullptr;
    A.lat_stride = L->latent_dim;
    A.packed = static_cast<const uint8_t*>(L->packed);
    A.x = x; A.t = t; A.y = y; A.ldj = ldj;
    A.ldj_mode = ldj ? ldj_mode : STB_LDJ_NONE;
    A.base_log_prob = base_log_prob;
    A.inverse = direction == STB_INVERSE;
    A.rows = rows;
    const long long tiles = (rows + kRows - 1) / kRows;
    if (tiles > 0x7fffffffLL) return set_error(STB_EINVAL, "too many rows");
    A.n_tiles = (int)tiles;
    const int n_sm = sm_count();
    // small conditioner on few dims (configs[3]): the 8-warp configuration, two CTAs per SM
    const uint32_t w_total = 6 * w1_block_bytes(H) + (L->net.n_linear == 3 ? (H / 16) * w2_block_bytes(H) : 0) + (H / 16) * w3_block_bytes();
    const bool small = (H == 64) && (L->dim <= 32) && (w_total <= kStages * kSlotBytes) && (tiles >= 2LL * n_sm);
    // wide conditioners: the pipelined kernel (TMEM-resident activations, GEMMs behind the activation waves)
    if (!small && H >= 128)
        return launch_persistent(tc_mlp_pipe_kernel, A, tiles, 1, kPipeThreads, pipe_smem_bytes(H), stream, "tc_mlp_pipe_kernel");
    const uint32_t smem = small ? Cfg<2>::smem_bytes(H) : Cfg<4>::smem_bytes(H);
    if (smem > 227 * 1024) return set_error(STB_ENOTSUP, "hidden width %d needs %u B of shared memory", H, smem);
    return small ? launch_persistent(tc_mlp_affine_kernel<2>, A, tiles, 2, Cfg<2>::kThreads, smem, stream, "tc_mlp_affine_kernel")
                 : launch_persistent(tc_mlp_affine_kernel<4>, A, tiles, 1, Cfg<4>::kThreads, smem, stream, "tc_mlp_affine_kernel");
}

namespace tcm {
// -----------------------------------------------------------------------------------------------
// CHAIN, four tiles in flight: tc_mlp_chain4_kernel
// -----------------------------------------------------------------------------------------------
// Same job as tc_mlp_chain_kernel for the shapes of BASELINE.json configs[3] (one hidden layer of 64 units, <= 16
// conditioner inputs incl. t, <= 16 transformed dims, dim <= 32), restructured around what the phase clocks of that
// kernel showed (profiles/r02_tcm_chain_phase_clocks.txt): a tile-layer is a chain of five dependent phases, so what
// matters is how many INDEPENDENT tiles an SM holds, and shared memory (a 32 KB fp16 hi|lo A operand per tile)
// capped that at two.  Here the hidden activations never touch shared memory: each thread (= row = TMEM lane)
// writes its row of h straight into TMEM with tcgen05.st -- into the accumulator columns it has just consumed --
// and GEMM2 reads its A operand from TMEM (tcgen05.mma, TMEM-sourced A).  A virtual CTA shrinks to ~21 KB and 128
// TMEM columns, FOUR of them share the resident weights, and because a thread owns its whole row (gather, activation,
// affine update) there is no cross-warp hazard between layers: no block barrier, no st.shared + proxy fence for h.
//   TMEM columns of one virtual CTA:  GEMM1 main [0,64) | corr [64,128)
//                                     h(kb): hi [16 kb, 16 kb + 8), lo [16 kb + 8, 16 kb + 16)   (over consumed main)
//                                     GEMM2 (N = 16 twice): ls main [64,80) sh main [80,96) ls corr [96,112) sh corr [112,128)
constexpr int kV4 = 4;
constexpr int kV4EpiWarps = 4;                        // per virtual CTA: thread = row
constexpr int kV4Threads = kV4 * (kV4EpiWarps + 1) * 32;        // 16 epilogue warps, then one issuer warp per virtual CTA
constexpr uint32_t kV4A1Part = kRows * 16 * 2;        // one bf16 part of the [128 x 16] first-layer operand
constexpr uint32_t kV4W1Bytes = 3 * 64 * 32;          // three bf16 parts of [64 x 16]
constexpr uint32_t kV4W3Bytes = 4 * kNOut * 64;       // four K blocks of [64 x 16] fp16 hi | lo
constexpr uint32_t kV4WBytes = kV4W1Bytes + kV4W3Bytes;
constexpr uint32_t kV4W3Used = 4 * 2 * 32 * 32;       // the rows in use, compacted: four K blocks of [32 x 16] hi | lo

template <int DUMMY>
__global__ void __launch_bounds__(kV4Threads, 1) tc_mlp_chain4_kernel(const ChainArgs A) {
    extern __shared__ __align__(1024) uint8_t smem[];
    __shared__ uint64_t w_full;
    __shared__ uint32_t tmem_base_s;
    constexpr int H = 64;

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const bool is_epi = warp < kV4 * kV4EpiWarps;
    const int vc = is_epi ? warp >> 2 : warp - kV4 * kV4EpiWarps;
    const int d = A.dim, L = A.n_layers, xs_stride = A.xs_stride;

    uint8_t* vbase = smem + A.sm_vc + (uint32_t)vc * A.vc_bytes;
    float* xs = reinterpret_cast<float*>(vbase);
    const uint32_t xs_bytes = ((uint32_t)kRows * xs_stride * 4 + 127) & ~127u;
    uint8_t* a1buf = vbase + xs_bytes;                                     // 3 x 4 KB
    VcBars* bars = reinterpret_cast<VcBars*>(a1buf + 3 * kV4A1Part);

    if (tid == 0) {
        mbar_init(&w_full, 1);
        for (int v = 0; v < kV4; ++v) {
            VcBars* b = reinterpret_cast<VcBars*>(smem + A.sm_vc + (uint32_t)v * A.vc_bytes + xs_bytes + 3 * kV4A1Part);
            mbar_init(&b->a_ready, kV4EpiWarps);
            mbar_init(&b->acc_ready, 1);
        }
        fence_mbar_init();
    }
    if (warp == 0) tmem_alloc(&tmem_base_s, 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_base_s + (uint32_t)vc * kVcCols;
    if (tid == 0) {                               // headers, biases and the weight blocks in use, once per CTA
        mbar_arrive_expect_tx(&w_full, (uint32_t)L * (kSmallBytes + kV4W1Bytes + kV4W3Used));
        for (int l = 0; l < L; ++l) {
            bulk_g2s(smem + (uint32_t)l * kSmallSlot, A.packed[l], kSmallBytes, &w_full);
            uint8_t* wdst = smem + A.sm_w + (uint32_t)l * kV4WBytes;
            // first Linear: K block 0 of the parts pb = 2, 1, 0 (blocks 0, 2, 4 of the image; blocks 1, 3, 5 are zero)
            for (int b = 0; b < 3; ++b) bulk_g2s(wdst + b * 2048, A.packed[l] + kOffW + (uint32_t)(2 * b) * 2048, 2048, &w_full);
            // last Linear: of every K block [64 x 16] hi | lo only the log-scale rows 0..15 and the shift rows 32..47 are in
            // use (<= 16 transformed dims); they are gathered into ONE [32 x 16] operand per part, so that the output GEMM
            // is one N = 32 UMMA per pass instead of two N = 16 ones (a UMMA costs a fixed ~38 clocks whatever N)
            for (int kb = 0; kb < 4; ++kb)
                for (int part = 0; part < 2; ++part)
                    for (int half = 0; half < 2; ++half)
                        bulk_g2s(wdst + kV4W1Bytes + kb * 2048 + part * 1024 + half * 512,
                                 A.packed[l] + kOffW + 6 * 2048 + kb * (kNOut * 64) + part * (kNOut * 32) + half * 1024, 512, &w_full);
        }
    }
    mbar_wait(&w_full, 0);
    if (A.permuted) {
        __syncthreads();
        for (int i = tid; i < L * (kK1 + kMaxTr); i += kV4Threads) {
            const int l = i / (kK1 + kMaxTr), k = i - l * (kK1 + kMaxTr);
            Header* h = reinterpret_cast<Header*>(smem + (uint32_t)l * kSmallSlot);
            if (k < kK1) h->cond_idx[k] = A.perm.phys[l][h->cond_idx[k]];
            else h->tr_idx[k - kK1] = A.perm.phys[l][h->tr_idx[k - kK1]];
        }
        __syncthreads();
    }

    const int dshift = ((d & (d - 1)) == 0) ? (31 - __clz(d)) : -1;
    const int n_vcta = (int)gridDim.x * kV4, my_vcta = (int)blockIdx.x * kV4 + vc;
    const int my_tiles = (A.n_tiles > my_vcta) ? (A.n_tiles - 1 - my_vcta) / n_vcta + 1 : 0;

    if (!is_epi) {
        // ---- UMMA issuer of this virtual CTA ---------------------------------------------------------------
        if (lane == 0) {
            const uint32_t idesc1 = make_idesc(FMT_BF16, 128, H);
            const uint32_t idesc3 = make_idesc(FMT_F16, 128, 32);
            const uint32_t a0 = smem_u32(a1buf);
            uint32_t ause = 0;
            for (int it = 0; it < my_tiles; ++it)
            for (int l = 0; l < L; ++l) {
                const uint32_t w1 = smem_u32(smem + A.sm_w + (uint32_t)l * kV4WBytes), w3 = w1 + kV4W1Bytes;
                mbar_wait_sleep(&bars->a_ready, ause & 1, 96); ++ause;
                tc_fence_after();
                uint32_t acc_m = 0, acc_c = 0;
                for (int b = 0; b < 3; ++b) {                      // bf16 parts pb = 2, 1, 0 of the first Linear
                    const int pb = 2 - b;
                    const uint64_t bd = make_smem_desc(w1 + (uint32_t)b * 2048, 128, 256);
                    for (int pa = 2; pa >= 0; --pa) {
                        if (pa == 2 && pb == 2) continue;
                        const uint64_t ad = make_smem_desc(a0 + pa * kV4A1Part, 128, 256);
                        if (pa == 0 && pb == 0) { umma_f16(tmem, ad, bd, idesc1, acc_m); acc_m = 1; }
                        else { umma_f16(tmem + H, ad, bd, idesc1, acc_c); acc_c = 1; }
                    }
                }
                umma_commit(&bars->acc_ready);
                mbar_wait_sleep(&bars->a_ready, ause & 1, 96); ++ause;
                tc_fence_after();
                // last Linear: A = h from TMEM, B = the compacted [log-scale 16 | shift 16] rows of every K block, N = 32
                {
                    const uint32_t dm = tmem + H, dc = dm + 32;
                    acc_m = acc_c = 0;
                    for (int kb = 0; kb < 4; ++kb) {
                        const uint32_t bb = w3 + (uint32_t)kb * 2048;
                        const uint64_t b_hi = make_smem_desc(bb, 128, 256), b_lo = make_smem_desc(bb + 1024, 128, 256);
                        const uint32_t a_hi = tmem + (uint32_t)kb * 16, a_lo = a_hi + 8;
                        umma_f16_ts(dc, a_lo, b_hi, idesc3, acc_c); acc_c = 1;
                        umma_f16_ts(dc, a_hi, b_lo, idesc3, 1);
                        umma_f16_ts(dm, a_hi, b_hi, idesc3, acc_m); acc_m = 1;
                    }
                }
                umma_commit(&bars->acc_ready);
            }
        }
    } else {
        // ---- epilogue: thread = row of this virtual CTA's tile ---------------------------------------------------
        const int q = warp & 3;
        const int row = q * 32 + lane;
        float* xrow = xs + row * xs_stride;
        float* xw = xs + q * 32 * xs_stride;                            // this warp's 32 rows (warp-private)
        const uint32_t lane_sel = (uint32_t)(q * 32) << 16;
        const bool want_ld = A.ldj_mode != STB_LDJ_NONE;
        const bool inverse = A.inverse != 0;
        const uint32_t a1_off = (uint32_t)(row >> 3) * 256 + (uint32_t)(row & 7) * 16;
        uint32_t acc_use = 0;

        for (int it = 0; it < my_tiles; ++it) {
            const long long row0 = ((long long)my_vcta + (long long)it * n_vcta) * kRows;
            const int nrows = (int)min((long long)kRows, A.rows - row0);
            const int wrows = max(0, min(32, nrows - q * 32));               // valid rows of this warp
            {   // ---- stage this warp's rows (coalesced), once per flow ------------------------------------------
                const float* xg = A.x + (row0 + q * 32) * d;
                const int n = wrows * d;
                if (dshift >= 2 && ((reinterpret_cast<uintptr_t>(xg) & 15) == 0)) {      // d a power of two >= 4: 16-byte loads
                    for (int i4 = lane; i4 < 8 * d; i4 += 32) {
                        const float4 v = (i4 * 4 < n) ? __ldg(reinterpret_cast<const float4*>(xg) + i4) : make_float4(0.f, 0.f, 0.f, 0.f);
                        const int r = (i4 * 4) >> dshift, c = (i4 * 4) & (d - 1);
                        float* dst = xw + r * xs_stride + c;
                        dst[0] = v.x; dst[1] = v.y; dst[2] = v.z; dst[3] = v.w;
                    }
                } else {
                    for (int i = lane; i < 32 * d; i += 32) {
                        const int r = i / d, c = i - r * d;
                        xw[r * xs_stride + c] = (i < n) ? __ldg(xg + i) : 0.f;
                    }
                }
                if (it + 1 < my_tiles && lane == 0) {                    // next tile of this virtual CTA -> L2
                    const long long nrow0 = ((long long)my_vcta + (long long)(it + 1) * n_vcta) * kRows + q * 32;
                    const long long nb = min(32LL, A.rows - nrow0) * d * 4;
                    const char* src = reinterpret_cast<const char*>(A.x + nrow0 * d);
                    if (nb >= 16 && ((reinterpret_cast<uintptr_t>(src) & 15) == 0))
                        asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(src), "r"((uint32_t)(nb & ~15LL)) : "memory");
                }
            }
            const float tv = (A.t != nullptr && row < nrows) ? __ldg(A.t + row0 + row) : 0.f;
            __syncwarp();
            float ld_acc = 0.f;
#pragma unroll 1
            for (int l = 0; l < L; ++l) {
                const uint8_t* small = smem + (uint32_t)l * kSmallSlot;
                const Header* hdr = reinterpret_cast<const Header*>(small);
                const float* b1s = reinterpret_cast<const float*>(small + kOffB1);
                const float* b3s = reinterpret_cast<const float*>(small + kOffB3);
                const int n_tr = hdr->n_tr, n_cond = hdr->n_cond, act = hdr->act, time_col = hdr->time_col;
                // ---- A1: the row's <= 16 conditioner inputs as three bf16 parts --------------------------------
#pragma unroll
                for (int kc = 0; kc < 2; ++kc) {
                    __align__(16) __nv_bfloat16 q0[8], q1[8], q2[8];
#pragma unroll
                    for (int u = 0; u < 8; ++u) {
                        const int k = kc * 8 + u;
                        const float v = (k < n_cond) ? xrow[hdr->cond_idx[k]] : ((k == time_col) ? tv : 0.f);
                        split_bf16x3(v, q0[u], q1[u], q2[u]);
                    }
                    *reinterpret_cast<uint4*>(a1buf + a1_off + kc * 128) = *reinterpret_cast<const uint4*>(q0);
                    *reinterpret_cast<uint4*>(a1buf + kV4A1Part + a1_off + kc * 128) = *reinterpret_cast<const uint4*>(q1);
                    *reinterpret_cast<uint4*>(a1buf + 2 * kV4A1Part + a1_off + kc * 128) = *reinterpret_cast<const uint4*>(q2);
                }
                tc_fence_before();
                fence_proxy_async_smem();
                __syncwarp();
                if (lane == 0) mbar_arrive(&bars->a_ready);
                // ---- hidden layer: accumulators -> h, written back into the TMEM columns just consumed ----------
                mbar_wait_sleep(&bars->acc_ready, acc_use & 1, 64); ++acc_use;
                tc_fence_after();
#pragma unroll 1
                for (int kb = 0; kb < 4; ++kb) {
                    float vm[16], vc_[16];
                    tmem_ld16(tmem + lane_sel + (uint32_t)kb * 16, vm);
                    tmem_ld16(tmem + lane_sel + H + (uint32_t)kb * 16, vc_);
                    tmem_ld_wait();
                    uint32_t hh[8], hl[8];
                    const float2* b2p = reinterpret_cast<const float2*>(b1s + kb * 16);
                    if (act == STB_ACT_TANH) {
#pragma unroll
                        for (int i = 0; i < 8; ++i)
                            tanh_split2(make_float2(vm[2 * i], vm[2 * i + 1]), make_float2(vc_[2 * i], vc_[2 * i + 1]),
                                        make_float2(1.f, 1.f), b2p[i], hh[i], hl[i]);
                    } else {
#pragma unroll
                        for (int i = 0; i < 8; ++i)
                            sigmoid_split2(make_float2(vm[2 * i], vm[2 * i + 1]), make_float2(vc_[2 * i], vc_[2 * i + 1]),
                                           make_float2(1.f, 1.f), b2p[i], hh[i], hl[i]);
                    }
                    tmem_st8(tmem + lane_sel + (uint32_t)kb * 16, hh);
                    tmem_st8(tmem + lane_sel + (uint32_t)kb * 16 + 8, hl);
                }
                tmem_st_wait();
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&bars->a_ready);
                // ---- output layer: affine transform of the row's transformed dims ------------------------------------
                mbar_wait_sleep(&bars->acc_ready, acc_use & 1, 64); ++acc_use;
                tc_fence_after();
                const float s_out = hdr->s_out;
                const bool cont = hdr->cont != 0;
#pragma unroll 1
                for (int og = 0; og * 8 < n_tr; ++og) {
                    float lm[8], lc[8], sm_[8], sc_[8];
                    tmem_ld8(tmem + lane_sel + H + og * 8, lm);
                    tmem_ld8(tmem + lane_sel + H + 32 + og * 8, lc);
                    tmem_ld8(tmem + lane_sel + H + 16 + og * 8, sm_);
                    tmem_ld8(tmem + lane_sel + H + 48 + og * 8, sc_);
                    tmem_ld_wait();
#pragma unroll
                    for (int u = 0; u < 8; ++u) {
                        const int ji = og * 8 + u;
                        if (ji < n_tr) {
                            const int j = hdr->tr_idx[ji];
                            float ls = fmaf(lm[u] + lc[u], s_out, b3s[ji]);
                            float sh = fmaf(sm_[u] + sc_[u], s_out, b3s[kMaxTr + ji]);
                            if (cont) {                        // coupling.py:199-205
                                ls *= hdr->ts_ls[ji] * tv;
                                sh *= hdr->ts_sh[ji] * tv;
                            }
                            const float xv = xrow[j];
                            if (inverse) { xrow[j] = (xv - sh) * exp_fast(-ls); ld_acc -= ls; }
                            else { xrow[j] = xv * exp_fast(ls) + sh; ld_acc += ls; }
                        }
                    }
                }
                tc_fence_before();
            }   // layers

            if (want_ld && row < nrows) {
                float tot = ld_acc;
                if (A.base_log_prob) {
                    float b = 0.f;
                    for (int c = 0; c < d; ++c) { const float v = xrow[c]; b += -0.5f * v * v - 0.91893853320467274178f; }
                    tot += b;
                }
                float* dst = A.ldj + row0 + row;
                *dst = (A.ldj_mode == STB_LDJ_ADD) ? (*dst + tot) : tot;
            }
            __syncwarp();
            if (A.y != nullptr) {                                        // this warp's rows out (coalesced)
                float* yg = A.y + (row0 + q * 32) * d;
                const int n = wrows * d;
                if (dshift >= 2 && !A.permuted && ((reinterpret_cast<uintptr_t>(yg) & 15) == 0)) {
                    for (int i4 = lane; i4 * 4 < n; i4 += 32) {
                        const int r = (i4 * 4) >> dshift, c = (i4 * 4) & (d - 1);
                        const float* src = xw + r * xs_stride + c;
                        reinterpret_cast<float4*>(yg)[i4] = make_float4(src[0], src[1], src[2], src[3]);
                    }
                } else {
                    for (int i = lane; i < n; i += 32) {
                        const int r = i / d, c = i - r * d;
                        yg[i] = xw[r * xs_stride + (A.permuted ? (int)A.perm.out_phys[c] : c)];
                    }
                }
            }
            __syncwarp();
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem_base_s, 512);
}

}  // namespace tcm

// ---- a run of affine / continuous-affine couplings of one flow in ONE launch ---------------------------------
namespace tcm {
static uint32_t layer_w_total(const stb_layer* L) {
    const int H = L->net.dims[1];
    return 6 * w1_block_bytes(H) + (L->net.n_linear == 3 ? (H / 16) * w2_block_bytes(H) : 0) + (H / 16) * w3_block_bytes();
}
constexpr int kChainV = 2;
static bool chain_layout(const stb_layer* const* layers, int n, ChainArgs* A, uint32_t* smem_bytes) {
    if (n < 2 || n > kMaxChainM) return false;
    const int d = layers[0]->dim;
    uint32_t w = 0;
    for (int i = 0; i < n; ++i) {
        const stb_layer* L = layers[i];
        if (!L->packed || !tcm_layer_supported(L) || L->dim != d || d > 32 || L->net.dims[1] != 64) return false;
        if (L->latent_dim != 0) return false;                      // `latent=` layers: one launch per layer
        if (L->packed_bytes < packed_bytes(64, L->net.n_linear - 1)) return false;
        if (A) { A->w_off[i] = w; A->w_bytes[i] = layer_w_total(L); A->packed[i] = static_cast<const uint8_t*>(L->packed); }
        w += layer_w_total(L);
    }
    const int xs_stride = d | 1;                                     // odd: column reads by row-threads stay conflict-free
    const uint32_t xs_bytes = ((uint32_t)kRows * xs_stride * 4 + 127) & ~127u;
    const uint32_t vc_bytes = (xs_bytes + kChainNCG * kRows * 4 + kRows * 4 + 128 + (uint32_t)kRows * 64 * 4 + 127) & ~127u;
    const uint32_t sm_w = ((uint32_t)n * kSmallSlot + 127) & ~127u;
    const uint32_t sm_vc = (sm_w + w + 127) & ~127u;
    const uint32_t total = sm_vc + kChainV * vc_bytes;
    if (total > 227 * 1024 - 1024) return false;                     // 1 KB: the kernel's static shared memory
    if (A) { A->n_layers = n; A->dim = d; A->xs_stride = xs_stride; A->sm_w = sm_w; A->sm_vc = sm_vc; A->vc_bytes = vc_bytes; }
    if (smem_bytes) *smem_bytes = total;
    return true;
}
}  // namespace tcm

namespace tcm {
// four-tiles-in-flight variant: one hidden layer, <= 16 conditioner inputs (incl. t) and <= 16 transformed dims per layer
static bool chain4_layout(const stb_layer* const* layers, int n, ChainArgs* A, uint32_t* smem_bytes) {
    if (n < 2 || n > kMaxChainM) return false;
    const int d = layers[0]->dim;
    for (int i = 0; i < n; ++i) {
        const stb_layer* L = layers[i];
        if (!L->packed || !tcm_layer_supported(L) || L->dim != d || d > 32 || L->net.dims[1] != 64) return false;
        if (L->latent_dim != 0) return false;                      // `latent=` layers: one launch per layer
        if (L->net.n_linear != 2 || L->packed_bytes < packed_bytes(64, 1)) return false;
        PackArgs pa;
        if (!fill_pack_args(L, pa)) return false;
        if (pa.m.n_cond + (pa.time_col >= 0 ? 1 : 0) > 16 || pa.m.n_tr > 16) return false;
        if (A) A->packed[i] = static_cast<const uint8_t*>(L->packed);
    }
    const int xs_stride = d | 1;
    const uint32_t xs_bytes = ((uint32_t)kRows * xs_stride * 4 + 127) & ~127u;
    const uint32_t vc_bytes = (xs_bytes + 3 * kV4A1Part + 128 + 127) & ~127u;
    const uint32_t sm_w = ((uint32_t)n * kSmallSlot + 127) & ~127u;
    const uint32_t sm_vc = (sm_w + (uint32_t)n * kV4WBytes + 127) & ~127u;
    const uint32_t total = sm_vc + kV4 * vc_bytes;
    if (total > 227 * 1024 - 1024) return false;
    if (A) { A->n_layers = n; A->dim = d; A->xs_stride = xs_stride; A->sm_w = sm_w; A->sm_vc = sm_vc; A->vc_bytes = vc_bytes; }
    if (smem_bytes) *smem_bytes = total;
    return true;
}
}  // namespace tcm

bool tcm_chain_supported(const stb_layer* const* layers, int n) {
    return tcm::chain4_layout(layers, n, nullptr, nullptr) || tcm::chain_layout(layers, n, nullptr, nullptr);
}

// layers[] in APPLICATION order (the caller reverses them for the inverse direction)
int tcm_chain_apply(const stb_layer* const* layers, int n, int direction, const float* x, const float* t, float* y,
                    float* ldj, int ldj_mode, int base_log_prob, int64_t rows, cudaStream_t stream,
                    const ChainPerm* perm) {
    using namespace tcm;
    ChainArgs A = {};
    uint32_t smem = 0;
    const bool four = chain4_layout(layers, n, &A, &smem);
    if (!four && !chain_layout(layers, n, &A, &smem)) return set_error(STB_EINVAL, "layers cannot be chained");
    if (perm) { A.permuted = 1; A.perm = *perm; }
    for (int i = 0; i < n; ++i)
        if (layers[i]->kind == STB_CONT_AFFINE && !t) return set_error(STB_EINVAL, "layer expects a time input");
    A.x = x; A.t = t; A.y = y; A.ldj = ldj;
    A.ldj_mode = ldj ? ldj_mode : STB_LDJ_NONE;
    A.base_log_prob = base_log_prob;
    A.inverse = direction == STB_INVERSE;
    A.rows = rows;
    const long long tiles = (rows + kRows - 1) / kRows;
    if (tiles > 0x7fffffffLL) return set_error(STB_EINVAL, "too many rows");
    A.n_tiles = (int)tiles;
    void (*kern)(ChainArgs) = four ? tc_mlp_chain4_kernel<0> : tc_mlp_chain_kernel<kChainV>;
    const int vper = four ? kV4 : kChainV;
    return launch_persistent(kern, A, (tiles + vper - 1) / vper, 1, four ? kV4Threads : kChainV * kVcThreads, smem, stream,
                             "tc_mlp_chain_kernel");
}

}  // namespace stb
