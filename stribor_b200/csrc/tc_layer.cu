// Tensor-core fused coupling layer for sm_100a (tcgen05 + TMEM + bulk-async copies).
//
// Scope of this file: st.Coupling(st.Spline(dim <= 64, 2 <= n_bins <= 16, 'quadratic' | 'cubic',
// latent_net = MLP(dim (+ latent), [64], dim * P)), mask), conditioning + latent columns <= 32 -- the BASELINE.json
// headline configuration (8 of these layers, d = 64, 16 bins) and its neighbours.  Three kernels: the per-layer kernel
// and its whole-flow (CHAIN) form described below (16 bins), and tc_spline_pair_kernel (two 128-row CTAs per SM, both A
// operands in TMEM: small batches, and every layer with fewer than 16 bins).
//
// One persistent CTA per SM, 19 warps (two issuers since round 1), tiles of 256 rows handled as two 128-row subtiles:
//   warp 0      producer: streams the packed last-Linear weights (24 KB chunks = 2 transformed
//               dims x 48 padded parameters x 64, fp16 hi | lo) L2 -> smem with cp.async.bulk
//               through a 3-stage mbarrier ring
//   warp 1      UMMA issuer (one lane): GEMM1  [128 x 32] x [32 x 64]  with both operands split
//               into three bf16 parts (exact 24-bit split, fp32 range) and the 8 leading partial
//               products; GEMM2 [128 x 64] x [64 x 96] per chunk as 3 fp16 passes
//               (hi*hi + lo*hi + hi*lo: fp32-grade products at fp16 tensor rate); accumulators
//               live in TMEM: 2 x 64 columns for GEMM1, 2 subtiles x 2 buffers x 96 for GEMM2
//               (this warp also allocates / frees the 512 TMEM columns)
//   warps 2-17  epilogue, four per scheduler: warps (s, q, g) own rows 32q..32q+31 of subtile s ==
//               TMEM lanes of sub-partition q (= warp id % 4); the two warps g = 0, 1 of a (s, q)
//               pair take one of the chunk's two dims each (and half of the row-level work: mask
//               gather + split for GEMM1's A operand, tanh of GEMM1's accumulator).  A thread is
//               one row: it pulls its dim's 48 parameters out of TMEM with tcgen05.ld (32 for the
//               softmaxes first, the derivative columns only after the bin is known, to stay under
//               112 registers) and evaluates the spline in registers, accumulating log|det J|.
// Per layer each row makes one HBM round trip (read y, write x, read/write ldj).
//
// Reference semantics restated here: flows/coupling.py:53-95, flows/spline.py:76-105,
// util/rational_quadratic_spline.py, util/cubic_spline.py, net/mlp.py:46-58, flow.py:42-47.
#include "common.cuh"
#include "stb_math.cuh"
#include "tc_common.cuh"
#include "tc_pack.cuh"
#include "tc_spline16.cuh"

namespace stb {
using namespace tc;

namespace tcl {
using namespace sp16;

constexpr int kHid = 64;             // hidden width
constexpr int kK1 = 32;              // padded number of conditioning columns (GEMM1 K)
constexpr int kPPad = 48;            // parameters per dim, padded (47 rqs / 34 cubic)
constexpr int kG = 2;                // transformed dims per weight chunk
constexpr int kChunkN = kG * kPPad;  // 96 = UMMA N of GEMM2
constexpr int kMaxDim = 64;
constexpr int kMaxTr = 32;
constexpr int kMaxChunks = kMaxTr / kG;
constexpr int kTileRows = 256;
constexpr int kXsStride = kMaxDim + 1;
constexpr int kStages = 3;
constexpr int kMaxChain = 8;           // layers of a flow fused into one launch (CHAIN kernels)
constexpr int kEpiPerSub = 2;          // epilogue warps per (subtile, TMEM sub-partition)
constexpr int kEpiWarps = 2 * 4 * kEpiPerSub;
constexpr int kEpiWarp0 = 3;           // warp 0 producer, warps 1 / 2 UMMA issuers of subtile 0 / 1
constexpr int kThreads = (kEpiWarp0 + kEpiWarps) * 32;
constexpr int kEpiThreads = kEpiWarps * 32;

// packed image (global memory, built by tc_pack_layer)
constexpr uint32_t kMagic = 0x53544232u;
struct Header {                      // 1024 bytes
    uint32_t magic;
    int32_t kind, dim, n_cond, n_tr, n_chunks, P, act;
    float s2;                        // power-of-two scale of the packed last-Linear weights
    uint32_t maxbits;                // scratch: max |W2| as uint bits
    int32_t cond_idx[kK1];
    int32_t tr_idx[kMaxTr];
    uint32_t noshift_mask;           // bit ji: softmax logits of transformed dim ji are provably within
                                     // +-100 (log2 units), so exp2 needs no max subtraction
    int32_t n_lat;                   // `latent=` columns of the conditioner input (coupling.py:64-65): GEMM1 columns
                                     // n_cond .. n_cond + n_lat - 1 are latent[row, 0 .. n_lat - 1]
    int32_t n_bins;                  // 2 .. 16 real bins; the packed layout always has 16 (padded bins: weight 0, bias -inf)
    int32_t pad[256 - 13 - kK1 - kMaxTr];
};
static_assert(sizeof(Header) == 1024, "header layout");
constexpr uint32_t kOffB1 = 1024;                                  // float[64]
constexpr uint32_t kOffB2 = kOffB1 + kHid * 4;                     // float[kMaxChunks * 96]
constexpr uint32_t kSmallBytes = kOffB2 + kMaxChunks * kChunkN * 4;    // 7424
constexpr uint32_t kOffW1 = 8192;                                  // 3 bf16 parts of [64][32], 4 KB each
constexpr uint32_t kW1Part = kHid * kK1 * 2;                       // 4096
constexpr uint32_t kW1Bytes = 3 * kW1Part;                         // 12288
constexpr uint32_t kA1Part = 128 * kK1 * 2;                        // 8192: one bf16 part of a subtile's A1
constexpr uint32_t kOffW2 = kOffW1 + kW1Bytes;                     // chunks of 24576 B
constexpr uint32_t kChunkBytes = 2 * kChunkN * kHid * 2;           // fp16 hi (12 KB) | lo (12 KB)
constexpr uint32_t kPackedBytes = kOffW2 + kMaxChunks * kChunkBytes;
constexpr uint32_t kHeadBytes = kOffW1 + kW1Bytes;                 // header | biases | first Linear: one ring item (CHAIN)
static_assert(kHeadBytes <= kChunkBytes, "the layer head fits a ring stage");

// shared memory map
constexpr uint32_t kSmXs = 0;                                      // float [256][65]
constexpr uint32_t kSmA = kSmXs + kTileRows * kXsStride * 4;       // 2 x 32 KB (A1 tf32 / h fp16, hi | lo)
constexpr uint32_t kABytes = 32768;
constexpr uint32_t kSmW1 = kSmA + 2 * kABytes;
constexpr uint32_t kSmB = kSmW1 + kW1Bytes;
constexpr uint32_t kSmSmall = kSmB + kStages * kChunkBytes;
constexpr uint32_t kSmBar = (kSmSmall + kSmallBytes + 15) & ~15u;
constexpr uint32_t kSmLd = kSmBar + 256;                           // float [2][256]: the other warps' log-det partials
constexpr uint32_t kSmemBytes = kSmLd + (kEpiPerSub - 1) * kTileRows * 4;
static_assert(kSmemBytes <= 227 * 1024, "shared memory budget");
static_assert(kSmA % 16 == 0 && kSmW1 % 16 == 0 && kSmB % 16 == 0 && kSmSmall % 16 == 0, "alignment");

struct Bars {
    uint64_t acc_full[2][2], acc_empty[2][2];
    uint64_t setup;
    uint64_t b_full[kStages], b_empty[kStages];
    uint64_t a1_ready[2], acc1_full[2], h_ready[2];
};
static_assert(sizeof(Bars) <= 256, "barrier block");

// TMEM columns
constexpr uint32_t kColAcc1 = 0;                 // + s * 64
constexpr uint32_t kColAcc2 = 128;               // + (s * 2 + buf) * 96
constexpr uint32_t kTmemCols = 512;

struct Args {
    const uint8_t* packed;
    const float* x;
    float* y;
    float* ldj;
    int ldj_mode;
    int base_log_prob;
    int inverse;
    float lower, upper;
    long long rows;
    int n_tiles;
    // CHAIN: several layers of one flow applied to a tile while it stays in shared memory
    int n_layers, dim;
    const uint8_t* chain_packed[kMaxChain];
    float lower_l[kMaxChain], upper_l[kMaxChain];
    int n_chunks_l[kMaxChain];
    const float* latent;               // [rows, lat_stride] or NULL
    int lat_stride;
    int32_t* bins;                     // BINS kernels: [rows, dim] searched bin per element (stb_layer_apply_bins)
    int permuted;                      // CHAIN: permutations between the layers, folded into the index lists
    ChainPerm perm;
};

// -----------------------------------------------------------------------------------------------
// the kernel
// -----------------------------------------------------------------------------------------------
// CHAIN = true: `n_layers` coupling layers of one flow (same dim and kind, same direction) are applied to a
// tile while it stays in shared memory -- the reference's layer loop (flow.py:104-107,118-125) inside the
// kernel: x is read and written once per flow instead of once per layer, the running log|det J| stays in a
// register.  Each layer's header + biases + first Linear (20 KB) travel through the weight ring as one more
// item ahead of its chunks; the epilogue warps copy the 7 KB small block out of the stage.
// BINS = true (parity instrument, never on the timed path): every element's searched bin goes to A.bins.
template <int KIND, bool INVERSE, bool CHAIN, bool BINS = false>
__global__ void __launch_bounds__(kThreads, 1) tc_spline_layer_kernel(const Args A) {
    extern __shared__ __align__(1024) uint8_t smem[];
    float* xs = reinterpret_cast<float*>(smem + kSmXs);
    uint8_t* abuf = smem + kSmA;
    uint8_t* w1s = smem + kSmW1;
    uint8_t* bst = smem + kSmB;
    const Header* hdr = reinterpret_cast<const Header*>(smem + kSmSmall);
    const float* b1s = reinterpret_cast<const float*>(smem + kSmSmall + kOffB1);
    const float* b2s = reinterpret_cast<const float*>(smem + kSmSmall + kOffB2);
    Bars* bars = reinterpret_cast<Bars*>(smem + kSmBar);
    float* ld_s = reinterpret_cast<float*>(smem + kSmLd);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

    // ---- one-time setup ------------------------------------------------------------------------
    if (tid == 0) {
        mbar_init(&bars->setup, 1);
        for (int i = 0; i < kStages; ++i) { mbar_init(&bars->b_full[i], 1); mbar_init(&bars->b_empty[i], 2); }
        for (int s = 0; s < 2; ++s) {
            mbar_init(&bars->a1_ready[s], kEpiWarps);          // every epilogue warp works on both subtiles' heads
            mbar_init(&bars->acc1_full[s], 1);
            mbar_init(&bars->h_ready[s], kEpiWarps);
            for (int b = 0; b < 2; ++b) { mbar_init(&bars->acc_full[s][b], 1); mbar_init(&bars->acc_empty[s][b], 8); }
        }
        fence_mbar_init();
    }
    __shared__ uint32_t tmem_base_s;      // own word: the allocator writes it, keep it away from the mbarrier block
    if (warp == 1) tmem_alloc(&tmem_base_s, kTmemCols);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_base_s;

    if (!CHAIN) {
        if (tid == 0) {                           // header + biases + packed first Linear
            mbar_arrive_expect_tx(&bars->setup, kSmallBytes + kW1Bytes);
            bulk_g2s(smem + kSmSmall, A.packed, kSmallBytes, &bars->setup);
            bulk_g2s(w1s, A.packed + kOffW1, kW1Bytes, &bars->setup);
        }
        mbar_wait(&bars->setup, 0);
    }

    const int n_layers = CHAIN ? A.n_layers : 1;
    const int d = CHAIN ? A.dim : hdr->dim;
    // per-layer quantities (CHAIN: re-read at every layer by the epilogue warps)
    int n_tr = CHAIN ? 0 : hdr->n_tr, n_cond = CHAIN ? 0 : hdr->n_cond, n_chunks = CHAIN ? 0 : hdr->n_chunks;
    int n_lat = CHAIN ? 0 : hdr->n_lat;
    int act = CHAIN ? 0 : hdr->act;
    float s2 = CHAIN ? 1.f : hdr->s2;
    float s2l = s2 * 1.4426950408889634f;
    const int dshift = ((d & (d - 1)) == 0) ? (31 - __clz(d)) : -1;       // d a power of two: divide by shifting
    const int my_tiles = (A.n_tiles > (int)blockIdx.x) ? (A.n_tiles - 1 - (int)blockIdx.x) / (int)gridDim.x + 1 : 0;

    if (warp == 0) {
        // ======================= producer: last-Linear weight chunks =============================
        if (lane == 0) {
            uint32_t cc = 0;
            for (int it = 0; it < my_tiles; ++it) {
                if (it + 1 < my_tiles) {           // pull the NEXT tile's rows into L2 while this one computes
                    const long long nrow0 = ((long long)blockIdx.x + (long long)(it + 1) * gridDim.x) * kTileRows;
                    const long long nb = min((long long)kTileRows, A.rows - nrow0) * d * 4;
                    const char* src = reinterpret_cast<const char*>(A.x + nrow0 * d);
                    if (nb >= 16 && ((reinterpret_cast<uintptr_t>(src) & 15) == 0))
                        asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(src), "r"((uint32_t)(nb & ~15LL)) : "memory");
                }
                for (int l = 0; l < n_layers; ++l) {
                    const uint8_t* img = CHAIN ? A.chain_packed[l] : A.packed;
                    const int nch = CHAIN ? A.n_chunks_l[l] : n_chunks;
                    if (CHAIN) {                   // the layer's head: header | biases | first Linear
                        const uint32_t st = cc % kStages, use = cc / kStages;
                        mbar_wait_relaxed(&bars->b_empty[st], (use & 1) ^ 1);
                        mbar_arrive_expect_tx(&bars->b_full[st], kHeadBytes);
                        bulk_g2s(bst + st * kChunkBytes, img, kHeadBytes, &bars->b_full[st]);
                        ++cc;
                    }
                    for (int c = 0; c < nch; ++c, ++cc) {
                        const uint32_t st = cc % kStages, use = cc / kStages;
                        mbar_wait_relaxed(&bars->b_empty[st], (use & 1) ^ 1);
                        mbar_arrive_expect_tx(&bars->b_full[st], kChunkBytes);
                        bulk_g2s(bst + st * kChunkBytes, img + kOffW2 + (size_t)c * kChunkBytes, kChunkBytes,
                                 &bars->b_full[st]);
                    }
                }
            }
        }
    } else if (warp < kEpiWarp0) {
        // ======================= UMMA issuers: warp 1 -> subtile 0, warp 2 -> subtile 1 ==========
        // One thread issues ~150 instructions per 12-UMMA group (descriptor arithmetic through the
        // uniform datapath); a single issuer for both subtiles was the critical path of the whole
        // kernel (measured: with the spline math removed the kernel ran only 1.24x faster).
        if (lane == 0) {
            const int s = warp - 1;
            const uint32_t idesc1 = make_idesc(FMT_BF16, 128, kHid);
            const uint32_t idesc2 = make_idesc(FMT_F16, 128, kChunkN);
            uint32_t cc = 0;                       // chunk counter (accumulator buffers)
            uint32_t rc = 0;                       // ring item counter (== cc unless CHAIN adds the layer heads)
            uint32_t hp = 0;                       // layer applications so far (phase of the head barriers)
            for (int it = 0; it < my_tiles; ++it)
            for (int l = 0; l < n_layers; ++l, ++hp) {
                const uint32_t tpar = hp & 1;
                const int nch = CHAIN ? A.n_chunks_l[l] : n_chunks;
                {                                  // GEMM1: conditioning columns -> hidden pre-activation
                    uint32_t b0 = smem_u32(w1s);
                    const uint32_t hst = rc % kStages;
                    if (CHAIN) {
                        mbar_wait_relaxed(&bars->b_full[hst], (rc / kStages) & 1);
                        b0 = smem_u32(bst + hst * kChunkBytes) + kOffW1;
                    }
                    mbar_wait_relaxed(&bars->a1_ready[s], tpar);
                    tc_fence_after();
                    const uint32_t a0 = smem_u32(abuf + s * kABytes);
                    const uint32_t dcol = tmem + kColAcc1 + s * kHid;
                    uint32_t acc = 0;
                    // x = x0 + x1 + x2, W = W0 + W1 + W2 (bf16 parts): every product except x2*W2,
                    // SMALLEST first -- the tensor core truncates the running accumulator at every
                    // step (measured: tools/tc_probe.py), so the big x0*W0 term must come last.
#pragma unroll
                    for (int p = 0; p < 8; ++p) {
                        // (pa,pb): (1,2) (2,1) (0,2) (1,1) (2,0) (0,1) (1,0) (0,0)
                        const int pa = (p == 0 || p == 3 || p == 6) ? 1 : ((p == 1 || p == 4) ? 2 : 0);
                        const int pb = (p == 0 || p == 2) ? 2 : ((p == 1 || p == 3 || p == 5) ? 1 : 0);
#pragma unroll
                        for (int ks = 0; ks < kK1 / 16; ++ks) {
                            umma_f16(dcol, make_smem_desc(a0 + pa * kA1Part + ks * 256, 128, 512),
                                     make_smem_desc(b0 + pb * kW1Part + ks * 256, 128, 512), idesc1, acc);
                            acc = 1;
                        }
                    }
                    umma_commit(&bars->acc1_full[s]);
                    if (CHAIN) { umma_commit(&bars->b_empty[hst]); ++rc; }
                }
                for (int c = 0; c < nch; ++c, ++cc, ++rc) {
                    const uint32_t st = rc % kStages, use = rc / kStages;
                    mbar_wait_relaxed(&bars->b_full[st], use & 1);
                    const uint32_t buf = cc & 1, buse = cc >> 1;
                    if (c == 0) mbar_wait_relaxed(&bars->h_ready[s], tpar);
                    mbar_wait_relaxed(&bars->acc_empty[s][buf], (buse & 1) ^ 1);
                    tc_fence_after();
                    const uint32_t a_hi = smem_u32(abuf + s * kABytes), a_lo = a_hi + 16384;
                    const uint32_t b_hi = smem_u32(bst + st * kChunkBytes), b_lo = b_hi + 12288;
                    const uint32_t dcol = tmem + kColAcc2 + (s * 2 + buf) * kChunkN;
                    uint32_t acc = 0;
                    // lo*hi, hi*lo, then hi*hi: small corrections first (accumulator truncation)
#pragma unroll
                    for (int p = 0; p < 3; ++p) {
                        const uint32_t aa = (p == 0) ? a_lo : a_hi, bb = (p == 1) ? b_lo : b_hi;
#pragma unroll
                        for (int ks = 0; ks < kHid / 16; ++ks) {
                            umma_f16(dcol, make_smem_desc(aa + ks * 256, 128, 1024),
                                     make_smem_desc(bb + ks * 256, 128, 1024), idesc2, acc);
                            acc = 1;
                        }
                    }
                    umma_commit(&bars->acc_full[s][buf]);
                    umma_commit(&bars->b_empty[st]);       // stage reusable once both subtiles' UMMAs retire (count 2)
                }
            }
        }
    } else if (warp >= kEpiWarp0) {
        // ======================= epilogue warps ==================================================
        // warp id % 4 fixes the TMEM sub-partition q; the six warps of a residue class are
        // (subtile s, r) for s in {0, 1}, r in {0, 1, 2}: the three warps of a (s, q) triple share the
        // 32 rows and take the transformed dims round-robin (dim n -> warp n % 3), and a third of the
        // row-level work each
        const int q = warp & 3;
        const int cls = (warp - (kEpiWarp0 + ((q - kEpiWarp0) & 3))) >> 2;
        const int s = cls & 1, r3 = cls >> 1;
        const int etid = tid - kEpiWarp0 * 32;
        const int rloc = q * 32 + lane;                         // row within the subtile
        const int rt = s * 128 + rloc;                          // row within the tile
        float* xrow = xs + rt * kXsStride;
        const uint32_t a_row_off = (uint32_t)(rloc >> 3) * 1024 + (uint32_t)(rloc & 7) * 16;
        const uint32_t lane_sel = (uint32_t)(q * 32) << 16;
        const bool want_ld = A.ldj_mode != STB_LDJ_NONE;
        float lo = A.lower, hi = A.upper;
        float inv_span = 1.f / (hi - lo);
        // loop-invariant addresses of the chunk loop, pinned in registers
        const uint32_t full_bar = pin(smem_u32(&bars->acc_full[s][0]));
        const uint32_t empty_bar = pin(smem_u32(&bars->acc_empty[s][0]));
        const uint32_t col_base = pin(tmem + lane_sel + kColAcc2 + (uint32_t)(s * 2) * kChunkN);
        const uint32_t tr_idx_a = pin(smem_u32(&hdr->tr_idx[0]));
        const uint32_t b2_a = pin(smem_u32(b2s));
        const uint32_t xrow_a = pin(smem_u32(xrow));
        uint32_t noshift_mask = CHAIN ? 0u : hdr->noshift_mask;
        uint32_t cc = 0, rc = 0, hp = 0;           // chunk / ring item / layer application counters (as the issuers')

        for (int it = 0; it < my_tiles; ++it) {
            const long long tile = (long long)blockIdx.x + (long long)it * gridDim.x;
            const long long row0 = tile * kTileRows;
            const int nrows = (int)min((long long)kTileRows, A.rows - row0);

            // ---- stage the x tile: coalesced global reads -> padded row-major smem ----------------
            {
                const float* xg = A.x + row0 * d;
                const int n = nrows * d;
                if ((d & 3) == 0 && ((reinterpret_cast<uintptr_t>(xg) & 15) == 0)) {
                    const int n4 = (kTileRows * d) >> 2;
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
                    for (int i = etid; i < kTileRows * d; i += kEpiThreads) {
                        const int r = i / d, c = i - r * d;
                        xs[r * kXsStride + c] = (i < n) ? __ldg(xg + i) : 0.f;
                    }
                }
            }
            named_bar_sync(1, kEpiThreads);
            float ld_acc = 0.f;                    // running log|det J| of this thread's elements (all layers)
#pragma unroll 1
            for (int l = 0; l < n_layers; ++l, ++hp) {
            const uint32_t tpar = hp & 1;
            if (CHAIN) {
                // this layer's header + biases out of its ring stage (the first Linear stays there for GEMM1)
                const uint32_t hst = rc % kStages;
                mbar_wait(&bars->b_full[hst], (rc / kStages) & 1);
                const uint4* src = reinterpret_cast<const uint4*>(bst + hst * kChunkBytes);
                uint4* dst = reinterpret_cast<uint4*>(smem + kSmSmall);
                for (int i = etid; i < (int)(kSmallBytes / 16); i += kEpiThreads) dst[i] = src[i];
                named_bar_sync(1, kEpiThreads);
                if (A.permuted) {             // logical -> physical tile columns of this layer (warp-uniform branch)
                    Header* h = const_cast<Header*>(hdr);
                    if (etid < kK1) { if (etid < h->n_cond) h->cond_idx[etid] = A.perm.phys[l][h->cond_idx[etid]]; }
                    else if (etid < kK1 + kMaxTr) h->tr_idx[etid - kK1] = A.perm.phys[l][h->tr_idx[etid - kK1]];
                    named_bar_sync(1, kEpiThreads);
                }
                n_tr = hdr->n_tr; n_cond = hdr->n_cond; n_chunks = hdr->n_chunks; act = hdr->act;
                n_lat = hdr->n_lat;
                s2 = hdr->s2; s2l = s2 * 1.4426950408889634f;
                noshift_mask = hdr->noshift_mask;
                lo = A.lower_l[l]; hi = A.upper_l[l]; inv_span = 1.f / (hi - lo);
                // keep the three in registers: ptxas otherwise re-derives them (indexed parameter loads and
                // the division) inside the element loop -- 2.4 % of all issued instructions, measured
                asm volatile("" : "+f"(lo), "+f"(hi), "+f"(inv_span));
                rc += 1u + (uint32_t)n_chunks;
            }

            // ---- tile head, software-pipelined over the two subtiles: every warp of a TMEM sub-partition
            // class helps with BOTH subtiles' rows (TMEM lanes are shared, only the columns differ), so
            // GEMM1 of subtile 0 runs under the A1 split of subtile 1, and GEMM1 of subtile 1 / the first
            // GEMM2 chunk of subtile 0 under the tanh passes.
            // A1: the row's conditioning columns as three bf16 parts, 8-column groups round-robin
#pragma unroll 1
            for (int sp = 0; sp < 2; ++sp) {
                const float* xr = xs + (sp * 128 + rloc) * kXsStride;
                uint8_t* a_p = abuf + sp * kABytes;
                const uint32_t a1_row_off = (uint32_t)(rloc >> 3) * 512 + (uint32_t)(rloc & 7) * 16;
#pragma unroll 1
                for (int kc = cls; kc < kK1 / 8; kc += 2 * kEpiPerSub) {
                    __align__(16) __nv_bfloat16 q0[8], q1[8], q2[8];
#pragma unroll
                    for (int u = 0; u < 8; ++u) {
                        const int k = kc * 8 + u;
                        float v = 0.f;
                        if (k < n_cond) v = xr[hdr->cond_idx[k]];
                        else if (k < n_cond + n_lat && sp * 128 + rloc < nrows)
                            v = __ldg(A.latent + (row0 + sp * 128 + rloc) * A.lat_stride + (k - n_cond));
                        split_bf16x3(v, q0[u], q1[u], q2[u]);
                    }
                    *reinterpret_cast<uint4*>(a_p + a1_row_off + kc * 128) = *reinterpret_cast<const uint4*>(q0);
                    *reinterpret_cast<uint4*>(a_p + kA1Part + a1_row_off + kc * 128) = *reinterpret_cast<const uint4*>(q1);
                    *reinterpret_cast<uint4*>(a_p + 2 * kA1Part + a1_row_off + kc * 128) = *reinterpret_cast<const uint4*>(q2);
                }
                fence_proxy_async_smem();
                __syncwarp();
                if (lane == 0) mbar_arrive(&bars->a1_ready[sp]);
            }
            // hidden layer: h = act(acc1 + b1) -> fp16 hi | lo A operand of GEMM2, 8 units at a time
#pragma unroll 1
            for (int sp = 0; sp < 2; ++sp) {
                uint8_t* a_p = abuf + sp * kABytes;
                mbar_wait(&bars->acc1_full[sp], tpar);
                tc_fence_after();
#pragma unroll 1
                for (int kc = cls; kc < kHid / 8; kc += 2 * kEpiPerSub) {
                    const int c0 = kc * 8;
                    float v[8];
                    tmem_ld8(tmem + lane_sel + kColAcc1 + sp * kHid + c0, v);
                    tmem_ld_wait();
                    __align__(16) __half hh[8], hl[8];
                    if (act == STB_ACT_TANH) {
#pragma unroll
                        for (int i = 0; i < 8; ++i) split_f16(tanh_fast(v[i] + b1s[c0 + i]), hh[i], hl[i]);
                    } else {
#pragma unroll
                        for (int i = 0; i < 8; ++i) v[i] = sigmoid_act(v[i] + b1s[c0 + i]);      // STB_ACT_SIGMOID
#pragma unroll
                        for (int i = 0; i < 8; ++i) split_f16(v[i], hh[i], hl[i]);
                    }
                    *reinterpret_cast<uint4*>(a_p + a_row_off + kc * 128) = *reinterpret_cast<const uint4*>(hh);
                    *reinterpret_cast<uint4*>(a_p + 16384 + a_row_off + kc * 128) = *reinterpret_cast<const uint4*>(hl);
                }
                tc_fence_before();
                fence_proxy_async_smem();
                __syncwarp();
                if (lane == 0) mbar_arrive(&bars->h_ready[sp]);
            }

            // ---- last Linear chunks out of TMEM + spline in registers: this warp's dim of each chunk ----
            // dims round-robin over the triple.  A warp visits chunks in increasing order with gaps <= 2,
            // so the phase parity it waits for on an accumulator buffer is never ambiguous: the
            // buffer's previous use (two chunks earlier) completed before a chunk this warp has
            // already consumed.
#pragma unroll 1
            for (int ji = r3; ji < kG * n_chunks; ji += kEpiPerSub) {
                const uint32_t ccc = cc + (uint32_t)(ji >> 1);
                const uint32_t buf = ccc & 1, buse = ccc >> 1;
                const int g = ji & 1;
                uint32_t j4;                                            // 4 * transformed column
                asm volatile("ld.shared.u32 %0, [%1];" : "=r"(j4) : "r"(tr_idx_a + 4u * (uint32_t)(ji < n_tr ? ji : 0)));
                j4 <<= 2;
                float xv;
                asm volatile("ld.shared.f32 %0, [%1];" : "=f"(xv) : "r"(xrow_a + j4));
                const bool inside = (ji < n_tr) && (xv >= lo) && (xv <= hi);
                const float* bb = b2s + ji * kPPad;
                mbar_wait_a(full_bar + buf * 8, buse & 1);
                tc_fence_after();
                const uint32_t col0 = col_base + buf * kChunkN + (uint32_t)g * kPPad;
                float out = xv, ld = 0.f;
                const bool shift = !((noshift_mask >> (ji & 31)) & 1u);
                const float2* bb2 = reinterpret_cast<const float2*>(bb);
                if (KIND == STB_RQS) {
                    RqsLoc loc;
                    {
                        float2 t[kBins];
                        tmem_ld16(col0, reinterpret_cast<float*>(t));
                        tmem_ld16(col0 + 16, reinterpret_cast<float*>(t) + 16);
                        tmem_ld_wait();
                        // (width_i, height_i) pairs, pre-multiplied by log2(e) (exp2-domain softmax): the
                        // bias table holds b * log2(e) for those 32 columns
#pragma unroll
                        for (int i = 0; i < kBins; ++i) t[i] = __ffma2_rn(t[i], f2(s2l), bb2[i]);
                        loc = rqs16_locate<INVERSE>(t, shift, lo, inv_span, xv);
                    }
                    float dd[16];
                    tmem_ld16(col0 + 2 * kBins, dd);
                    tmem_ld_wait();
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive_a(empty_bar + buf * 8);     // TMEM buffer free again
                    if (inside) {
                        // derivative parameter AT knot i (1..15) is column 32 + i - 1; box ends are constants
                        float r0, r1;
                        pick_pair16(dd, loc.k, r0, r1);
                        const float u0 = (loc.k == 0) ? STB_RQS_EDGE_CONST : fmaf(r0, s2, bb[2 * kBins + loc.k - 1]);
                        const float u1 = (loc.k == kBins - 1) ? STB_RQS_EDGE_CONST : fmaf(r1, s2, bb[2 * kBins + loc.k]);
                        rqs16_finish<INVERSE>(loc, u0, u1, lo, hi, want_ld, xv, out, ld);
                    }
                    if (BINS && ji < n_tr && rt < nrows) A.bins[(row0 + rt) * d + (j4 >> 2)] = inside ? loc.k : -1;
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
                        sel = cubic16_locate<INVERSE>(t, shift, u);
                    }
                    float dd[8];
                    tmem_ld8(col0 + 2 * kBins, dd);
                    tmem_ld_wait();
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive_a(empty_bar + buf * 8);
                    if (inside) {
                        const float ul = fmaf(dd[0], s2, bb[2 * kBins]), ur = fmaf(dd[1], s2, bb[2 * kBins + 1]);
                        cubic16_finish<INVERSE>(sel, ul, ur, lo, hi, want_ld, u, out, ld);
                    }
                    if (BINS && ji < n_tr && rt < nrows) A.bins[(row0 + rt) * d + (j4 >> 2)] = inside ? sel.k : -1;
                }
                if (ji < n_tr) asm volatile("st.shared.f32 [%0], %1;" ::"r"(xrow_a + j4), "f"(out) : "memory");
                ld_acc += ld;
            }
            cc += (uint32_t)n_chunks;
            // next layer of the chain: every warp's outputs are in the tile, nobody reads this layer's biases any more
            if (CHAIN && l + 1 < n_layers) named_bar_sync(1, kEpiThreads);
            }   // layers

            // ---- per-row log|det J|: the pair's two partials (+ UnitNormal log-density of the output row) ---
            if (r3 < kEpiPerSub - 1) ld_s[r3 * kTileRows + rt] = ld_acc;
            named_bar_sync(1, kEpiThreads);
            if (r3 == kEpiPerSub - 1 && want_ld && rt < nrows) {      // fixed summation order: deterministic
                float tot = ld_s[rt];
#pragma unroll
                for (int o = 1; o < kEpiPerSub - 1; ++o) tot += ld_s[o * kTileRows + rt];
                tot += ld_acc;
                if (A.base_log_prob) {
                    float b = 0.f;
                    for (int c = 0; c < d; ++c) { const float v = xrow[c]; b += -0.5f * v * v - 0.91893853320467274178f; }
                    tot += b;
                }
                float* dst = A.ldj + row0 + rt;
                *dst = (A.ldj_mode == STB_LDJ_ADD) ? (*dst + tot) : tot;
            }

            // ---- y tile out (coalesced); log_prob callers that do not want the latent rows pass y == NULL -------
            if (A.y != nullptr) {
                float* yg = A.y + row0 * d;
                const int n = nrows * d;
                if (CHAIN && A.permuted) {                            // the accumulated permutation, on the way out
                    for (int i = etid; i < n; i += kEpiThreads) {
                        const int r = (dshift >= 0) ? (i >> dshift) : i / d, c = i - r * d;
                        yg[i] = xs[r * kXsStride + A.perm.out_phys[c]];
                    }
                } else if ((d & 3) == 0 && ((reinterpret_cast<uintptr_t>(yg) & 15) == 0)) {
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

    // ---- teardown --------------------------------------------------------------------------------------
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem, kTmemCols);
}

// -----------------------------------------------------------------------------------------------
// the whole-flow kernel as TWO independent CTAs per SM: tc_spline_pair_kernel
// -----------------------------------------------------------------------------------------------
// Same layers, same arithmetic, same packed image and the same bits out as the CHAIN kernel above, reorganised around
// what its per-warp phase clocks showed (8 layers): per 256-row tile and layer the 16 epilogue warps spend
// 8.5 k of 46.8 k clocks in the layer HEAD (A1 split -> GEMM1 -> tanh -> first chunk) with the tensor pipe idle, and the
// issuers 26 % of theirs waiting for accumulator buffers.  One CTA cannot overlap a layer's head with anything: the next
// layer needs every output of this one.  Two CTAs per SM, each with its own 128-row tile, do -- their heads fall into
// each other's chunk phases.  To fit twice (114.7 KB of shared memory, 256 TMEM columns, 320 threads x 96 registers per
// CTA) the A operands leave shared memory:
//   * GEMM1's A operand (the row's conditioning columns as three bf16 parts, 48 columns) is written with tcgen05.st
//     into the columns of accumulator buffer 1, which is idle between two layers, and read from there by TMEM-sourced
//     UMMAs (the first chunk that lands in that buffer is issued after GEMM1 and executes after it);
//   * the hidden activations go back into GEMM1's accumulator columns in place (fp16 hi at +0, lo at +8 of every
//     16-column block) and GEMM2 reads them from there: no shared-memory A buffer, no proxy fence in the layer head.
// Each CTA streams its own copy of the weight chunks (2 x 404 KB per 256 rows and layer, ~40 % of the L2 slices' rate).
constexpr int kPRows = 128;
constexpr int kPEpiWarp0 = 2;                                // warp 0 producer, warp 1 issuer
constexpr int kPEpiWarps = 8;                                // (TMEM sub-partition q, half r3): two per scheduler
constexpr int kPThreads = (kPEpiWarp0 + kPEpiWarps) * 32;
constexpr int kPEpiThreads = kPEpiWarps * 32;
constexpr uint32_t kPSmXs = 0;                                          // float [128][65]; column 64 carries log-det partials
constexpr uint32_t kPSmB = kPRows * kXsStride * 4;
constexpr uint32_t kPSmSmall = kPSmB + kStages * kChunkBytes;
constexpr uint32_t kPSmBar = (kPSmSmall + kSmallBytes + 15) & ~15u;
constexpr uint32_t kPSmemBytes = kPSmBar + 256;
static_assert(kPSmB % 128 == 0 && kPSmSmall % 16 == 0, "alignment");
static_assert(2 * (kPSmemBytes + 1024) <= 228 * 1024, "two CTAs per SM");
struct PBars {
    uint64_t acc_full[2], acc_empty[2];
    uint64_t b_full[kStages], b_empty[kStages];
    uint64_t a1_ready, acc1_full, h_ready;
    uint32_t tmem_base;
};
static_assert(sizeof(PBars) <= 256, "barrier block");
constexpr uint32_t kPColH = 0;                               // GEMM1 accumulator, then h in place
constexpr uint32_t kPColAcc = kHid;                          // + buf * 96
constexpr uint32_t kPColA1 = kPColAcc + kChunkN;             // inside buffer 1: part pa at + pa * 16, K step ks at + ks * 8
constexpr uint32_t kPTmemCols = 256;

__device__ __forceinline__ void tmem_st4(uint32_t taddr, const uint32_t* r) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1, %2, %3, %4};" ::"r"(taddr), "r"(r[0]), "r"(r[1]),
                 "r"(r[2]), "r"(r[3])
                 : "memory");
}

// FULL = false: layers with fewer than 16 bins (2 .. 16, read per layer from the header; tc_spline16.cuh)
template <int KIND, bool INVERSE, bool FULL = true>
__global__ void __launch_bounds__(kPThreads, 2) tc_spline_pair_kernel(const Args A) {
    extern __shared__ __align__(128) uint8_t smem_p[];      // (1024 would cost a kilobyte of static padding: 2 CTAs then need all 228 KB)
    uint8_t* smem = smem_p;
    float* xs = reinterpret_cast<float*>(smem + kPSmXs);
    uint8_t* bst = smem + kPSmB;
    const Header* hdr = reinterpret_cast<const Header*>(smem + kPSmSmall);
    const float* b1s = reinterpret_cast<const float*>(smem + kPSmSmall + kOffB1);
    const float* b2s = reinterpret_cast<const float*>(smem + kPSmSmall + kOffB2);
    PBars* bars = reinterpret_cast<PBars*>(smem + kPSmBar);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    if (tid == 0) {
        for (int i = 0; i < kStages; ++i) { mbar_init(&bars->b_full[i], 1); mbar_init(&bars->b_empty[i], 1); }
        mbar_init(&bars->a1_ready, kPEpiWarps);
        mbar_init(&bars->acc1_full, 1);
        mbar_init(&bars->h_ready, kPEpiWarps);
        for (int b = 0; b < 2; ++b) { mbar_init(&bars->acc_full[b], 1); mbar_init(&bars->acc_empty[b], kPEpiWarps); }
        fence_mbar_init();
    }
    if (warp == 1) tmem_alloc(&bars->tmem_base, kPTmemCols);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = bars->tmem_base;

    const int n_layers = A.n_layers;
    const int d = A.dim;
    const int dshift = ((d & (d - 1)) == 0) ? (31 - __clz(d)) : -1;
    const int my_tiles = (A.n_tiles > (int)blockIdx.x) ? (A.n_tiles - 1 - (int)blockIdx.x) / (int)gridDim.x + 1 : 0;

    if (warp == 0) {
        // ======================= producer: per layer the head item, then the last Linear's chunks =======================
        if (lane == 0) {
            uint32_t rc = 0;
            for (int it = 0; it < my_tiles; ++it) {
                if (it + 1 < my_tiles) {
                    const long long nrow0 = ((long long)blockIdx.x + (long long)(it + 1) * gridDim.x) * kPRows;
                    const long long nb = min((long long)kPRows, A.rows - nrow0) * d * 4;
                    const char* src = reinterpret_cast<const char*>(A.x + nrow0 * d);
                    if (nb >= 16 && ((reinterpret_cast<uintptr_t>(src) & 15) == 0))
                        asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(src), "r"((uint32_t)(nb & ~15LL)) : "memory");
                }
                for (int l = 0; l < n_layers; ++l) {
                    const uint8_t* img = A.chain_packed[l];
                    const int nch = A.n_chunks_l[l];
                    for (int c = -1; c < nch; ++c, ++rc) {
                        const uint32_t st = rc % kStages, use = rc / kStages;
                        mbar_wait_relaxed(&bars->b_empty[st], (use & 1) ^ 1);
                        const uint32_t bytes = (c < 0) ? kHeadBytes : kChunkBytes;
                        mbar_arrive_expect_tx(&bars->b_full[st], bytes);
                        bulk_g2s(bst + st * kChunkBytes, (c < 0) ? img : img + kOffW2 + (size_t)c * kChunkBytes, bytes, &bars->b_full[st]);
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ======================= UMMA issuer: both A operands come from TMEM ============================================
        if (lane == 0) {
            const uint32_t idesc1 = make_idesc(FMT_BF16, 128, kHid);
            const uint32_t idesc2 = make_idesc(FMT_F16, 128, kChunkN);
            uint32_t cc = 0, rc = 0, hp = 0;
            for (int it = 0; it < my_tiles; ++it)
            for (int l = 0; l < n_layers; ++l, ++hp) {
                const uint32_t tpar = hp & 1;
                const int nch = A.n_chunks_l[l];
                {
                    const uint32_t hst = rc % kStages;
                    mbar_wait_relaxed(&bars->b_full[hst], (rc / kStages) & 1);
                    const uint32_t b0 = smem_u32(bst + hst * kChunkBytes) + kOffW1;
                    mbar_wait_relaxed(&bars->a1_ready, tpar);
                    tc_fence_after();
                    uint32_t acc = 0;
                    // the same eight partial products in the same order as the kernel above (smallest first)
#pragma unroll
                    for (int p = 0; p < 8; ++p) {
                        const int pa = (p == 0 || p == 3 || p == 6) ? 1 : ((p == 1 || p == 4) ? 2 : 0);
                        const int pb = (p == 0 || p == 2) ? 2 : ((p == 1 || p == 3 || p == 5) ? 1 : 0);
#pragma unroll
                        for (int ks = 0; ks < kK1 / 16; ++ks) {
                            umma_f16_ts(tmem + kPColH, tmem + kPColA1 + pa * 16 + ks * 8,
                                        make_smem_desc(b0 + pb * kW1Part + ks * 256, 128, 512), idesc1, acc);
                            acc = 1;
                        }
                    }
                    umma_commit(&bars->acc1_full);
                    umma_commit(&bars->b_empty[hst]);
                    ++rc;
                }
                for (int c = 0; c < nch; ++c, ++cc, ++rc) {
                    const uint32_t st = rc % kStages, use = rc / kStages;
                    mbar_wait_relaxed(&bars->b_full[st], use & 1);
                    const uint32_t buf = cc & 1, buse = cc >> 1;
                    if (c == 0) mbar_wait_relaxed(&bars->h_ready, tpar);
                    mbar_wait_relaxed(&bars->acc_empty[buf], (buse & 1) ^ 1);
                    tc_fence_after();
                    const uint32_t b_hi = smem_u32(bst + st * kChunkBytes), b_lo = b_hi + 12288;
                    const uint32_t dcol = tmem + kPColAcc + buf * kChunkN;
                    uint32_t acc = 0;
#pragma unroll
                    for (int p = 0; p < 3; ++p) {                  // lo*hi, hi*lo, hi*hi
                        const uint32_t a_off = (p == 0) ? 8u : 0u, bb = (p == 1) ? b_lo : b_hi;
#pragma unroll
                        for (int ks = 0; ks < kHid / 16; ++ks) {
                            umma_f16_ts(dcol, tmem + kPColH + ks * 16 + a_off, make_smem_desc(bb + ks * 256, 128, 1024), idesc2, acc);
                            acc = 1;
                        }
                    }
                    umma_commit(&bars->acc_full[buf]);
                    umma_commit(&bars->b_empty[st]);
                }
            }
        }
    } else {
        // ======================= epilogue warps: (q, r3), thread = row ======================================================
        const int q = warp & 3;
        const int r3 = (warp - kPEpiWarp0) >> 2;
        const int etid = tid - kPEpiWarp0 * 32;
        const int rt = q * 32 + lane;
        float* xrow = xs + rt * kXsStride;
        const uint32_t lane_sel = (uint32_t)(q * 32) << 16;
        const bool want_ld = A.ldj_mode != STB_LDJ_NONE;
        const uint32_t full_bar = pin(smem_u32(&bars->acc_full[0]));
        const uint32_t empty_bar = pin(smem_u32(&bars->acc_empty[0]));
        const uint32_t col_base = pin(tmem + lane_sel + kPColAcc);
        const uint32_t tr_idx_a = pin(smem_u32(&hdr->tr_idx[0]));
        const uint32_t xrow_a = pin(smem_u32(xrow));
        uint32_t cc = 0, rc = 0, hp = 0;

        for (int it = 0; it < my_tiles; ++it) {
            const long long tile = (long long)blockIdx.x + (long long)it * gridDim.x;
            const long long row0 = tile * kPRows;
            const int nrows = (int)min((long long)kPRows, A.rows - row0);
            {   // ---- stage the x tile ---------------------------------------------------------------------------
                const float* xg = A.x + row0 * d;
                const int n = nrows * d;
                if ((d & 3) == 0 && ((reinterpret_cast<uintptr_t>(xg) & 15) == 0)) {
                    const int n4 = (kPRows * d) >> 2;
                    for (int i0 = etid; i0 < n4; i0 += kPEpiThreads * 4) {
                        float4 v[4];
#pragma unroll
                        for (int u = 0; u < 4; ++u) {
                            const int i = i0 + u * kPEpiThreads;
                            v[u] = (i < n4 && i * 4 < n) ? __ldg(reinterpret_cast<const float4*>(xg) + i)
                                                         : make_float4(0.f, 0.f, 0.f, 0.f);
                        }
#pragma unroll
                        for (int u = 0; u < 4; ++u) {
                            const int i = i0 + u * kPEpiThreads;
                            if (i < n4) {
                                const int r = (dshift >= 0) ? ((i * 4) >> dshift) : (i * 4) / d, c = (i * 4) - r * d;
                                float* dst = xs + r * kXsStride + c;
                                dst[0] = v[u].x; dst[1] = v[u].y; dst[2] = v[u].z; dst[3] = v[u].w;
                            }
                        }
                    }
                } else {
                    for (int i = etid; i < kPRows * d; i += kPEpiThreads) {
                        const int r = i / d, c = i - r * d;
                        xs[r * kXsStride + c] = (i < n) ? __ldg(xg + i) : 0.f;
                    }
                }
            }
            named_bar_sync(1, kPEpiThreads);
            float ld_acc = 0.f;
#pragma unroll 1
            for (int l = 0; l < n_layers; ++l, ++hp) {
                const uint32_t tpar = hp & 1;
                {   // this layer's header + biases out of its ring stage (the first Linear stays there for GEMM1)
                    const uint32_t hst = rc % kStages;
                    mbar_wait(&bars->b_full[hst], (rc / kStages) & 1);
                    const uint4* src = reinterpret_cast<const uint4*>(bst + hst * kChunkBytes);
                    uint4* dst = reinterpret_cast<uint4*>(smem + kPSmSmall);
                    for (int i = etid; i < (int)(kSmallBytes / 16); i += kPEpiThreads) dst[i] = src[i];
                    named_bar_sync(1, kPEpiThreads);
                    if (A.permuted) {
                        Header* h = const_cast<Header*>(hdr);
                        if (etid < kK1) { if (etid < h->n_cond) h->cond_idx[etid] = A.perm.phys[l][h->cond_idx[etid]]; }
                        else if (etid < kK1 + kMaxTr) h->tr_idx[etid - kK1] = A.perm.phys[l][h->tr_idx[etid - kK1]];
                        named_bar_sync(1, kPEpiThreads);
                    }
                }
                const int n_tr = hdr->n_tr, n_cond = hdr->n_cond, n_chunks = hdr->n_chunks, act = hdr->act;
                const int n_lat = hdr->n_lat;
                const int K = FULL ? kBins : hdr->n_bins;
                const float s2 = hdr->s2, s2l = s2 * 1.4426950408889634f;
                const uint32_t noshift_mask = hdr->noshift_mask;
                float lo = A.lower_l[l], hi = A.upper_l[l], inv_span = 1.f / (hi - lo);
                asm volatile("" : "+f"(lo), "+f"(hi), "+f"(inv_span));
                rc += 1u + (uint32_t)n_chunks;

                // ---- A1 into TMEM: this warp's two 8-column groups of the row's conditioning columns, three bf16 parts ----
#pragma unroll 1
                for (int kc = r3; kc < kK1 / 8; kc += 2) {
                    __align__(16) __nv_bfloat16 q0[8], q1[8], q2[8];
#pragma unroll
                    for (int u = 0; u < 8; ++u) {
                        const int k = kc * 8 + u;
                        float v = 0.f;
                        if (k < n_cond) v = xrow[hdr->cond_idx[k]];
                        else if (k < n_cond + n_lat && rt < nrows) v = __ldg(A.latent + (row0 + rt) * A.lat_stride + (k - n_cond));
                        split_bf16x3(v, q0[u], q1[u], q2[u]);
                    }
                    const uint32_t col = tmem + lane_sel + kPColA1 + (uint32_t)(kc >> 1) * 8 + (uint32_t)(kc & 1) * 4;
                    tmem_st4(col, reinterpret_cast<const uint32_t*>(q0));
                    tmem_st4(col + 16, reinterpret_cast<const uint32_t*>(q1));
                    tmem_st4(col + 32, reinterpret_cast<const uint32_t*>(q2));
                }
                tmem_st_wait();
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&bars->a1_ready);
                // ---- hidden layer in place: this warp's 32 of the 64 units ----------------------------------------------------
                mbar_wait(&bars->acc1_full, tpar);
                tc_fence_after();
#pragma unroll 1
                for (int blk = 0; blk < 2; ++blk) {
                    const int c0 = r3 * 32 + blk * 16;
                    float v[16];
                    tmem_ld16(tmem + lane_sel + kPColH + c0, v);
                    tmem_ld_wait();
                    uint32_t hh[8], hl[8];
                    if (act == STB_ACT_TANH) {
#pragma unroll
                        for (int i = 0; i < 8; ++i)
                            split_f16x2_sat(tanh_fast(v[2 * i] + b1s[c0 + 2 * i]), tanh_fast(v[2 * i + 1] + b1s[c0 + 2 * i + 1]), hh[i], hl[i]);
                    } else {
#pragma unroll
                        for (int i = 0; i < 8; ++i)
                            split_f16x2_sat(sigmoid_act(v[2 * i] + b1s[c0 + 2 * i]), sigmoid_act(v[2 * i + 1] + b1s[c0 + 2 * i + 1]), hh[i], hl[i]);
                    }
                    tmem_st8(tmem + lane_sel + kPColH + c0, hh);
                    tmem_st8(tmem + lane_sel + kPColH + c0 + 8, hl);
                }
                tmem_st_wait();
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&bars->h_ready);

                // ---- last Linear chunks out of TMEM + spline in registers: this warp's dim of each chunk (as above) ----
#pragma unroll 1
                for (int ji = r3; ji < kG * n_chunks; ji += 2) {
                    const uint32_t ccc = cc + (uint32_t)(ji >> 1);
                    const uint32_t buf = ccc & 1, buse = ccc >> 1;
                    const int g = ji & 1;
                    uint32_t j4;
                    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(j4) : "r"(tr_idx_a + 4u * (uint32_t)(ji < n_tr ? ji : 0)));
                    j4 <<= 2;
                    float xv;
                    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(xv) : "r"(xrow_a + j4));
                    const bool inside = (ji < n_tr) && (xv >= lo) && (xv <= hi);
                    const float* bb = b2s + ji * kPPad;
                    mbar_wait_a(full_bar + buf * 8, buse & 1);
                    tc_fence_after();
                    const uint32_t col0 = col_base + buf * kChunkN + (uint32_t)g * kPPad;
                    float out = xv, ld = 0.f;
                    const bool shift = !((noshift_mask >> (ji & 31)) & 1u);
                    const float2* bb2 = reinterpret_cast<const float2*>(bb);
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
                        if (lane == 0) mbar_arrive_a(empty_bar + buf * 8);
                        if (inside) {
                            float r0, r1;
                            pick_pair16(dd, loc.k, r0, r1);
                            const float u0 = (loc.k == 0) ? STB_RQS_EDGE_CONST : fmaf(r0, s2, bb[2 * kBins + loc.k - 1]);
                            const float u1 = (loc.k == K - 1) ? STB_RQS_EDGE_CONST : fmaf(r1, s2, bb[2 * kBins + loc.k]);
                            rqs16_finish<INVERSE>(loc, u0, u1, lo, hi, want_ld, xv, out, ld, K);
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
                        if (lane == 0) mbar_arrive_a(empty_bar + buf * 8);
                        if (inside) {
                            const float ul = fmaf(dd[0], s2, bb[2 * kBins]), ur = fmaf(dd[1], s2, bb[2 * kBins + 1]);
                            cubic16_finish<INVERSE>(sel, ul, ur, lo, hi, want_ld, u, out, ld, K);
                        }
                    }
                    if (ji < n_tr) asm volatile("st.shared.f32 [%0], %1;" ::"r"(xrow_a + j4), "f"(out) : "memory");
                    ld_acc += ld;
                }
                cc += (uint32_t)n_chunks;
                // next layer: every warp's outputs are in the tile, nobody reads this layer's biases or its accumulators
                if (l + 1 < n_layers) named_bar_sync(1, kPEpiThreads);
            }   // layers

            // ---- per-row log|det J| (+ UnitNormal log-density of the output row): fixed summation order ------------------
            if (r3 == 0) xrow[kMaxDim] = ld_acc;
            named_bar_sync(1, kPEpiThreads);
            if (r3 == 1 && want_ld && rt < nrows) {
                float tot = xrow[kMaxDim];
                tot += ld_acc;
                if (A.base_log_prob) {
                    float b = 0.f;
                    for (int c = 0; c < d; ++c) { const float v = xrow[c]; b += -0.5f * v * v - 0.91893853320467274178f; }
                    tot += b;
                }
                float* dst = A.ldj + row0 + rt;
                *dst = (A.ldj_mode == STB_LDJ_ADD) ? (*dst + tot) : tot;
            }
            if (A.y != nullptr) {
                float* yg = A.y + row0 * d;
                const int n = nrows * d;
                if (A.permuted) {
                    for (int i = etid; i < n; i += kPEpiThreads) {
                        const int r = (dshift >= 0) ? (i >> dshift) : i / d, c = i - r * d;
                        yg[i] = xs[r * kXsStride + A.perm.out_phys[c]];
                    }
                } else if ((d & 3) == 0 && ((reinterpret_cast<uintptr_t>(yg) & 15) == 0)) {
                    const int n4 = n >> 2;
                    for (int i = etid; i < n4; i += kPEpiThreads) {
                        const int r = (dshift >= 0) ? ((i * 4) >> dshift) : (i * 4) / d, c = (i * 4) - r * d;
                        const float* src = xs + r * kXsStride + c;
                        reinterpret_cast<float4*>(yg)[i] = make_float4(src[0], src[1], src[2], src[3]);
                    }
                } else {
                    for (int i = etid; i < n; i += kPEpiThreads) {
                        const int r = i / d, c = i - r * d;
                        yg[i] = xs[r * kXsStride + c];
                    }
                }
            }
            named_bar_sync(1, kPEpiThreads);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem, kPTmemCols);
}

// -----------------------------------------------------------------------------------------------
// packing
// -----------------------------------------------------------------------------------------------
// the image's layout for spline64_pack_kernel (tc_pack.cuh)
struct PackLayout {
    using Hdr = Header;
    static constexpr uint32_t kMagic = tcl::kMagic, kOffB1 = tcl::kOffB1, kOffW1 = tcl::kOffW1;
    static constexpr int kK1 = tcl::kK1, kMaxTr = tcl::kMaxTr;
    static __device__ void header_extra(Header*, const SplinePackArgs&) {}
};

// the shared spline gate, then this file's conditioner: MLP[64]
static_assert(kMaxTr == kK1, "spline_gate bounds the transformed dims by GEMM1's K");
static bool admit(const stb_layer* L, MaskSplit& m) {
    return spline_gate(L, kMaxDim, kK1, m) && L->net.n_linear == 2 && L->net.dims[1] == kHid;
}

}  // namespace tcl

bool tc_layer_supported(const stb_layer* L) {
    tcl::MaskSplit m;
    return tcl::admit(L, m);
}

uint64_t tc_packed_bytes(const stb_layer*) { return tcl::kPackedBytes; }

int tc_pack_layer(const stb_layer* L, void* out, cudaStream_t stream) {
    using namespace tcl;
    SplinePackArgs a;
    if (!admit(L, a.m)) return set_error(STB_ENOTSUP, "layer has no tensor-core path");
    a.out = static_cast<uint8_t*>(out);
    a.n_chunks = (a.m.n_tr + kG - 1) / kG;
    a.n_lat = L->latent_dim; a.n_bins = L->n_bins;
    a.kind = L->kind; a.dim = L->dim; a.P = spline_params_per_dim(L->kind, L->n_bins);
    a.act = L->net.activation;
    a.W1 = L->net.W[0]; a.b1 = L->net.b[0]; a.W2 = L->net.W[1]; a.b2 = L->net.b[1];
    const BoundArgs b = spline_bound_args(a.m, a.W2, a.b2, kHid, a.P, a.n_bins, a.act,
                                          a.out + offsetof(Header, noshift_mask));
    return pack_image(out, sizeof(Header), stream, "tc_pack", [&] {
        pack_pass(spline64_maxabs_kernel<PackLayout>, 64, 256, stream, a);
        pack_pass(spline64_pack_kernel<PackLayout>, 296, 256, stream, a);
        pack_pass(tc_bound_kernel, 1, kMaxTr * 32, stream, b);
    });
}

namespace tcl {
// the two-CTA whole-flow kernel over A.n_layers >= 1 layers (A.chain_packed / lower_l / upper_l / n_chunks_l filled)
static int launch_pair(Args& A, int kind, bool full, int64_t rows, cudaStream_t stream) {
    void (*kern)(Args) = pick_variant(kind, A.inverse, full, [](auto K, auto I, auto F) { return tc_spline_pair_kernel<K, I, F>; });
    const long long ptiles = (rows + kPRows - 1) / kPRows;
    if (ptiles > 0x7fffffffLL) return set_error(STB_EINVAL, "too many rows");
    A.n_tiles = (int)ptiles;
    const cudaError_t pe = cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
    if (pe != cudaSuccess) return set_error(STB_ECUDA, "cudaFuncSetAttribute: %s", cudaGetErrorString(pe));
    return launch_persistent(kern, A, ptiles, 2, kPThreads, kPSmemBytes, stream, "tc_spline_pair_kernel");
}
}  // namespace tcl

int tc_layer_apply(const stb_layer* L, int direction, const float* x, const float* latent, float* y, float* ldj,
                   int ldj_mode, int base_log_prob, int64_t rows, cudaStream_t stream, int32_t* bins) {
    using namespace tcl;
    if (L->packed_bytes < kPackedBytes) return set_error(STB_EINVAL, "packed image too small");
    Args A = {};
    A.bins = bins;
    A.latent = L->latent_dim > 0 ? latent : nullptr;
    A.lat_stride = L->latent_dim;
    if (L->n_bins != kBins) {            // fewer than 16 bins: the padded-bin variant lives in the two-CTA kernel
        if (bins) return set_error(STB_ENOTSUP, "the bin-index instrument of the tensor-core path covers 16-bin layers");
        MaskSplit m;
        if (!admit(L, m)) return set_error(STB_EINVAL, "layer has no tensor-core path");
        A.x = x; A.y = y; A.ldj = ldj;
        A.ldj_mode = ldj ? ldj_mode : STB_LDJ_NONE;
        A.base_log_prob = base_log_prob;
        A.inverse = direction == STB_INVERSE;
        A.rows = rows;
        A.n_layers = 1; A.dim = L->dim;
        A.chain_packed[0] = static_cast<const uint8_t*>(L->packed);
        A.lower_l[0] = L->lower; A.upper_l[0] = L->upper;
        A.n_chunks_l[0] = (m.n_tr + kG - 1) / kG;
        return launch_pair(A, L->kind, false, rows, stream);
    }
    A.packed = static_cast<const uint8_t*>(L->packed);
    A.x = x; A.y = y; A.ldj = ldj;
    A.ldj_mode = ldj ? ldj_mode : STB_LDJ_NONE;
    A.base_log_prob = base_log_prob;
    A.inverse = direction == STB_INVERSE;
    A.lower = L->lower; A.upper = L->upper;
    A.rows = rows;
    const long long tiles = (rows + kTileRows - 1) / kTileRows;
    if (tiles > 0x7fffffffLL) return set_error(STB_EINVAL, "too many rows");
    A.n_tiles = (int)tiles;

    void (*kern)(Args) = pick_variant(L->kind, A.inverse, bins != nullptr,
                                      [](auto K, auto I, auto B) { return tc_spline_layer_kernel<K, I, false, B>; });
    return launch_persistent(kern, A, tiles, 1, kThreads, kSmemBytes, stream, "tc_spline_layer_kernel");
}


// ---- a run of layers of one flow in ONE launch (flow.py:104-107 / 118-125 inside the kernel) -----------
bool tc_chain_supported(const stb_layer* const* layers, int n) {
    using namespace tcl;
    if (n < 2 || n > kMaxChain) return false;
    for (int i = 0; i < n; ++i) {
        const stb_layer* L = layers[i];
        if (!L->packed || L->packed_bytes < kPackedBytes || !tc_layer_supported(L)) return false;
        if (L->kind != layers[0]->kind || L->dim != layers[0]->dim) return false;
        if (L->latent_dim != layers[0]->latent_dim) return false;          // one latent row layout for the whole launch
    }
    return true;
}

// layers[] in APPLICATION order (the caller reverses them for the inverse direction)
int tc_chain_apply(const stb_layer* const* layers, int n, int direction, const float* x, const float* latent, float* y,
                   float* ldj, int ldj_mode, int base_log_prob, int64_t rows, cudaStream_t stream, const ChainPerm* perm) {
    using namespace tcl;
    if (!tc_chain_supported(layers, n)) return set_error(STB_EINVAL, "layers cannot be chained");
    Args A = {};
    A.latent = layers[0]->latent_dim > 0 ? latent : nullptr;
    A.lat_stride = layers[0]->latent_dim;
    if (A.lat_stride > 0 && !latent) return set_error(STB_EINVAL, "layer expects a latent input");
    if (perm) { A.permuted = 1; A.perm = *perm; }
    A.packed = static_cast<const uint8_t*>(layers[0]->packed);
    A.x = x; A.y = y; A.ldj = ldj;
    A.ldj_mode = ldj ? ldj_mode : STB_LDJ_NONE;
    A.base_log_prob = base_log_prob;
    A.inverse = direction == STB_INVERSE;
    A.lower = layers[0]->lower; A.upper = layers[0]->upper;
    A.rows = rows;
    A.n_layers = n;
    A.dim = layers[0]->dim;
    for (int i = 0; i < n; ++i) {
        MaskSplit m;
        if (!admit(layers[i], m)) return set_error(STB_EINVAL, "layer has no tensor-core path");
        A.chain_packed[i] = static_cast<const uint8_t*>(layers[i]->packed);
        A.lower_l[i] = layers[i]->lower; A.upper_l[i] = layers[i]->upper;
        A.n_chunks_l[i] = (m.n_tr + kG - 1) / kG;
    }
    const long long tiles = (rows + kTileRows - 1) / kTileRows;
    if (tiles > 0x7fffffffLL) return set_error(STB_EINVAL, "too many rows");
    A.n_tiles = (int)tiles;
    // Two independent 128-row CTAs per SM instead of one 256-row CTA.  Measured on the headline workload (2^22 rows):
    // 1.73e8 vs 1.77e8 samples/s -- the heads do fall into the other CTA's chunk phases, but the kernel is bound by
    // the epilogue's instruction stream, not by that bubble, so nothing is gained; it IS faster when there are fewer
    // 256-row tiles than SMs (twice as many CTAs to spread over the machine), which is when it is selected -- and it
    // is the kernel of layers with fewer than 16 bins.
    bool full = true;
    for (int i = 0; i < n; ++i) full = full && layers[i]->n_bins == kBins;
    const bool use_pair = !full || tiles < (long long)sm_count();
    if (use_pair) return launch_pair(A, layers[0]->kind, full, rows, stream);
    void (*kern)(Args) = pick_variant(layers[0]->kind, A.inverse, [](auto K, auto I) { return tc_spline_layer_kernel<K, I, true>; });
    return launch_persistent(kern, A, tiles, 1, kThreads, kSmemBytes, stream, "tc_spline_layer_kernel (chain)");
}

}  // namespace stb
