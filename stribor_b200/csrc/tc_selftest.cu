// Bring-up / regression check of the tcgen05 building blocks in tc_common.cuh: a single-CTA
// GEMM  D[128, N] = A[128, K] * B[N, K]^T  that packs its operands into the no-swizzle K-major
// core-matrix layout, issues UMMAs from one thread, and reads the accumulator back from TMEM.
// Exposed as stb_tc_selftest (include/stribor_b200.h); tests/test_gpu_tc.py compares it with a
// PyTorch matmul for fp16 / tf32, single-pass and the 3-pass hi/lo split the layer kernel uses.
#include "common.cuh"
#include "tc_common.cuh"
#include "tc_pack.cuh"

namespace stb {
using namespace tc;

__device__ void pack_operand(uint8_t* hi_s, uint8_t* lo_s, const float* g, int rows, int K, int tf32) {
    for (int i = threadIdx.x; i < rows * K; i += blockDim.x) {
        const int r = i / K, k = i - r * K;
        const float v = g[i];
        if (tf32) {
            float hi, lo;
            split_tf32(v, hi, lo);
            const uint32_t off = core_off(r, k, K, 4);
            *reinterpret_cast<float*>(hi_s + off) = hi;
            *reinterpret_cast<float*>(lo_s + off) = lo;
        } else {
            __half hi, lo;
            split_f16(v, hi, lo);
            const uint32_t off = core_off(r, k, K, 2);
            *reinterpret_cast<__half*>(hi_s + off) = hi;
            *reinterpret_cast<__half*>(lo_s + off) = lo;
        }
    }
}

__global__ void __launch_bounds__(128) tc_selftest_kernel(const float* A, const float* B, float* D, int K,
                                                          int N, int mode, int variant) {
    extern __shared__ __align__(128) uint8_t smem[];
    __shared__ uint64_t bar;
    __shared__ uint32_t tmem_base_s;
    const int tf32 = mode & 1, split = mode >> 1;
    const int elem = tf32 ? 4 : 2, epc = 16 / elem, chunks = K / epc;
    const uint32_t a_bytes = 128u * K * elem, b_bytes = (uint32_t)N * K * elem;
    uint8_t* a_hi = smem;
    uint8_t* a_lo = a_hi + a_bytes;
    uint8_t* b_hi = a_lo + a_bytes;
    uint8_t* b_lo = b_hi + b_bytes;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    // variant bit 2 / bit 3: A / B is given TRANSPOSED (A [K,128], B [K,N]) and consumed MN-major.  The
    // core-matrix packing of the [K rows, M cols] matrix is the same: an MN-major view needs no copy
    // (tc_wide.cu reuses its K-major buffers this way for the gradient products).
    const bool a_mn = (variant & 4) != 0, b_mn = (variant & 8) != 0;
    if (a_mn) pack_operand(a_hi, a_lo, A, K, 128, tf32);
    else pack_operand(a_hi, a_lo, A, 128, K, tf32);
    if (b_mn) pack_operand(b_hi, b_lo, B, K, N, tf32);
    else pack_operand(b_hi, b_lo, B, N, K, tf32);
    fence_proxy_async_smem();

    // variant bit 4: the A operand (fp16 hi | lo) lives in TMEM behind the accumulator -- lane = row, two K elements per
    // 32-bit column -- written by its row's thread with tcgen05.st and consumed by TMEM-sourced UMMAs
    const bool a_tmem = (variant & 16) != 0;
    const uint32_t col_a = ((uint32_t)N + 31u) & ~31u;
    uint32_t ncols = 32;
    while (ncols < (a_tmem ? col_a + (uint32_t)K : (uint32_t)N)) ncols <<= 1;
    if (warp == 0) tmem_alloc(&tmem_base_s, ncols);
    if (threadIdx.x == 0) {
        mbar_init(&bar, 1);
        fence_mbar_init();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tbase = tmem_base_s;

    if (a_tmem) {
        const int row = warp * 32 + lane;
        const uint32_t lane_sel = (uint32_t)(warp * 32) << 16;
        for (int k0 = 0; k0 < K; k0 += 16) {
            uint32_t hi[8], lo[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) split_f16x2_sat(A[(size_t)row * K + k0 + 2 * j], A[(size_t)row * K + k0 + 2 * j + 1], hi[j], lo[j]);
            tmem_st8(tbase + lane_sel + col_a + (uint32_t)(k0 / 2), hi);
            tmem_st8(tbase + lane_sel + col_a + (uint32_t)(K / 2 + k0 / 2), lo);
        }
        tmem_st_wait();
        tc_fence_before();
        __syncthreads();
        tc_fence_after();
    }

    if (threadIdx.x == 0) {
        const uint32_t kstride = 128, gstride = (uint32_t)chunks * 128;
        const uint32_t lbo = (variant & 1) ? gstride : kstride, sbo = (variant & 1) ? kstride : gstride;
        const bool small_first = (variant & 2) != 0;       // correction passes before hi*hi
        const uint32_t idesc = make_idesc(tf32 ? FMT_TF32 : FMT_F16, 128, N) | (a_mn ? kIdescAMajorMN : 0u) | (b_mn ? kIdescBMajorMN : 0u);
        // MN-major: SBO = next 16 bytes of M / N (128 B apart), LBO = next 8 rows of K
        const uint32_t a_lbo = (uint32_t)(128 / epc) * 128, b_lbo = (uint32_t)(N / epc) * 128;
        const int ksteps = chunks / 2;
        const int npass = split ? 3 : 1;
        uint32_t acc = 0;
        for (int pp = 0; pp < npass; ++pp) {
            const int p = (split && small_first) ? (pp + 1) % 3 : pp;   // lo*hi, hi*lo, hi*hi
            const uint8_t* as = (p == 1) ? a_lo : a_hi;          // hi*hi, lo*hi, hi*lo
            const uint8_t* bs = (p == 2) ? b_lo : b_hi;
            for (int ks = 0; ks < ksteps; ++ks) {
                const uint32_t kk = 32 / elem / 8;                // 8-row K groups per UMMA (fp16: 2, tf32: 1)
                const uint64_t ad = a_mn ? make_smem_desc(smem_u32(as) + ks * kk * a_lbo, a_lbo, 128)
                                       : make_smem_desc(smem_u32(as) + ks * 2 * kstride, lbo, sbo);
                const uint64_t bd = b_mn ? make_smem_desc(smem_u32(bs) + ks * kk * b_lbo, b_lbo, 128)
                                       : make_smem_desc(smem_u32(bs) + ks * 2 * kstride, lbo, sbo);
                if (a_tmem) umma_f16_ts(tbase, tbase + col_a + (uint32_t)((p == 1) ? K / 2 : 0) + (uint32_t)ks * 8, bd, idesc, acc);
                else if (tf32) umma_tf32(tbase, ad, bd, idesc, acc);
                else umma_f16(tbase, ad, bd, idesc, acc);
                acc = 1;
            }
        }
        umma_commit(&bar);
    }
    mbar_wait(&bar, 0);
    tc_fence_after();

    const int row = warp * 32 + lane;
    for (int c0 = 0; c0 < N; c0 += 16) {
        float v[16];
        tmem_ld16(tbase + ((uint32_t)(warp * 32) << 16) + c0, v);
        tmem_ld_wait();
#pragma unroll
        for (int i = 0; i < 16; ++i) D[(size_t)row * N + c0 + i] = v[i];
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tbase, ncols);
}

}  // namespace stb

extern "C" int stb_tc_selftest(const float* A, const float* B, float* D, int32_t K, int32_t N, int32_t mode,
                               int32_t variant, void* stream) {
    using namespace stb;
    const int tf32 = mode & 1;
    if (mode < 0 || mode > 3) return set_error(STB_EINVAL, "mode must be 0..3");
    if ((variant & 16) && (tf32 || (variant & 4) || N + K > 480)) return set_error(STB_EINVAL, "TMEM-sourced A: fp16, K-major, N + K <= 480");
    if (K < (tf32 ? 8 : 16) || K % (tf32 ? 8 : 16) || N < 16 || N > 256 || N % 16)
        return set_error(STB_EINVAL, "K must be a multiple of the UMMA K, N a multiple of 16 <= 256");
    const size_t smem = (size_t)(128 + N) * K * (tf32 ? 4 : 2) * 2;
    if (smem > 200 * 1024) return set_error(STB_EINVAL, "operands too large for one CTA");
    cudaError_t e = cudaFuncSetAttribute(tc_selftest_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return set_error(STB_ECUDA, "cudaFuncSetAttribute: %s", cudaGetErrorString(e));
    tc_selftest_kernel<<<1, 128, smem, (cudaStream_t)stream>>>(A, B, D, K, N, mode, variant);
    count_launch();
    e = cudaGetLastError();
    if (e != cudaSuccess) return set_error(STB_ECUDA, "tc_selftest launch: %s", cudaGetErrorString(e));
    return STB_OK;
}
