// sm_100a building blocks used by the tensor-core path: mbarrier, bulk async copy (TMA
// engine, 1-D), tcgen05 (TMEM allocation, UMMA issue / commit, TMEM loads), the shared-
// memory matrix descriptors, named barriers, MUFU-based exp2 / division and the precision
// splits.  Everything is inline PTX; nothing here exists on older parts.
//
// Operand layout (both A and B are K-major, SWIZZLE_NONE "interleaved" canonical layout):
// a matrix of R rows x K elements is stored as 8-row x 16-byte core matrices,
//     byte(r, k) = (r / 8) * SBO + (k_chunk) * LBO + (r % 8) * 16 + (k % EPC) * sizeof(elem)
// with EPC = 16 / sizeof(elem) elements per chunk, k_chunk = k / EPC, LBO = 128 (the K-
// adjacent core matrix follows immediately) and SBO = (K / EPC) * 128 (next 8-row group).
// One UMMA consumes 32 bytes of K (2 chunks): fp16 K=16, tf32 K=8.
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

namespace stb {
namespace tc {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// ---- mbarrier ---------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
// try_wait with a suspend-time hint: the thread sleeps in hardware until the phase flips or the
// hint (ns) expires, instead of burning issue slots that the epilogue warps of the same SM
// sub-partition need (ncu: the retry loops were 15 % of all issued instructions before this).
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity), "r"(1000000u)
        : "memory");
    return ok != 0;
}
// Bounded wait: a protocol bug traps (launch fails with an error) instead of hanging the GPU.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    uint32_t spins = 0;
    while (!mbar_try_wait(bar, parity)) {
        if (++spins > (1u << 26)) {
            if ((threadIdx.x & 31) == 0)
                printf("stribor_b200: mbarrier wait timed out (block %d thread %d smem 0x%x parity %u)\n",
                       (int)blockIdx.x, (int)threadIdx.x, smem_u32(bar), parity);
            __trap();
        }
    }
}
// the same on a pre-converted shared-memory address (hot loops: saves the generic -> shared
// conversion, which ptxas otherwise rematerialises at every use)
__device__ __forceinline__ void mbar_arrive_a(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait_a(uint32_t bar, uint32_t parity) {
    uint32_t spins = 0;
    for (;;) {
        uint32_t ok;
        asm volatile(
            "{\n"
            ".reg .pred p;\n"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n"
            "selp.u32 %0, 1, 0, p;\n"
            "}\n"
            : "=r"(ok)
            : "r"(bar), "r"(parity), "r"(1000000u)
            : "memory");
        if (ok) break;
        if (++spins > (1u << 26)) {
            printf("stribor_b200: mbarrier wait timed out (block %d thread %d bar %u parity %u)\n", (int)blockIdx.x,
                   (int)threadIdx.x, bar, parity);
            __trap();
        }
    }
}
// keep a loop-invariant value in its register (ptxas otherwise recomputes index arithmetic from
// threadIdx in every iteration of the hot loop)
__device__ __forceinline__ uint32_t pin(uint32_t v) {
    asm volatile("" : "+r"(v));
    return v;
}

// wait with a sleep between polls: for epilogue warps whose wait is long by construction (the other warp
// group's turn, a product group in flight) -- a tight try_wait loop was 17 % of all issued instructions of
// the training kernel, taken from the warps doing arithmetic on the same scheduler
__device__ __forceinline__ void mbar_wait_sleep(uint64_t* bar, uint32_t parity, uint32_t ns) {
    uint32_t spins = 0;
    while (!mbar_try_wait(bar, parity)) {
        __nanosleep(ns);
        if (++spins > (1u << 26)) {
            if ((threadIdx.x & 31) == 0)
                printf("stribor_b200: mbarrier wait timed out (block %d thread %d smem 0x%x parity %u)\n",
                       (int)blockIdx.x, (int)threadIdx.x, smem_u32(bar), parity);
            __trap();
        }
    }
}

// same, for single-lane roles that can afford to back off (producer / issuer)
__device__ __forceinline__ void mbar_wait_relaxed(uint64_t* bar, uint32_t parity) {
    uint32_t spins = 0;
    while (!mbar_try_wait(bar, parity)) {
        __nanosleep(256);
        if (++spins > (1u << 26)) {
            if ((threadIdx.x & 31) == 0)
                printf("stribor_b200: mbarrier wait timed out (block %d thread %d smem 0x%x parity %u)\n",
                       (int)blockIdx.x, (int)threadIdx.x, smem_u32(bar), parity);
            __trap();
        }
    }
}

// ---- proxies / fences -------------------------------------------------------------------------
__device__ __forceinline__ void fence_proxy_async_smem() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_before() {
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}

// ---- 1-D bulk copy global -> shared, completion on an mbarrier (UBLKCP) ------------------------
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
            smem_u32(smem_dst)),
        "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar))
        : "memory");
}

// ---- TMEM ------------------------------------------------------------------------------------------
// one full warp; writes the TMEM base address to *dst (shared memory)
__device__ __forceinline__ void tmem_alloc(uint32_t* dst, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst)),
                 "r"(ncols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}

// 16 consecutive fp32 columns of this thread's TMEM lane (lane = 32 * (warp % 4) + laneid)
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float* v) {
    uint32_t r[16];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr)
        : "memory");
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}
// 8 consecutive fp32 columns
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, float* v) {
    uint32_t r[8];
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(taddr)
                 : "memory");
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// 8 consecutive 32-bit columns of this thread's TMEM lane <- registers (the A operand of a TMEM-sourced UMMA:
// two 16-bit K elements per column, K-major)
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t* r) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr), "r"(r[0]),
                 "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
                 : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// ---- UMMA -------------------------------------------------------------------------------------------
// shared-memory matrix descriptor, K-major, no swizzle (see header comment)
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);            // start address        bits [ 0,14)
    d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;      // leading byte offset  bits [16,30)
    d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;      // stride byte offset   bits [32,46)
    d |= (uint64_t)1 << 46;                                // descriptor version 1 (sm_100)
    return d;                                              // base offset 0, SWIZZLE_NONE
}

// instruction descriptor: fp32 accumulate, A and B K-major, dense
enum { FMT_F16 = 0, FMT_BF16 = 1, FMT_TF32 = 2 };
__host__ __device__ constexpr uint32_t make_idesc(int fmt, int M, int N) {
    return (1u << 4) | ((uint32_t)fmt << 7) | ((uint32_t)fmt << 10) | ((uint32_t)(N >> 3) << 17) |
           ((uint32_t)(M >> 4) << 24);
}

// MN-major operands (the K-major core-matrix buffer of the TRANSPOSED matrix, consumed in place):
// canonical no-swizzle form ((T,1,m),(8,k)):((1,T,SBO),(1T,LBO)) -- SBO = stride between 16-byte groups
// along M / N, LBO = stride between 8-row groups along K
constexpr uint32_t kIdescAMajorMN = 1u << 15;
constexpr uint32_t kIdescBMajorMN = 1u << 16;

// D[tmem] (+)= A[smem] * B[smem]^T ; issued by ONE thread
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                         uint32_t accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// the same with the A operand read from TMEM ([128 lanes x K/2 columns], written with tmem_st8): the activations of
// one GEMM feed the next without a shared-memory round trip (no st.shared, no generic->async proxy fence)
__device__ __forceinline__ void umma_f16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc,
                                            uint32_t accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n"
        "}\n" ::"r"(tmem_d),
        "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                          uint32_t accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// arrive on an mbarrier once every UMMA issued so far by this thread has completed
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(
                     smem_u32(bar))
                 : "memory");
}

// ---- arithmetic ---------------------------------------------------------------------------------
__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}
// exp through ex2.approx.  In the spline softmaxes, with the maximum subtracted, the arguments are <= 0, so the absolute
// error of every term is <= ~2.5 ulp of the LARGEST term (= 1), i.e. the same absolute accuracy on
// the bin sizes as a 2-ulp expf.  Measured on the GPU against the fp64 oracle
// (profiles/r01_tc_accuracy.txt): accurate expf, IEEE division and a true e_i / sum quotient change
// the mean log-det error by < 7 %; only compensated cumulative sums help (12 %) and cost ~90
// instructions per element.
__device__ __forceinline__ float ex2_approx(float v) {
    float r;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(v));
    return r;
}

// a / b to ~1 ulp: MUFU.RCP + one residual correction (4 instructions instead of ~10 for the
// IEEE sequence; the operands here are never subnormal / huge)
__device__ __forceinline__ float fdiv(float a, float b) {
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(b));
    const float q = a * r;
    return fmaf(fmaf(-q, b, a), r, q);
}

// ---- precision splits -----------------------------------------------------------------------------
__device__ __forceinline__ float to_tf32_rna(float v) {
    uint32_t r;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(v));
    return __uint_as_float(r);
}
// v ~= hi + lo with hi, lo exactly representable in tf32
__device__ __forceinline__ void split_tf32(float v, float& hi, float& lo) {
    hi = to_tf32_rna(v);
    lo = to_tf32_rna(v - hi);
}
// v == b0 + b1 + b2 exactly (3 x 8 significant bits), each part bf16: fp32 range, so no
// restriction on |v|
__device__ __forceinline__ void split_bf16x3(float v, __nv_bfloat16& b0, __nv_bfloat16& b1, __nv_bfloat16& b2) {
    b0 = __float2bfloat16_rn(v);
    const float r1 = v - __bfloat162float(b0);
    b1 = __float2bfloat16_rn(r1);
    b2 = __float2bfloat16_rn(r1 - __bfloat162float(b1));
}
// two values -> packed fp16 hi | lo, saturating (F2FP.SATFINITE.PACK_AB: one instruction per pair and part)
__device__ __forceinline__ void split_f16x2_sat(float a, float b, uint32_t& hi, uint32_t& lo) {
    asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(hi) : "f"(b), "f"(a));
    const __half2 h = *reinterpret_cast<const __half2*>(&hi);
    const float ra = a - __low2float(h), rb = b - __high2float(h);
    asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(lo) : "f"(rb), "f"(ra));
}
// v ~= hi + lo with hi, lo fp16 (|v| <= ~6e4; lo lands in the subnormal range for |v| < 0.25,
// where its absolute resolution 2^-25 is still below fp32's for O(1) accumulations)
__device__ __forceinline__ void split_f16(float v, __half& hi, __half& lo) {
    hi = __float2half_rn(v);
    lo = __float2half_rn(v - __half2float(hi));
}

}  // namespace tc
}  // namespace stb
