// Thin inline-PTX layer for sm_100a: mbarrier, bulk (TMA) copies, tcgen05 MMA / TMEM.
//
// Operand layout used throughout the tcgen05 engine ("canonical K-major, no swizzle"):
// a [rows x K] bf16 operand is stored as [K/8][rows][8], i.e. 16-byte "core rows" of 8
// consecutive K elements, 8 of them (128 B) forming a core matrix.  In UMMA descriptor terms
//   SBO (stride between 8-row groups along M/N) = 128 B
//   LBO (stride between core matrices along K)  = rows * 16 B
// One tcgen05.mma (kind::f16) consumes K = 16, i.e. two K-core-matrices: advancing K by 16
// adds 2 * LBO to the start address.  The same layout is used in global memory, so a whole
// operand tile is one contiguous cp.async.bulk copy (no tensor map, no swizzle to mismatch).
#pragma once

#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_fp8.h>
#include <stdint.h>

namespace cf {
namespace ptx {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// ---------------------------------------------------------------- mbarrier
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.shared::cta.b64 st, [%0];\n\t}" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.expect_tx.shared::cta.b64 st, [%0], %1;\n\t}" ::"r"(smem_u32(bar)),
                 "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
// Non-blocking probe (try_wait may suspend the thread for a system-dependent time): use this
// when polling several barriers in turn.
__device__ __forceinline__ bool mbar_test_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    while (!mbar_try_wait(bar, parity)) {
    }
}

// ---------------------------------------------------------------- proxies / fences
// generic-proxy smem writes -> visible to the async proxy (UMMA operand reads, bulk copies)
__device__ __forceinline__ void fence_proxy_async_smem() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_before_sync() {
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after_sync() {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}

// ---------------------------------------------------------------- bulk copy (TMA, 1-D)
// global -> shared, completion signalled on an mbarrier as transaction bytes
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(smem_dst)),
                 "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

// L2 prefetch of a contiguous global range (no shared-memory destination, no completion event)
__device__ __forceinline__ void bulk_prefetch_l2(const void* gmem_src, uint32_t bytes) {
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(gmem_src), "r"(bytes) : "memory");
}

// ---------------------------------------------------------------- TMEM
template <int kCols>
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_result) {      // one full warp
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_result)),
                 "n"(kCols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template <int kCols>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr) {           // the same warp
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(kCols) : "memory");
}

// ---------------------------------------------------------------- UMMA descriptors
// Shared-memory matrix descriptor, K-major, SWIZZLE_NONE (see header comment).
__host__ __device__ constexpr uint64_t make_smem_desc(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);
    d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
    d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
    d |= (uint64_t)1 << 46;                       // descriptor version (sm_100)
    return d;                                     // base_offset 0, lbo_mode 0, layout SWIZZLE_NONE (0)
}

// Instruction descriptor: kind::f16, A = B = bf16 (K-major), D = f32, M x N tile.
__host__ __device__ constexpr uint32_t make_idesc_bf16(int m, int n) {
    return (1u << 4)                              // D format f32
           | (1u << 7)                            // A format bf16
           | (1u << 10)                           // B format bf16
           | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}

// kind::f16 with A = B = fp16; and kind::f8f6f4 with A = B = e5m2 (format code 1, like bf16 above).
__host__ __device__ constexpr uint32_t make_idesc_f16(int m, int n) {
    return (1u << 4) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}
__host__ __device__ constexpr uint32_t make_idesc_e5m2(int m, int n) { return make_idesc_bf16(m, n); }

// D[tmem] (+)= A[smem] * B[smem]; issued by ONE thread.
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}

// Warp-converged issue: every lane executes the statement, the instruction itself is predicated on
// `elected` (exactly one lane).  Keeps descriptor arithmetic on the uniform datapath instead of the
// per-lane "waterfall" loop the compiler emits around tcgen05.mma in divergent code.
__device__ __forceinline__ uint32_t elect_one() {
    uint32_t pred;
    asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
    return pred;
}
__device__ __forceinline__ void umma_bf16_pred(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                               uint32_t accumulate, uint32_t elected) {
    asm volatile(
        "{\n\t.reg .pred p, q;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "setp.ne.b32 q, %5, 0;\n\t"
        "@q tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate), "r"(elected)
        : "memory");
}
__device__ __forceinline__ void umma_bf16_ts_pred(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc,
                                                  uint32_t accumulate, uint32_t elected) {
    asm volatile(
        "{\n\t.reg .pred p, q;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "setp.ne.b32 q, %5, 0;\n\t"
        "@q tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}" ::"r"(tmem_d),
        "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate), "r"(elected)
        : "memory");
}
__device__ __forceinline__ void umma_commit_pred(uint64_t* bar, uint32_t elected) {
    asm volatile(
        "{\n\t.reg .pred q;\n\t"
        "setp.ne.b32 q, %1, 0;\n\t"
        "@q tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t}" ::"r"(smem_u32(bar)),
        "r"(elected)
        : "memory");
}

// kind::f8f6f4 (8-bit operands, K = 32 per instruction, byte-identical descriptors to a K = 16 bf16 MMA)
__device__ __forceinline__ void umma_f8_pred(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                             uint32_t accumulate, uint32_t elected) {
    asm volatile(
        "{\n\t.reg .pred p, q;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "setp.ne.b32 q, %5, 0;\n\t"
        "@q tcgen05.mma.cta_group::1.kind::f8f6f4 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate), "r"(elected)
        : "memory");
}
__device__ __forceinline__ void umma_f8_ts_pred(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc,
                                                uint32_t accumulate, uint32_t elected) {
    asm volatile(
        "{\n\t.reg .pred p, q;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "setp.ne.b32 q, %5, 0;\n\t"
        "@q tcgen05.mma.cta_group::1.kind::f8f6f4 [%0], [%1], %2, %3, p;\n\t}" ::"r"(tmem_d),
        "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate), "r"(elected)
        : "memory");
}

// Same with the A operand in tensor memory (".ts" form): A[128 x 16] bf16 occupies lanes 0..127
// and 8 consecutive 32-bit columns starting at `tmem_a`, two K elements per column (even k in the
// low half).
__device__ __forceinline__ void umma_bf16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}" ::"r"(tmem_d),
        "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}

// mbarrier arrives when all tcgen05.mma previously issued by this thread have completed
// (implies tcgen05.fence::before_thread_sync).
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// ---------------------------------------------------------------- TMEM <-> registers
// 32 lanes x 32-bit, 16 consecutive columns: thread i of the warp gets lane (base_lane + i).
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float* v) {
    uint32_t r[16];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr)
        : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}
// Issue only (no wait): pair with tmem_ld_wait() before using the values.
__device__ __forceinline__ void tmem_ld16_nowait(uint32_t taddr, uint32_t* r) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const float* v) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};" ::"r"(taddr),
        "r"(__float_as_uint(v[0])), "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])), "r"(__float_as_uint(v[3])),
        "r"(__float_as_uint(v[4])), "r"(__float_as_uint(v[5])), "r"(__float_as_uint(v[6])), "r"(__float_as_uint(v[7])),
        "r"(__float_as_uint(v[8])), "r"(__float_as_uint(v[9])), "r"(__float_as_uint(v[10])), "r"(__float_as_uint(v[11])),
        "r"(__float_as_uint(v[12])), "r"(__float_as_uint(v[13])), "r"(__float_as_uint(v[14])), "r"(__float_as_uint(v[15]))
        : "memory");
}
__device__ __forceinline__ void tmem_st8_u32(uint32_t taddr, const uint32_t* v) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"r"(taddr), "r"(v[0]), "r"(v[1]),
                 "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7])
                 : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// ---------------------------------------------------------------- packed fp32 pairs (FFMA2 / FADD2 / FMUL2)
// sm_100 executes two fp32 operations per lane in one instruction: half the issue slots for the
// epilogues' elementwise math (they are bound by instruction issue, not by the FMA pipe).
__device__ __forceinline__ uint64_t pack2(float2 a) {
    uint64_t r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(a.x), "f"(a.y));
    return r;
}
__device__ __forceinline__ float2 unpack2(uint64_t r) {
    float2 a;
    asm("mov.b64 {%0, %1}, %2;" : "=f"(a.x), "=f"(a.y) : "l"(r));
    return a;
}
__device__ __forceinline__ float2 ffma2(float2 a, float2 b, float2 c) {
    uint64_t d;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(pack2(a)), "l"(pack2(b)), "l"(pack2(c)));
    return unpack2(d);
}
__device__ __forceinline__ float2 fmul2(float2 a, float2 b) {
    uint64_t d;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(pack2(a)), "l"(pack2(b)));
    return unpack2(d);
}
__device__ __forceinline__ float2 fadd2(float2 a, float2 b) {
    uint64_t d;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(pack2(a)), "l"(pack2(b)));
    return unpack2(d);
}
__device__ __forceinline__ float2 splat2(float x) { return make_float2(x, x); }

// ---------------------------------------------------------------- split bf16 ("bf16x3")
// x ~= hi + lo with hi = bf16(x), lo = bf16(x - hi); a product a*b is evaluated as
// a_hi*b_hi + a_lo*b_hi + a_hi*b_lo with fp32 accumulation (error ~2^-16 relative).
__device__ __forceinline__ void split_bf16(float x, __nv_bfloat16& hi, __nv_bfloat16& lo) {
    hi = __float2bfloat16_rn(x);
    lo = __float2bfloat16_rn(x - __bfloat162float(hi));
}
// Pack two floats' hi parts and lo parts into bf16x2 words (element 0 in the low half).
// Uses the packed conversion (F2FP, FMA/ALU pipes) - the scalar F2F.BF16 runs on the XU pipe,
// which the GRU epilogue needs for its transcendentals.
__device__ __forceinline__ void split_bf16x2(float x0, float x1, uint32_t& hi, uint32_t& lo) {
    const __nv_bfloat162 h = __floats2bfloat162_rn(x0, x1);
    hi = *reinterpret_cast<const uint32_t*>(&h);
    const float2 r = ffma2(make_float2(__uint_as_float(hi << 16), __uint_as_float(hi & 0xffff0000u)), splat2(-1.f),
                           make_float2(x0, x1));                          // x - hi, both at once
    const __nv_bfloat162 l = __floats2bfloat162_rn(r.x, r.y);
    lo = *reinterpret_cast<const uint32_t*>(&l);
}

// ---------------------------------------------------------------- fp16 + e5m2 corrections ("f16e5")
// x = h + l with h = fp16(x) (11 significant bits) and l the exact remainder.  A product a*w is
// evaluated as  a_h*w_h  (one fp16 MMA)  +  [a_l*S | a_h/S] . [w_h/S ; w_l*S]  (one e5m2 MMA over the
// doubled K, at twice the 16-bit rate): the two correction terms are 2^-12 of the product, so the
// 3 significant bits of e5m2 keep the total near 2^-15; S = 2^6 puts both a_l*S (~2^-12 |a| S) and
// a_h/S into e5m2's normal range (>= 2^-14) for every |a| >= 2^-8 - smaller values only carry
// absolute errors below 2^-19 |w|.  Two pass-equivalents instead of the three of bf16x3.
//
// Storage form of an A operand ("compact": 3 bytes per value in HBM, 4 in shared / tensor memory):
//   main  m  = fp16(a_h / S)          - the fp16 MMA multiplies it with fp16(S w_h), so the scale cancels
//   lo byte  = e5m2(a_l * S)          - rounded to nearest
//   hi byte  = the TOP BYTE of m      - e5m2 has fp16's sign and exponent layout, so the upper byte of an fp16 IS
//                                       the e5m2 of the same value, truncated to two mantissa bits
// The hi bytes are a pure byte shuffle of the main plane (one PRMT per four values), so they are never
// stored in HBM: layer outputs travel as main + lo (3 B / value) and the consumer rebuilds the hi slab
// in shared memory.  Truncating instead of rounding that byte biases the a_h*w_l correction by at most
// 2^-3 of a 2^-12 term (emulated end to end: max |dp| 3.4e-5 vs 2.7e-5, tests/tools/precision_emulation.py).
constexpr float kCorrScale = 64.f;
// fp16 tops out at 65504 and the corrections need |a| >= 2^-8: the engine uses this format where the
// activations are GRU states in (-1, 1) (the 128-wide layers); the layer fed by the conv stack, whose
// activations span 2^-10 .. 60 (and 4.5e5 behind a full-scale spike), stays split bf16.  The fp16
// conversion saturates rather than produce infinities.
// Two values -> fp16x2 word of the down-scaled main parts (element 0 in the low half) and the
// e5m2x2 of the scaled remainders (element 0 in the low byte).
__device__ __forceinline__ void split_f16e5x2(float x0, float x1, uint32_t& main, uint32_t& lo) {
    uint32_t h32;
    asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(h32) : "f"(x1), "f"(x0));   // saturating: no infinities
    const __half2 m = __hmul2(*reinterpret_cast<const __half2*>(&h32), __floats2half2_rn(1.f / kCorrScale, 1.f / kCorrScale));
    main = *reinterpret_cast<const uint32_t*>(&m);
    // remainder against what the main plane really holds, a_h = S m (below 2^-8 the down-scaled value is an fp16
    // subnormal and loses bits; the remainder byte picks them up):  S (x - S m) = S x - S^2 m
    const float2 l = ffma2(__half22float2(m), splat2(-kCorrScale * kCorrScale), fmul2(make_float2(x0, x1), splat2(kCorrScale)));
    lo = __nv_cvt_float2_to_fp8x2(l, __NV_SATFINITE, __NV_E5M2);
}
// hi bytes of four consecutive values from their two main words
__device__ __forceinline__ uint32_t f16e5_hi4(uint32_t m01, uint32_t m23) { return __byte_perm(m01, m23, 0x7531); }
// 16 values (one K = 16 chunk of an operand row): 8 fp16x2 words + 16 remainder bytes + 16 hi bytes
__device__ __forceinline__ void split_f16e5_chunk(const float* v, uint32_t* main, uint32_t* lo4, uint32_t* hi4) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        uint32_t la, lb;
        split_f16e5x2(v[4 * j], v[4 * j + 1], main[2 * j], la);
        split_f16e5x2(v[4 * j + 2], v[4 * j + 3], main[2 * j + 1], lb);
        lo4[j] = la | (lb << 16);
        hi4[j] = f16e5_hi4(main[2 * j], main[2 * j + 1]);
    }
}

// ---------------------------------------------------------------- activations (MUFU)
__device__ __forceinline__ float ex2_approx(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float rcp_approx(float x) {
    float y;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float fast_sigmoid(float x) {
    // 1 / (1 + 2^(-x log2 e)): one ex2 + one rcp, relative error ~2^-22
    return rcp_approx(1.f + ex2_approx(-1.4426950408889634f * x));
}
__device__ __forceinline__ float fast_tanh(float x) {
    // (1 - e) / (1 + e), e = exp(-2|x|): no cancellation for large |x|, ~1e-7 absolute near 0
    const float e = ex2_approx(-2.8853900817779268f * fabsf(x));
    return copysignf((1.f - e) * rcp_approx(1.f + e), x);
}

// Four reciprocals from one MUFU.RCP: r = 1 / (a0 a1 a2 a3), then back-multiplication.
// Callers keep every a_i in [1, 5e8] so the product cannot overflow.
__device__ __forceinline__ void rcp4(const float* a, float* inv) {
    const float p01 = a[0] * a[1], p23 = a[2] * a[3];
    const float r = rcp_approx(p01 * p23);
    const float r01 = r * p23, r23 = r * p01;
    inv[0] = r01 * a[1];
    inv[1] = r01 * a[0];
    inv[2] = r23 * a[3];
    inv[3] = r23 * a[2];
}
// sigmoid of four values: 4 x ex2 + 1 x rcp.  The exponent is clamped at 20 (sigmoid(-20) = 2e-9),
// which bounds 1 + e^-x by 4.9e8 and the product of four by 5.7e34.
__device__ __forceinline__ void sigmoid4(const float* x, float* y) {
    float a[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) a[i] = 1.f + ex2_approx(fminf(-1.4426950408889634f * x[i], 28.853900817779268f));
    rcp4(a, y);
}
// tanh of four values: (1 - e) / (1 + e), e = exp(-2|x|) in (0, 1]; 4 x ex2 + 1 x rcp.
__device__ __forceinline__ void tanh4(const float* x, float* y) {
    float e[4], a[4], inv[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        e[i] = ex2_approx(-2.8853900817779268f * fabsf(x[i]));
        a[i] = 1.f + e[i];
    }
    rcp4(a, inv);
#pragma unroll
    for (int i = 0; i < 4; ++i) y[i] = copysignf((1.f - e[i]) * inv[i], x[i]);
}

// Exponent-domain variants for pre-activations that were already multiplied by -log2(e)
// (sigmoid) or by 2 log2(e) (tanh) when the weights were packed: one instruction less per value.
//   sigmoid(x) = 1 / (1 + 2^z),      z = -x log2 e
//   tanh(x)    = 1 - 2 / (1 + 2^z),  z = 2 x log2 e     (absolute error ~1e-7 near 0)
__device__ __forceinline__ float tanh_approx(float x) {
    float y;
    asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
// Fused "bias + activation" on exponent-domain accumulators: y = act(acc + b).
// With MUFU.TANH the bias add folds into the argument scaling (one FFMA): callers pass bk = b * k.
#ifndef CF_PRECISE_ACT
constexpr float kSigArgScale = -0.34657359027997264f;     // z * (-ln2 / 2): sigmoid(x) = 0.5 + 0.5 tanh(x / 2)
constexpr float kTanhArgScale = 0.34657359027997264f;      // z * ( ln2 / 2): tanh(x)
__device__ __forceinline__ float sigmoid_zb(float acc, float bk) { return fmaf(tanh_approx(fmaf(acc, kSigArgScale, bk)), 0.5f, 0.5f); }
__device__ __forceinline__ float tanh_zb(float acc, float bk) { return tanh_approx(fmaf(acc, kTanhArgScale, bk)); }
// two values at a time: packed argument / result arithmetic around the two MUFU.TANH
__device__ __forceinline__ float2 sigmoid_zb2(float2 acc, float2 bk) {
    const float2 z = ffma2(acc, splat2(kSigArgScale), bk);
    return ffma2(make_float2(tanh_approx(z.x), tanh_approx(z.y)), splat2(0.5f), splat2(0.5f));
}
__device__ __forceinline__ float2 tanh_zb2(float2 acc, float2 bk) {
    const float2 z = ffma2(acc, splat2(kTanhArgScale), bk);
    return make_float2(tanh_approx(z.x), tanh_approx(z.y));
}
#endif
#ifndef CF_PRECISE_ACT
// Default: MUFU.TANH based activations, one MUFU + one FMA-pipe instruction per gate value.
// Measured end to end on B200 (tools/accuracy_check.py, 240 000 positions, shipped weights):
// max |dp| 2.0e-5 - indistinguishable from the ex2/rcp formulation below (1.6e-5), both dominated
// by the split-bf16 operand error.  The chip runs this kernel at its power cap, so the ~30 % fewer
// epilogue instructions translate into ~4 % more throughput.  -DCF_PRECISE_ACT selects ex2 + rcp.
__device__ __forceinline__ void sigmoid4_z(const float* z, float* y) {
#pragma unroll
    for (int i = 0; i < 4; ++i) y[i] = fmaf(tanh_approx(z[i] * -0.34657359027997264f), 0.5f, 0.5f);
}
__device__ __forceinline__ void tanh4_z(const float* z, float* y) {
#pragma unroll
    for (int i = 0; i < 4; ++i) y[i] = tanh_approx(z[i] * 0.34657359027997264f);
}
#else
__device__ __forceinline__ void sigmoid4_z(const float* z, float* y) {
    float a[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) a[i] = 1.f + ex2_approx(fminf(z[i], 28.853900817779268f));
    rcp4(a, y);
}
__device__ __forceinline__ void tanh4_z(const float* z, float* y) {
    float a[4], inv[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) a[i] = 1.f + ex2_approx(fminf(z[i], 28.853900817779268f));
    rcp4(a, inv);
#pragma unroll
    for (int i = 0; i < 4; ++i) y[i] = fmaf(-2.f, inv[i], 1.f);
}
#endif

}  // namespace ptx
}  // namespace cf
