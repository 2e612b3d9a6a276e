// smz_tc_ptx.cuh — PTX wrappers shared by the tensor-core network-step kernels (smz_net_bf16.cu, smz_net_tc32.cu):
// mbarriers, bulk (TMA) copies, proxy / tcgen05 fences, UMMA shared-memory descriptors, the tensor-memory-A form of
// tcgen05.mma, TMEM allocation, tcgen05.commit, the tcgen05.ld / tcgen05.st shapes the epilogues use, and the head-layer reductions (softmax expectation over the categorical
// support, muzero_model.py:575-591).
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdio.h>

namespace smz_tc {

// ---------------------------------------------------------------------------------------------
// PTX wrappers
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned s32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(unsigned long long* bar, unsigned count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(s32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long* bar, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(s32(bar)), "r"(bytes) : "memory");
}
// bounded wait: a protocol error becomes a trap (CUDA error), never a hung GPU
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, unsigned parity) {
  const unsigned addr = s32(bar);
#pragma unroll 1
  for (unsigned spin = 0; spin < (1u << 26); ++spin) {
    unsigned ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(addr), "r"(parity)
        : "memory");
    if (ok) return;
  }
  printf("smz bf16: mbarrier wait timed out (block %d thread %d)\n", blockIdx.x, threadIdx.x);
  __trap();
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, unsigned bytes, unsigned long long* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(s32(dst)),
               "l"(src), "r"(bytes), "r"(s32(bar))
               : "memory");
}
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ unsigned long long umma_desc(unsigned smem_addr, unsigned lbo_bytes, unsigned sbo_bytes) {
  // SmemDescriptor (cute/arch/mma_sm100_desc.hpp): start>>4 [0,14), LBO>>4 [16,30), SBO>>4 [32,46),
  // version=1 [46,48), layout_type SWIZZLE_NONE=0 [61,64)
  return (unsigned long long)((smem_addr & 0x3FFFFu) >> 4) | ((unsigned long long)(lbo_bytes >> 4) << 16) |
         ((unsigned long long)(sbo_bytes >> 4) << 32) | (1ull << 46);
}

// one lane of a converged warp, chosen by the hardware (elect.sync): ptxas keeps operands of the elected region in
// uniform registers instead of wrapping every tcgen05.mma into an ELECT / R2UR.BROADCAST loop
__device__ __forceinline__ bool elect_one() {
  unsigned pred;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(pred));
  return pred != 0;
}
// tcgen05.mma kind::f16 with A read from tensor memory ("TS"): tmem_a = column (and lane 0) of the operand, which holds
// row m of A in the lane of accumulator row m and two bf16 per 32-bit column (K index 2j in the low half of column j),
// so a K = 16 step advances tmem_a by 8 columns.  B stays a shared-memory descriptor.
__device__ __forceinline__ void umma_ts(unsigned tmem_d, unsigned tmem_a, unsigned long long bdesc, unsigned idesc, unsigned accum) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}" ::"r"(tmem_d),
      "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accum)
      : "memory");
}
// whole warp: ncols TMEM columns, their address written to *base in shared memory; then give up the allocation permit
__device__ __forceinline__ void tmem_alloc(unsigned* base, unsigned ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(s32(base)), "r"(ncols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(unsigned base, unsigned ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(base), "r"(ncols) : "memory");
}
__device__ __forceinline__ void umma_commit(unsigned long long* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(s32(bar)) : "memory");
}
// 32 lanes x 32 consecutive fp32 columns -> 32 registers per thread (thread t <-> lane base+t)
__device__ __forceinline__ void tmem_ld32(unsigned taddr, float* v) {
  unsigned r[32];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}

// 32 lanes x 16 columns, no wait (pair with tmem_wait_ld)
__device__ __forceinline__ void tmem_ld16_nowait(unsigned taddr, unsigned* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

__device__ __forceinline__ unsigned pack_bf16(float lo, float hi) {
  __nv_bfloat162 p = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<unsigned*>(&p);
}

__device__ __forceinline__ float ex2f(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// partial softmax-expectation over this thread's 32 logits (columns col0..col0+31 of an S-wide head):
// running max m, z = sum e^(x-m), y = sum (c - S/2) e^(x-m)
struct SoftPart { float m, z, y; };
// Padded columns (>= S) need no predicate: their bias is -1e30 in the weight image, so e == 0.
__device__ __forceinline__ SoftPart soft_part(const float* x, int col0, int S) {
  SoftPart p{-1e30f, 0.f, 0.f};
#pragma unroll
  for (int i = 0; i < 32; ++i) p.m = fmaxf(p.m, x[i]);
  const float base = (float)(col0 - S / 2);
#pragma unroll
  for (int i = 0; i < 32; ++i) {
    const float e = ex2f((x[i] - p.m) * 1.4426950408889634f);
    p.z += e;
    p.y = fmaf(base + (float)i, e, p.y);
  }
  return p;
}
// inverse_transform_with_support (muzero_model.py:575-591) from the two halves' partials
__device__ __forceinline__ float support_scalar(SoftPart a, SoftPart b) {
  const float m = fmaxf(a.m, b.m);
  const float sa = ex2f((a.m - m) * 1.4426950408889634f);     // a fully padded half has z == y == 0
  const float sb = ex2f((b.m - m) * 1.4426950408889634f);
  const float y = (a.y * sa + b.y * sb) / (a.z * sa + b.z * sb);
  const float inner = __fadd_rn(1.f, __fmul_rn(0.004f, __fadd_rn(__fadd_rn(fabsf(y), 1.f), 0.001f)));
  const float t = __fdiv_rn(__fsub_rn(__fsqrt_rn(inner), 1.f), 0.002f);
  const float mag = __fsub_rn(__fmul_rn(t, t), 1.f);
  return y > 0.f ? mag : (y < 0.f ? -mag : 0.f);
}

__device__ __forceinline__ void tmem_ld8_nowait(unsigned taddr, unsigned* r) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr)
               : "memory");
}

// 16 lanes x (8 * X) columns: 4 * X registers per thread, group g = regs 4g..4g+3 = {row t/4: cols 2(t%4), +1; row t/4+8: same}
__device__ __forceinline__ void tmem_ld16x256_x2(unsigned taddr, unsigned* r) {
  asm volatile("tcgen05.ld.sync.aligned.16x256b.x2.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr)
               : "memory");
}
__device__ __forceinline__ void tmem_ld16x256_x1(unsigned taddr, unsigned* r) {
  asm volatile("tcgen05.ld.sync.aligned.16x256b.x1.b32 {%0, %1, %2, %3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
               : "r"(taddr)
               : "memory");
}
__device__ __forceinline__ void tmem_ld16x256_x4(unsigned taddr, unsigned* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.16x256b.x4.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}

// 16 lanes x (4 * X) columns, the store-side twin of the 16x256b fragment above for packed bf16 pairs: repetition i
// writes r[2i] to lane t/4 and r[2i+1] to lane t/4 + 8, column 4i + t%4 (probe in tools/microbench/a_operand_handoff.cu,
// result in profiles/r3_a_operand_handoff.txt).
// No wait: pair with tmem_wait_st before the hand-off to the MMA issuer.
__device__ __forceinline__ void tmem_st16x128_x1(unsigned taddr, unsigned r0, unsigned r1) {
  asm volatile("tcgen05.st.sync.aligned.16x128b.x1.b32 [%0], {%1, %2};" ::"r"(taddr), "r"(r0), "r"(r1) : "memory");
}
__device__ __forceinline__ void tmem_st16x128_x2(unsigned taddr, const unsigned* r) {
  asm volatile("tcgen05.st.sync.aligned.16x128b.x2.b32 [%0], {%1, %2, %3, %4};" ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]),
               "r"(r[3])
               : "memory");
}
__device__ __forceinline__ void tmem_st16x128_x4(unsigned taddr, const unsigned* r) {
  asm volatile("tcgen05.st.sync.aligned.16x128b.x4.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr), "r"(r[0]), "r"(r[1]),
               "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
               : "memory");
}
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

__device__ __forceinline__ SoftPart soft_merge(SoftPart a, SoftPart b) {
  const float m = fmaxf(a.m, b.m);
  const float sa = ex2f((a.m - m) * 1.4426950408889634f), sb = ex2f((b.m - m) * 1.4426950408889634f);
  return SoftPart{m, a.z * sa + b.z * sb, a.y * sa + b.y * sb};
}
__device__ __forceinline__ SoftPart soft_quad(SoftPart p) {    // merge over the 4 lanes that share a row
#pragma unroll
  for (int off = 1; off <= 2; off <<= 1) {
    SoftPart o{__shfl_xor_sync(0xffffffffu, p.m, off), __shfl_xor_sync(0xffffffffu, p.z, off), __shfl_xor_sync(0xffffffffu, p.y, off)};
    p = soft_merge(p, o);
  }
  return p;
}

}  // namespace smz_tc
