// Inline-PTX building blocks for the sm_100a kernels: mbarrier, TMA (cp.async.bulk.tensor), tcgen05 (MMA, TMEM
// alloc / ld / commit / fences) and the shared-memory / instruction descriptors of the UMMA unit.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace mt {
namespace sm100 {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ---- mbarrier --------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
// Bounded wait: a protocol bug must not hang the GPU.  try_wait suspends the warp in hardware for a time slice; the
// clock is consulted once per 4096 failed polls and the kernel traps after ~2 s, so a broken protocol surfaces as a
// launch error instead of a hung box.  The wait is inlined dozens of times per kernel and the persistent kernels run
// their item hand-over code once per item (cold in the instruction cache), so the slow path is kept to a few
// instructions: no printf, no argument set-up (compile with -DMT_DEBUG_WAIT to get the barrier address printed).
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  const long long t0 = clock64();
  uint32_t polls = 0;
#pragma unroll 1
  while (!mbar_try_wait(bar, parity)) {
    if ((++polls & 4095u) == 0 && clock64() - t0 > 4000000000ll) {
#ifdef MT_DEBUG_WAIT
      printf("modaltune_b200: mbarrier timeout (block %d thread %d bar %u parity %u)\n", blockIdx.x, threadIdx.x, bar,
             parity);
#endif
      __trap();
    }
  }
}

// ---- proxies / fences --------------------------------------------------------------------------------------------------
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// ---- TMA ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void tma_prefetch_desc(const void* desc) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(desc)) : "memory");
}
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const void* desc, uint32_t bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      :
      : "r"(dst), "l"(reinterpret_cast<uint64_t>(desc)), "r"(bar), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}

__device__ __forceinline__ void tma_load_4d(uint32_t dst, const void* desc, uint32_t bar, int c0, int c1, int c2,
                                            int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      :
      : "r"(dst), "l"(reinterpret_cast<uint64_t>(desc)), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}

__device__ __forceinline__ void tma_load_2d(uint32_t dst, const void* desc, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      :
      : "r"(dst), "l"(reinterpret_cast<uint64_t>(desc)), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}

// ---- CTA pairs (cta_group::2): two CTAs of a cluster execute one M = 256 MMA; operands are split across their shared
// memories, accumulators across their tensor memories.  Shared-memory addresses of barriers that BOTH CTAs signal
// refer to the even (leader) CTA: the peer bit of a shared::cluster address is bit 24.
static constexpr uint32_t kPeerBitMask = 0xFEFFFFFFu;
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// TMA load issued by either CTA of the pair; the transaction bytes are credited to the LEADER's mbarrier
__device__ __forceinline__ void tma_load_2d_pair(uint32_t dst, const void* desc, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      :
      : "r"(dst), "l"(reinterpret_cast<uint64_t>(desc)), "r"(bar & kPeerBitMask), "r"(c0), "r"(c1)
      : "memory");
}
// arrive on the leader CTA's barrier from either CTA of the pair
__device__ __forceinline__ void mbar_arrive_leader(uint32_t bar) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(bar & kPeerBitMask) : "memory");
}
__device__ __forceinline__ void tmem_alloc_pair(uint32_t dst_smem, uint32_t cols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(cols) : "memory");
}
__device__ __forceinline__ void tmem_relinquish_pair() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t addr, uint32_t cols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(addr), "r"(cols) : "memory");
}
// D[tmem of both CTAs] (+)= A[smem of both CTAs] * B[smem halves of both CTAs]; issued by ONE thread of the leader CTA
__device__ __forceinline__ void umma_ss_pair(uint32_t tmem_d, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      :
      : "r"(tmem_d), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// completion of the pair's MMAs -> the barrier at this offset in BOTH CTAs
__device__ __forceinline__ void umma_commit_pair(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(bar), "h"((uint16_t)3) : "memory");
}

// global[coords] += smem box (element-wise add in L2; the element type comes from the tensor map)
__device__ __forceinline__ void tma_reduce_add_3d(const void* desc, uint32_t src, int c0, int c1, int c2) {
  asm volatile("cp.reduce.async.bulk.tensor.3d.global.shared::cta.add.bulk_group [%0, {%2, %3, %4}], [%1];"
               :
               : "l"(reinterpret_cast<uint64_t>(desc)), "r"(src), "r"(c0), "r"(c1), "r"(c2)
               : "memory");
}
// smem box -> global[coords] (plain store; rows / columns outside the tensor are clipped)
__device__ __forceinline__ void tma_store_2d(const void* desc, uint32_t src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
               :
               : "l"(reinterpret_cast<uint64_t>(desc)), "r"(src), "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void bulk_commit_group() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_group_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
__device__ __forceinline__ void bulk_wait_group_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void named_bar_sync(int id, int threads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(threads) : "memory");
}

// ---- TMEM --------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t dst_smem, uint32_t cols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(cols) : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t addr, uint32_t cols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(addr), "r"(cols) : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// 32 lanes x 32 consecutive fp32 columns: thread i of the warp gets lane (base_lane + i), columns [col, col+32)
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float (&v)[32]) {
  uint32_t* r = reinterpret_cast<uint32_t*>(v);
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
}
// 32 lanes x 64 consecutive fp32 columns (half of a 128-column score row per thread)
__device__ __forceinline__ void tmem_ld64(uint32_t taddr, float* v) {
  uint32_t* r = reinterpret_cast<uint32_t*>(v);
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x64.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32, %33, %34, %35, %36, %37, %38, %39, %40, %41, %42, %43, %44, %45, %46, %47, %48, %49, %50, %51, %52, %53, %54, %55, %56, %57, %58, %59, %60, %61, %62, %63}, [%64];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31]), "=r"(r[32]), "=r"(r[33]), "=r"(r[34]), "=r"(r[35]), "=r"(r[36]), "=r"(r[37]), "=r"(r[38]), "=r"(r[39]), "=r"(r[40]), "=r"(r[41]), "=r"(r[42]), "=r"(r[43]), "=r"(r[44]), "=r"(r[45]), "=r"(r[46]), "=r"(r[47]), "=r"(r[48]), "=r"(r[49]), "=r"(r[50]), "=r"(r[51]), "=r"(r[52]), "=r"(r[53]), "=r"(r[54]), "=r"(r[55]), "=r"(r[56]), "=r"(r[57]), "=r"(r[58]), "=r"(r[59]), "=r"(r[60]), "=r"(r[61]), "=r"(r[62]), "=r"(r[63])
               : "r"(taddr)
               : "memory");
}
__device__ __forceinline__ float fmax3(float a, float b, float c) {
  float r;
  asm("max.f32 %0, %1, %2, %3;" : "=f"(r) : "f"(a), "f"(b), "f"(c));
  return r;
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float (&v)[16]) {
  uint32_t* r = reinterpret_cast<uint32_t*>(v);
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}

// 32 lanes x 16 consecutive 32-bit columns, registers -> TMEM (thread i of the warp writes lane base_lane + i)
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
      :
      : "r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]),
        "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}

__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t (&r)[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};"
               :
               : "r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
               : "memory");
}
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, float (&v)[8]) {
  uint32_t* r = reinterpret_cast<uint32_t*>(v);
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr)
               : "memory");
}
__device__ __forceinline__ void tmem_ld4(uint32_t taddr, float (&v)[4]) {
  uint32_t* r = reinterpret_cast<uint32_t*>(v);
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
               : "r"(taddr)
               : "memory");
}
__device__ __forceinline__ void red_add_v4(float* addr, float a, float b, float c, float d) {
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(addr), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}

// ---- UMMA --------------------------------------------------------------------------------------------------------------
// shared-memory matrix descriptor (cute::UMMA::SmemDescriptor): start address, leading / stride byte offsets (>>4),
// version = 1 (Blackwell), layout type 2 = SWIZZLE_128B.
__device__ __forceinline__ uint64_t umma_smem_desc(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;  // version
  d |= (uint64_t)2 << 61;  // SWIZZLE_128B
  return d;
}
// instruction descriptor for kind::f16 with bf16 A/B and fp32 accumulate (cute::UMMA::InstrDescriptor)
__host__ __device__ constexpr uint32_t umma_idesc_bf16(int M, int N, int a_mn_major, int b_mn_major) {
  return (1u << 4)                        // c_format = F32
         | (1u << 7)                      // a_format = BF16
         | (1u << 10)                     // b_format = BF16
         | ((uint32_t)a_mn_major << 15)   // 0 = K-major
         | ((uint32_t)b_mn_major << 16)
         | ((uint32_t)(N >> 3) << 17)
         | ((uint32_t)(M >> 4) << 24);
}
// D[tmem] (+)= A[smem] * B[smem]; issued by ONE thread on behalf of the CTA
__device__ __forceinline__ void umma_ss(uint32_t tmem_d, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      :
      : "r"(tmem_d), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// D[tmem] (+)= A[tmem] * B[smem]
__device__ __forceinline__ void umma_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
      :
      : "r"(tmem_d), "r"(tmem_a), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// One elected lane of a fully converged warp.  The compiler knows exactly one thread passes an elect.sync predicate
// and emits the UTCHMMA stream without the per-instruction serialisation loop it needs for `lane == 0`.
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
  return pred != 0;
}
// advance a shared-memory matrix descriptor by a byte offset (start-address field, 16-byte units)
__device__ __forceinline__ uint64_t umma_desc_adv(uint64_t desc, uint32_t bytes) { return desc + (uint64_t)(bytes >> 4); }

// make an mbarrier track the completion of every tcgen05 operation issued so far by this thread
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}

__device__ __forceinline__ float ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// 2^x on the FMA / ALU pipes (Cody-Waite split + degree-3 minimax polynomial on [-0.5, 0.5], relative error 7.5e-5,
// below the bf16 rounding of the probabilities it feeds): takes part of the exponentials off the 16 / clk MUFU unit,
// which bounds the forward kernel at head_dim 48.  x is clamped to >= -125 (result >= 2^-125, never a denormal).
__device__ __forceinline__ float ex2_poly(float x) {
  x = fmaxf(x, -125.f);
  const float t = x + 12582912.f;             // 1.5 * 2^23: the integer part lands in the low mantissa bits
  const float f = x - (t - 12582912.f);       // fraction in [-0.5, 0.5]
  float p = fmaf(f, 0x1.c3f76p-5f, 0x1.f0de1ap-3f);
  p = fmaf(p, f, 0x1.62f31ap-1f);
  p = fmaf(p, f, 0x1.fff692p-1f);
  return __uint_as_float(__float_as_uint(p) + (__float_as_uint(t) << 23));   // p * 2^n through the exponent field
}
// two fp32 FMAs / adds in one instruction (FFMA2 / FADD2, sm_100): halves the issue slots of element-wise fp32 loops
__device__ __forceinline__ float2 ffma2(float2 a, float2 b, float2 c) {
  uint64_t ra = *reinterpret_cast<uint64_t*>(&a), rb = *reinterpret_cast<uint64_t*>(&b);
  uint64_t rc = *reinterpret_cast<uint64_t*>(&c), rd;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(rd) : "l"(ra), "l"(rb), "l"(rc));
  return *reinterpret_cast<float2*>(&rd);
}
__device__ __forceinline__ float2 fadd2(float2 a, float2 b) {
  uint64_t ra = *reinterpret_cast<uint64_t*>(&a), rb = *reinterpret_cast<uint64_t*>(&b), rd;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(rd) : "l"(ra), "l"(rb));
  return *reinterpret_cast<float2*>(&rd);
}
__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}

}  // namespace sm100
}  // namespace mt
