// tc_prims.cuh -- sm_100a primitives used by the tensor-core kernels: mbarrier, TMA (cp.async.bulk.tensor), tcgen05
// (alloc / mma / commit / ld / st / fences) and UMMA descriptors.  Inline PTX only; no CUTLASS dependency.
// Bit layouts follow cute/arch/mma_sm100_desc.hpp (SmemDescriptor, InstrDescriptor) of the vendored CUTLASS tree.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <stdint.h>

namespace tc {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ bool elect_one() {
  uint32_t pred = 0;
  asm volatile(
      "{\n\t.reg .pred P;\n\telect.sync _|P, 0xffffffff;\n\tselp.u32 %0, 1, 0, P;\n\t}\n"
      : "=r"(pred));
  return pred != 0;
}

// ---- mbarrier -------------------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred P;\n\tmbarrier.try_wait.parity.shared::cta.b64 P, [%1], %2;\n\tselp.u32 %0, 1, 0, P;\n\t}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// Bounded spin: a kernel bug must surface as a trap (reported by the next CUDA call), never as a hung GPU.  The report is out of
// line: the wait is inlined at dozens of sites of latency-bound kernels whose code should stay small.
static __device__ __noinline__ void mbar_timeout(uint64_t* bar, uint32_t parity) {
  printf("fql_b200: mbarrier timeout (block %d thread %d bar %p parity %u)\n", blockIdx.x, threadIdx.x, (void*)bar, parity);
  __trap();
}
// The same bounded wait with the spin loop INSIDE the asm block, for warps whose 32 lanes run a single-thread role's loop together
// (TMA producer, MMA issuer): a C++ loop with a per-lane exit makes every value carried around it "possibly divergent" to the
// compiler, and each tcgen05.mma / tcgen05.commit / TMA behind it is then wrapped in an ELECT + R2UR.BROADCAST waterfall.
__device__ __forceinline__ void mbar_wait_u(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t.reg .pred P1, P2;\n\t.reg .u32 c;\n\tmov.u32 c, 0;\n"
      "W_LOOP:\n\tmbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n\t@P1 bra W_DONE;\n\t"
      "add.u32 c, c, 1;\n\tsetp.lt.u32 P2, c, 0x4000000;\n\t@P2 bra W_LOOP;\n\ttrap;\n"
      "W_DONE:\n\t}\n" ::"r"(smem_u32(bar)), "r"(parity)
      : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if (++spins > (1u << 26)) mbar_timeout(bar, parity);
  }
}

// ---- thread-block cluster ----------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire;" ::: "memory");
}
// mbar_wait_u for a barrier that takes arrivals from other CTAs of the cluster (acquire at cluster scope)
__device__ __forceinline__ void mbar_wait_cluster_u(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t.reg .pred P1, P2;\n\t.reg .u32 c;\n\tmov.u32 c, 0;\n"
      "WC_LOOP:\n\tmbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 P1, [%0], %1;\n\t@P1 bra WC_DONE;\n\t"
      "add.u32 c, c, 1;\n\tsetp.lt.u32 P2, c, 0x4000000;\n\t@P2 bra WC_LOOP;\n\ttrap;\n"
      "WC_DONE:\n\t}\n" ::"r"(smem_u32(bar)), "r"(parity)
      : "memory");
}

// ---- TMA --------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
// pull one box of a tiled tensor into L2 (no smem destination, no completion)
__device__ __forceinline__ void tma_prefetch_2d(const CUtensorMap* m, int c0, int c1) {
  asm volatile("cp.async.bulk.prefetch.tensor.2d.L2.global.tile [%0, {%1, %2}];" ::"l"(reinterpret_cast<uint64_t>(m)), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
// generic-proxy smem writes -> visible to the async proxy (UMMA / TMA reads of smem)
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// ---- tcgen05 ------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t cols) {  // one full warp
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(cols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t cols) {  // the allocating warp
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
// D[tmem] (+)= A[smem] * B[smem]; issued by ONE thread
__device__ __forceinline__ void umma_bf16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Four consecutive k-steps (one 64-wide K block) from ONE asm block: the descriptors advance by constant adds inside PTX, so
// ptxas materialises the uniform-register operands once instead of an R2UR round trip before every UTCHMMA.
__device__ __forceinline__ void umma_bf16_x4(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint64_t a_step, uint64_t b_step,
                                             uint32_t idesc, uint32_t accumulate_first) {
  asm volatile(
      "{\n\t.reg .pred p, q;\n\t.reg .b64 a1, a2, a3, b1, b2, b3;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "setp.eq.b32 q, 0, 0;\n\t"
      "add.u64 a1, %1, %5;\n\tadd.u64 b1, %2, %6;\n\t"
      "add.u64 a2, a1, %5;\n\tadd.u64 b2, b1, %6;\n\t"
      "add.u64 a3, a2, %5;\n\tadd.u64 b3, b2, %6;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], a1, b1, %3, q;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], a2, b2, %3, q;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], a3, b3, %3, q;\n\t}\n"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate_first), "l"(a_step), "l"(b_step)
      : "memory");
}
// Two consecutive k-steps (one 32-wide K sub-block), same idea.
__device__ __forceinline__ void umma_bf16_x2(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint64_t a_step, uint64_t b_step,
                                             uint32_t idesc, uint32_t accumulate_first) {
  asm volatile(
      "{\n\t.reg .pred p, q;\n\t.reg .b64 a1, b1;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "setp.eq.b32 q, 0, 0;\n\t"
      "add.u64 a1, %1, %5;\n\tadd.u64 b1, %2, %6;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], a1, b1, %3, q;\n\t}\n"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate_first), "l"(a_step), "l"(b_step)
      : "memory");
}
// arrive on an mbarrier when all previously issued tcgen05.mma of this thread have completed (implies fence::before)
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// 32 lanes x 32 columns of 32 bit: thread i of the warp gets columns [c, c+32) of TMEM lane (lane_base + i)
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
        "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]),
        "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
        "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
        "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]), "r"(r[18]), "r"(r[19]),
        "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]), "r"(r[28]), "r"(r[29]),
        "r"(r[30]), "r"(r[31])
      : "memory");
}
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// ---- descriptors ------------------------------------------------------------------------------------------------
// Shared-memory matrix descriptor, SWIZZLE_128B, version 1 (sm_100).  lbo/sbo in bytes.
//   K-major  operand ([rows][64 bf16] tiles, 128 B rows, 8-row swizzle atoms): sbo = 1024 (next 8 rows), lbo unused (=16)
//   MN-major operand ([k][64 bf16] tiles, 128 B rows):  lbo = bytes between consecutive 64-element MN chunks,
//                                                       sbo = 1024 (next 8 k-rows)
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr, uint32_t lbo, uint32_t sbo) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3FFF);
  d |= (uint64_t)((lbo >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;  // version = 1
  d |= (uint64_t)2 << 61;  // SWIZZLE_128B
  return d;
}
// Same for a K-major tile of 64-byte rows ([rows][32] bf16) in the SWIZZLE_64B layout (8-row groups sbo bytes apart).
__device__ __forceinline__ uint64_t make_smem_desc_sw64(uint32_t saddr, uint32_t lbo, uint32_t sbo) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3FFF);
  d |= (uint64_t)((lbo >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;  // version = 1
  d |= (uint64_t)4 << 61;  // SWIZZLE_64B
  return d;
}
// Instruction descriptor for kind::f16 with bf16 operands, fp32 accumulate.  a_mn / b_mn: operand is MN-major.
__host__ __device__ constexpr uint32_t make_idesc_bf16(uint32_t M, uint32_t N, bool a_mn, bool b_mn) {
  return (1u << 4)                      // c_format  = F32
         | (1u << 7)                    // a_format  = BF16
         | (1u << 10)                   // b_format  = BF16
         | ((a_mn ? 1u : 0u) << 15)     // a_major
         | ((b_mn ? 1u : 0u) << 16)     // b_major
         | ((N >> 3) << 17)             // n_dim
         | ((M >> 4) << 24);            // m_dim
}

// Byte offset of the 16-byte chunk (row r, chunk c of 8) inside a [rows][128 B] SWIZZLE_128B tile whose base is 1024-aligned.
__device__ __forceinline__ uint32_t sw128_off(uint32_t r, uint32_t c) { return r * 128u + ((c ^ (r & 7u)) << 4); }

__device__ __forceinline__ float tanh_approx(float x) {
  float y;
  asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

}  // namespace tc
