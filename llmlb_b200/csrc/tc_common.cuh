// PTX wrappers shared by the tcgen05 GEMM kernels (1-CTA gemm_tc.cu, 2-CTA gemm_tc2.cu):
// mbarrier, TMA tensor loads / L2 prefetch, tcgen05 mma / commit / ld, UMMA smem descriptors.
#pragma once
#include <cuda.h>

#include "common.cuh"
#include "tp_common.cuh"

namespace llmlb {

// internal epilogue (not in the public header): fp32 partial product of K-split `ks` stored at
// out + ks * n_tokens * out_stride; the consumer adds the slots in a fixed order (deterministic)
constexpr int kEpiPartialF32 = 4;
// tensor parallel, protocol B (tp_common.cuh): the fp32 partial of token row t, K-split ks, goes
// straight into the slot of the rank that OWNS the row: part (rank * split_k + ks), row t % rpr
constexpr int kEpiPushRS = 5;
// the same for narrow steps (batched decode, T <= kTpLLTokens): every pushed 8-byte word carries two bf16 values of
// adjacent output features AND the collective's epoch, so the owner's reduce kernel spins on the data itself —
// no system fence per CTA, no ticket, no flag round at the end of the GEMM grid (tp_common.cuh, "LL" variant)
constexpr int kEpiPushRSLL = 6;
constexpr uint32_t kTpLLTokens = 128;
struct TpPushRS {
  TpCtx ctx;
  uint32_t coll;      // kEpiPushRS: collective index within the step (slot = coll & 1)
  uint32_t rpr;       // kEpiPushRS: token rows per owner rank = ceil(n_tokens / size)
  uint32_t wait_coll_plus1;   // any epilogue: the activation operand is y of collective (this - 1): the TMA
                              // producer waits for its all-gather flags before the first activation load (0 = none)
  // in-kernel K-split of the store epilogues (bf16 / SiLU*up / fp32): fp32 partial tiles parked in sk_ws,
  // one arrival counter per output tile in sk_cnt (zero between launches); nullptr = no K-split
  float* sk_ws;
  unsigned int* sk_cnt;
};
constexpr size_t kSkWsBytes = size_t(148) * 128 * 256 * 4;   // every CTA of a full grid parks one 128 x 256 fp32 tile
constexpr uint32_t kSkCounters = 256;
constexpr int kBM = 128;          // weight rows per tile  (UMMA M)
constexpr int kBK = 64;           // bf16 per K slab = 128 B = one swizzle row
constexpr int kTcThreads = 384;    // 4 control warps (TMA, MMA, TMEM alloc, spare) + 8 epilogue warps

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)),
               "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred P1;\n"
      "LAB_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
      "@P1 bra DONE;\n"
      "bra LAB_WAIT;\n"
      "DONE:\n"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* tmap, uint64_t* bar,
                                            int32_t c0, int32_t c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, "
      "{%3, %4}], [%2];" ::"r"(smem_u32(smem_dst)),
      "l"(tmap), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
// pull a tile into L2 only (no smem, no barrier): hides HBM latency behind the smem ring
__device__ __forceinline__ void tma_prefetch_l2_2d(const CUtensorMap* tmap, int32_t c0, int32_t c1) {
  asm volatile("cp.async.bulk.prefetch.tensor.2d.L2.global [%0, {%1, %2}];" ::"l"(tmap), "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void tc_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(
                   smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void tc_mma(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc,
                                       uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void tc_ld16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
        "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]),
        "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tc_wait_ld() {
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// K-major, 128B-swizzled operand tile: rows of 128 B, 8-row groups 1024 B apart (SBO),
// descriptor version 1 (Blackwell), layout type 2 (SWIZZLE_128B), LBO unused (=1).
__device__ __forceinline__ uint64_t make_sw128_desc(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= uint64_t((smem_addr >> 4) & 0x3FFF);
  d |= uint64_t(1) << 16;
  d |= uint64_t(1024 >> 4) << 32;
  d |= uint64_t(1) << 46;
  d |= uint64_t(2) << 61;
  return d;
}

__device__ __forceinline__ void epi_bar() {  // the 8 epilogue warps only
  asm volatile("bar.sync 1, 256;" ::: "memory");
}
// tile configuration shared by the 1-CTA kernels (gemm_tc.cu, gemm_sk.cu)
template <int BN>
struct TcCfg {
  static constexpr int kStageBytes = kBM * kBK * 2 + BN * kBK * 2;
  static constexpr int kStages = (BN >= 256) ? 4 : (BN >= 128 ? 6 : 8);
  static constexpr int kTmemCols = (2 * BN < 32) ? 32 : 2 * BN;  // power of two for BN in set
  static constexpr int kSmemBytes = kStages * kStageBytes + 1024 /*align*/ + 256 /*barriers*/;
  // bf16 x bf16 -> f32, A and B K-major, M=128, N=BN
  static constexpr uint32_t kIdesc =
      (1u << 4) | (1u << 7) | (1u << 10) | (uint32_t(BN >> 3) << 17) | (uint32_t(kBM >> 4) << 24);
};

}  // namespace llmlb
