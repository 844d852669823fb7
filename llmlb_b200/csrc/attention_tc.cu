// Prefill attention on the 5th-generation tensor cores (SURVEY §8 a2.6): causal GQA flash attention
// over the paged KV cache with tcgen05.mma, accumulators in TMEM, operands staged by TMA.
//
// One CTA per (q tile of up to 128 rows, q head).  Per KV block of 128 tokens (two 64-token pages):
//
//   S[128 q, 128 kv]  = Q · K^T      tcgen05.mma M=128 N=128, 8 k-steps over head_dim 128; Q and K
//                                    K-major in 128B-swizzled shared memory (TMA boxes of 64 columns)
//   softmax           8 warps, thread = (row, column half): tcgen05.ld of the S row, scale + causal mask,
//                                    running max / sum in registers (online softmax), P as bf16 into
//                                    shared memory in the 128B-swizzled K-major layout of an A operand
//   PV[128 q, 128 d]  = P · V        tcgen05.mma, A = P (shared), B = V **MN-major**: a V page is
//                                    [token][d] (d contiguous), which is exactly the MN-major
//                                    128B-swizzle canonical layout ((8,n),(8,k)):((1,LBO),(8,SBO)) in
//                                    16-byte units: LBO = distance between the two 64-wide d halves,
//                                    SBO = 1024 B between 8-token groups — no transposed copy of V
//   O (registers)     = O * corr + PV   tcgen05.ld of the fresh PV block (the rescale happens in
//                                    registers, so TMEM never needs a read-modify-write)
//
// Warp roles (384 threads): warp 0 lane 0 TMA producer (Q once; K/V pages of block j+1 while block j
// computes, 2 stages), warp 1 lane 0 MMA issuer, warp 2 TMEM allocator, warps 4..11 softmax.
// K/V pages are addressed through ONE 5-D tensor map per pool [layer][page][kv head][64][128];
// q rows through a 2-D map over the qkv activation.  Masked scores are exactly 0 in P, and pages
// only ever hold finite values (the pool is zero-filled at creation), so stale tokens past the
// causal horizon contribute exactly nothing.
// Algorithmic work: 4 * n_rows * kv_len * 128 flop per (tile, head) (half of it above the diagonal
// is masked but still issued inside a 128-block).
#include <cuda.h>

#include "../../include/llmlb_b200.h"
#include "common.cuh"
#include "tc_common.cuh"

namespace llmlb {

constexpr int kAtRows = 128;        // q rows per CTA (UMMA M)
constexpr int kAtBlock = 128;       // kv tokens per block (UMMA N of S, K of PV)
constexpr int kAtThreads = 384;
constexpr int kAtStages = 2;
constexpr uint32_t kAtSlab = kAtRows * 64 * 2;          // 16 KiB: 128 rows x 64 bf16, one swizzle slab
constexpr uint32_t kAtQBytes = 2 * kAtSlab;             // Q: two 64-wide d slabs
constexpr uint32_t kAtKBytes = 2 * kAtSlab;             // K block: [d half][page a | page b][64 tok][64 d]
constexpr uint32_t kAtVBytes = 2 * kAtSlab;
constexpr uint32_t kAtPBytes = 2 * kAtSlab;             // P: two 64-wide kv slabs
constexpr uint32_t kAtSmem = kAtQBytes + kAtStages * (kAtKBytes + kAtVBytes) + kAtPBytes + 1024 /*align*/ + 256 /*barriers*/;
constexpr uint32_t kAtTmemCols = 256;                   // S: columns 0..127, PV: 128..255
// bf16 x bf16 -> f32, M = 128, N = 128; bit 16 = B operand MN-major
constexpr uint32_t kIdescQK = (1u << 4) | (1u << 7) | (1u << 10) | (uint32_t(128 >> 3) << 17) | (uint32_t(128 >> 4) << 24);
constexpr uint32_t kIdescPV = kIdescQK | (1u << 16);

__device__ __forceinline__ void tma_load_5d(void* smem_dst, const CUtensorMap* tmap, uint64_t* bar, int32_t c0, int32_t c1,
                                            int32_t c2, int32_t c3, int32_t c4) {
  asm volatile(
      "cp.async.bulk.tensor.5d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, %7}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(tmap), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
      : "memory");
}
// MN-major, 128B swizzle: LBO = bytes between 64-element atoms along MN, SBO = bytes between 8-row groups along K
__device__ __forceinline__ uint64_t make_sw128_mn_desc(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= uint64_t((smem_addr >> 4) & 0x3FFF);
  d |= uint64_t((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= uint64_t((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= uint64_t(1) << 46;   // descriptor version 1 (Blackwell)
  d |= uint64_t(2) << 61;   // SWIZZLE_128B
  return d;
}
__device__ __forceinline__ void softmax_bar() { asm volatile("bar.sync 1, 256;" ::: "memory"); }

__global__ void __launch_bounds__(kAtThreads, 1)
prefill_attention_kernel_tc(const __grid_constant__ CUtensorMap tmap_q, const __grid_constant__ CUtensorMap tmap_k,
                            const __grid_constant__ CUtensorMap tmap_v, uint32_t layer,
                            const int32_t* __restrict__ block_tables, uint32_t bt_stride, const int4* __restrict__ tiles,
                            __nv_bfloat16* __restrict__ out, uint32_t n_heads, uint32_t n_kv, uint32_t pdl) {
  extern __shared__ uint8_t at_smem_dyn[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(at_smem_dyn) + 1023) & ~uintptr_t(1023));
  uint8_t* sq = smem;
  uint8_t* skv = sq + kAtQBytes;                                   // [stage][K | V]
  uint8_t* sp = skv + kAtStages * (kAtKBytes + kAtVBytes);
  uint64_t* bars = reinterpret_cast<uint64_t*>(sp + kAtPBytes);
  uint64_t* q_full = bars;
  uint64_t* kv_full = bars + 1;        // [2]
  uint64_t* kv_empty = bars + 3;       // [2]
  uint64_t* s_full = bars + 5;
  uint64_t* p_full = bars + 6;
  uint64_t* o_full = bars + 7;
  uint64_t* o_free = bars + 8;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 9);
  __shared__ float s_xmax[2][2][kAtRows];   // [block parity][column half][row]: row maxima exchanged between the halves
  __shared__ float s_xsum[2][kAtRows];

  if (pdl) asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int4 tile = tiles[blockIdx.x];
  const uint32_t q_row0 = tile.x, n_rows = tile.y, pos0 = tile.z, bt_row = tile.w;
  const uint32_t head = blockIdx.y, kvh = head / (n_heads / n_kv);
  const uint32_t kv_len = pos0 + n_rows;                           // causal horizon of the tile
  const uint32_t n_blocks = (kv_len + kAtBlock - 1) / kAtBlock;
  const uint32_t n_pages = (kv_len + kPageTokens - 1) / kPageTokens;

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmap_q) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmap_k) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmap_v) : "memory");
  }
  if (warp == 1 && lane == 0) {
    mbar_init(q_full, 1);
    for (int i = 0; i < kAtStages; ++i) { mbar_init(kv_full + i, 1); mbar_init(kv_empty + i, 1); }
    mbar_init(s_full, 1);
    mbar_init(p_full, 8);     // one arrival per softmax warp
    mbar_init(o_full, 1);
    mbar_init(o_free, 8);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(kAtTmemCols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  // everything above overlapped the previous kernel's tail; qkv / the pages it wrote are needed from here on
  if (pdl) asm volatile("griddepcontrol.wait;" ::: "memory");

  // (setmaxnreg 48 / 224 between the control and the softmax warpgroups was tried: ptxas then spills
  // 648 bytes instead of 40 — the cap is applied to the whole kernel body — so the split is not used)
  if (warp == 0) {
    if (lane == 0) {   // ---- TMA producer ----
      const int32_t* bt = block_tables + size_t(bt_row) * bt_stride;
      mbar_expect_tx(q_full, kAtQBytes);
      tma_load_2d(sq, &tmap_q, q_full, int32_t(head * kHeadDim), int32_t(q_row0));
      tma_load_2d(sq + kAtSlab, &tmap_q, q_full, int32_t(head * kHeadDim + 64), int32_t(q_row0));
      for (uint32_t j = 0; j < n_blocks; ++j) {
        const uint32_t stage = j & 1, phase = (j >> 1) & 1;
        mbar_wait(kv_empty + stage, phase ^ 1);
        const int32_t pa = bt[2 * j];
        const int32_t pb = (2 * j + 1 < n_pages) ? bt[2 * j + 1] : pa;   // absent page: any valid page, fully masked
        uint8_t* sk = skv + stage * (kAtKBytes + kAtVBytes);
        uint8_t* sv = sk + kAtKBytes;
        mbar_expect_tx(kv_full + stage, kAtKBytes + kAtVBytes);
#pragma unroll
        for (int h = 0; h < 2; ++h) {   // d half; per half: page a then page b, 8 KiB each
          tma_load_5d(sk + h * kAtSlab, &tmap_k, kv_full + stage, h * 64, 0, int32_t(kvh), pa, int32_t(layer));
          tma_load_5d(sk + h * kAtSlab + kAtSlab / 2, &tmap_k, kv_full + stage, h * 64, 0, int32_t(kvh), pb, int32_t(layer));
          tma_load_5d(sv + h * kAtSlab, &tmap_v, kv_full + stage, h * 64, 0, int32_t(kvh), pa, int32_t(layer));
          tma_load_5d(sv + h * kAtSlab + kAtSlab / 2, &tmap_v, kv_full + stage, h * 64, 0, int32_t(kvh), pb, int32_t(layer));
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {   // ---- MMA issuer ----
      const uint32_t tmem_s = tmem_base, tmem_o = tmem_base + 128;
      mbar_wait(q_full, 0);
      for (uint32_t j = 0; j < n_blocks; ++j) {
        const uint32_t stage = j & 1;
        mbar_wait(kv_full + stage, (j >> 1) & 1);
        tc_fence_after();
        const uint32_t sk = smem_u32(skv + stage * (kAtKBytes + kAtVBytes));
        const uint32_t sv = sk + kAtKBytes;
        // S = Q K^T: k-step ks covers d [16 ks, 16 ks + 16): slab ks / 4, 32 bytes per step inside the swizzle row
#pragma unroll
        for (int ks = 0; ks < 8; ++ks) {
          const uint64_t adesc = make_sw128_desc(smem_u32(sq) + (ks >> 2) * kAtSlab) + uint64_t((ks & 3) * 2);
          const uint64_t bdesc = make_sw128_desc(sk + (ks >> 2) * kAtSlab) + uint64_t((ks & 3) * 2);
          tc_mma(tmem_s, adesc, bdesc, kIdescQK, ks > 0 ? 1u : 0u);
        }
        tc_commit(s_full);
        // PV needs P(j) in shared memory and the previous PV block drained from TMEM
        mbar_wait(p_full, j & 1);
        if (j > 0) mbar_wait(o_free, (j - 1) & 1);
        tc_fence_after();
        // PV = P V: k-step ks covers kv tokens [16 ks, 16 ks + 16): P slab ks / 4; V rows advance 16 x 128 B
#pragma unroll
        for (int ks = 0; ks < 8; ++ks) {
          const uint64_t adesc = make_sw128_desc(smem_u32(sp) + (ks >> 2) * kAtSlab) + uint64_t((ks & 3) * 2);
          const uint64_t bdesc = make_sw128_mn_desc(sv + ks * 2048, kAtSlab, 1024);
          tc_mma(tmem_o, adesc, bdesc, kIdescPV, ks > 0 ? 1u : 0u);
        }
        tc_commit(kv_empty + stage);   // K and V of this stage are free once these MMAs retire
        tc_commit(o_full);
      }
    }
  } else if (warp >= 4) {   // ---- softmax + output: thread = (row, 64-column half) ----
    const uint32_t q = warp & 3, half = (warp - 4) >> 2;
    const uint32_t row = q * 32 + lane;
    const uint32_t t_lane = tmem_base + ((q * 32) << 16);
    const float scale = rsqrtf(float(kHeadDim)) * 1.4426950408889634f;
    const uint32_t q_pos = pos0 + row;
    float o[64];
#pragma unroll
    for (int i = 0; i < 64; ++i) o[i] = 0.f;
    float m_run = -INFINITY, l_run = 0.f;
    uint8_t* prow = sp + half * kAtSlab + row * 128;
    for (uint32_t j = 0; j < n_blocks; ++j) {
      mbar_wait(s_full, j & 1);
      tc_fence_after();
      const uint32_t kv0 = j * kAtBlock + half * 64;
      // pass 1: row maximum of my 64 columns
      float mx = -INFINITY;
#pragma unroll
      for (int c = 0; c < 64; c += 16) {
        uint32_t r[16];
        tc_ld16(t_lane + half * 64 + c, r);
        tc_wait_ld();
#pragma unroll
        for (int i = 0; i < 16; ++i)
          if (kv0 + c + i <= q_pos) mx = fmaxf(mx, __uint_as_float(r[i]) * scale);
      }
      s_xmax[j & 1][half][row] = mx;
      softmax_bar();
      const float m_new = fmaxf(m_run, fmaxf(mx, s_xmax[j & 1][half ^ 1][row]));
      const float mu = (m_new == -INFINITY) ? 0.f : m_new;
      const float corr = exp2f(m_run - mu);   // m_run = -inf -> 0
      m_run = m_new;
      // pass 2: p = exp2(s - m), row sum, P as bf16 into the swizzled A-operand layout
      float rsum = 0.f;
#pragma unroll
      for (int c = 0; c < 64; c += 16) {
        uint32_t r[16];
        tc_ld16(t_lane + half * 64 + c, r);
        tc_wait_ld();
        float pv[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) {
          const float s = (kv0 + c + i <= q_pos) ? __uint_as_float(r[i]) * scale : -INFINITY;
          pv[i] = exp2f(s - mu);
          rsum += pv[i];
        }
#pragma unroll
        for (int g = 0; g < 2; ++g) {   // two 16-byte chunks of 8 bf16
          const uint32_t chunk = uint32_t(c / 8 + g);
          uint4 w;
          w.x = pack_bf16(pv[8 * g + 0], pv[8 * g + 1]); w.y = pack_bf16(pv[8 * g + 2], pv[8 * g + 3]);
          w.z = pack_bf16(pv[8 * g + 4], pv[8 * g + 5]); w.w = pack_bf16(pv[8 * g + 6], pv[8 * g + 7]);
          *reinterpret_cast<uint4*>(prow + ((chunk ^ (row & 7)) << 4)) = w;
        }
      }
      l_run = l_run * corr + rsum;
      // P is read by the tensor core (async proxy): make the generic-proxy stores visible, then signal
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(p_full);
      // O = O * corr + PV(j)
      mbar_wait(o_full, j & 1);
      tc_fence_after();
#pragma unroll
      for (int c = 0; c < 64; c += 16) {
        uint32_t r[16];
        tc_ld16(t_lane + 128 + half * 64 + c, r);
        tc_wait_ld();
#pragma unroll
        for (int i = 0; i < 16; ++i) o[c + i] = o[c + i] * corr + __uint_as_float(r[i]);
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(o_free);
    }
    // the two column halves of a row hold partial sums under the same running maximum
    s_xsum[half][row] = l_run;
    softmax_bar();
    const float inv = 1.f / (s_xsum[0][row] + s_xsum[1][row]);
    if (row < n_rows) {
      __nv_bfloat16* dst = out + size_t(q_row0 + row) * n_heads * kHeadDim + size_t(head) * kHeadDim + half * 64;
#pragma unroll
      for (int c = 0; c < 64; c += 8) {
        uint4 w;
        w.x = pack_bf16(o[c] * inv, o[c + 1] * inv); w.y = pack_bf16(o[c + 2] * inv, o[c + 3] * inv);
        w.z = pack_bf16(o[c + 4] * inv, o[c + 5] * inv); w.w = pack_bf16(o[c + 6] * inv, o[c + 7] * inv);
        *reinterpret_cast<uint4*>(dst + c) = w;
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(kAtTmemCols) : "memory");
  }
}

// ----------------------------------------------------------------- host side ----------------
int make_tmap_nd(CUtensorMap* m, const void* base, uint32_t rank, const uint64_t* dims, const uint64_t* strides_bytes,
                 const uint32_t* box);

// q rows: 2-D over the qkv activation [n_tokens, width], box = 64 columns x 128 rows
int make_tmap_attn_q(CUtensorMap* m, const void* qkv, uint64_t n_tokens, uint64_t width) {
  const uint64_t dims[2] = {width, n_tokens}, strides[1] = {width * 2};
  const uint32_t box[2] = {64, (uint32_t)kAtRows};
  return make_tmap_nd(m, qkv, 2, dims, strides, box);
}
// K or V pool [n_layers][n_pages][n_kv][64 tokens][128]: 5-D, box = 64 columns x 64 tokens of one (layer, page, head)
int make_tmap_attn_kv(CUtensorMap* m, const void* pool, uint64_t n_layers, uint64_t n_pages, uint64_t n_kv) {
  const uint64_t dims[5] = {(uint64_t)kHeadDim, (uint64_t)kPageTokens, n_kv, n_pages, n_layers};
  const uint64_t page_bytes = uint64_t(kPageTokens) * kHeadDim * 2;
  const uint64_t strides[4] = {uint64_t(kHeadDim) * 2, page_bytes, page_bytes * n_kv, page_bytes * n_kv * n_pages};
  const uint32_t box[5] = {64, (uint32_t)kPageTokens, 1, 1, 1};
  return make_tmap_nd(m, pool, 5, dims, strides, box);
}

int prefill_attention_tc_launch(const CUtensorMap& mq, const CUtensorMap& mk, const CUtensorMap& mv, uint32_t layer,
                                const int32_t* block_tables, uint32_t bt_stride, const int32_t* tiles, uint32_t n_tiles,
                                void* out, uint32_t n_heads, uint32_t n_kv, bool pdl, cudaStream_t st) {
  if (n_tiles == 0) return LLMLB_OK;
  static bool configured = false;
  if (!configured) {
    LLMLB_CUDA_CHECK(cudaFuncSetAttribute(prefill_attention_kernel_tc, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kAtSmem));
    configured = true;
  }
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(n_tiles, n_heads);
  cfg.blockDim = dim3(kAtThreads);
  cfg.dynamicSmemBytes = kAtSmem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl ? 1 : 0;
  LLMLB_CUDA_CHECK(cudaLaunchKernelEx(&cfg, prefill_attention_kernel_tc, mq, mk, mv, layer, block_tables, bt_stride,
                                      (const int4*)tiles, (__nv_bfloat16*)out, n_heads, n_kv, pdl ? 1u : 0u));
  LLMLB_LAUNCH_CHECK();
  return LLMLB_OK;
}

}  // namespace llmlb

using namespace llmlb;

// a2.6 on tcgen05.  tiles: int32[n_tiles][4] = {first q row, q rows in tile (<= 128), position of the
// first row, row into block_tables}.  k_pages / v_pages: ONE layer's pool [n_pages][n_kv][64][128].
extern "C" int llmlb_op_prefill_attention_tc(const void* qkv, uint32_t n_tokens, const void* k_pages, const void* v_pages,
                                             uint32_t n_pages, const int32_t* block_tables, uint32_t bt_stride,
                                             const int32_t* tiles, uint32_t n_tiles, void* out, uint32_t n_heads,
                                             uint32_t n_kv, void* stream) {
  if (!qkv || !k_pages || !v_pages || !block_tables || !tiles || !out || n_kv == 0 || n_heads % n_kv || n_tokens == 0 || n_pages == 0) {
    set_error("llmlb_op_prefill_attention_tc: bad argument");
    return LLMLB_E_INVALID_ARG;
  }
  CUtensorMap mq, mk, mv;
  int rc = make_tmap_attn_q(&mq, qkv, n_tokens, uint64_t(n_heads + 2 * n_kv) * kHeadDim);
  if (rc) return rc;
  rc = make_tmap_attn_kv(&mk, k_pages, 1, n_pages, n_kv);
  if (rc) return rc;
  rc = make_tmap_attn_kv(&mv, v_pages, 1, n_pages, n_kv);
  if (rc) return rc;
  return prefill_attention_tc_launch(mq, mk, mv, 0, block_tables, bt_stride, tiles, n_tiles, out, n_heads, n_kv, false,
                                     (cudaStream_t)stream);
}
