// Prefill projections, 2-CTA tcgen05 variant (cta_group::2): a CTA PAIR (thread-block cluster of
// 2 on one TPC) owns a 256-row slab of W x BN tokens.  Each CTA stages only ITS 128 weight rows
// and HALF of the token tile; the pair's tensor cores read both halves, so the activation
// operand crosses L2->SM once per pair instead of once per CTA (32 KiB instead of 48 KiB per
// K slab per SM).  Round-1 profile of the 1-CTA kernel: tensor pipe 49-60 % busy with L2->SM
// traffic at 9.3 TB/s — the operand feed, not the MMA rate, was the limit.
//
//   leader CTA (cluster rank 0) : its warp 1 issues every tcgen05.mma.cta_group::2 for the pair
//   both CTAs                   : TMA producer (completes on the LEADER's full barrier), TMEM
//                                 allocator, 4 epilogue warps reading their own 128 TMEM lanes
//   barriers                    : full[stage]   leader, count 2 (leader expect_tx + peer arrive)
//                                 empty[stage]  per CTA, count 1, tcgen05.commit multicast 0b11
//                                 tfull[acc]    per CTA, count 1, commit multicast 0b11
//                                 tempty[acc]   leader, count 16 (8 epilogue warps x 2 CTAs)
#include <cuda.h>

#include "../../include/llmlb_b200.h"
#include "common.cuh"
#include "tc_common.cuh"

namespace llmlb {

static __device__ TraceBuf d_trace_tc2;
void tc2_set_trace(const TraceBuf& tb) { cudaMemcpyToSymbol(d_trace_tc2, &tb, sizeof(tb)); }
constexpr uint32_t kPeerBitMask = 0xFEFFFFFFu;  // clears the CTA-rank bit of a shared::cluster address

__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\nbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// TMA load whose completion bytes are credited to the LEADER CTA's barrier (same smem offset)
__device__ __forceinline__ void tma_load_2d_2sm(void* smem_dst, const CUtensorMap* tmap, uint64_t* bar,
                                                int32_t c0, int32_t c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(tmap), "r"(smem_u32(bar) & kPeerBitMask), "r"(c0), "r"(c1)
      : "memory");
}
// arrive (count 1) on the barrier at the same offset in the leader CTA
__device__ __forceinline__ void mbar_arrive_leader(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(smem_u32(bar) & kPeerBitMask)
               : "memory");
}
__device__ __forceinline__ void tc_commit_2sm(uint64_t* bar) {  // arrives on `bar` in BOTH CTAs
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
      ::"r"(smem_u32(bar)), "h"(uint16_t(3))
      : "memory");
}
__device__ __forceinline__ void tc_mma_2sm(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                           uint32_t accumulate) {
  asm volatile(
      "{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n}\n"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}

template <int BN>
struct Tc2Cfg {
  static constexpr int kHalfN = BN / 2;                                  // tokens staged per CTA
  static constexpr int kStageBytes = kBM * kBK * 2 + kHalfN * kBK * 2;   // per CTA
  static constexpr int kStages = (BN >= 256) ? 6 : 8;
  static constexpr int kTmemCols = 2 * BN;
  static constexpr int kSmemBytes = kStages * kStageBytes + 1024 + 256;
  // bf16 x bf16 -> f32, K-major A and B, M = 256 (pair), N = BN
  static constexpr uint32_t kIdesc =
      (1u << 4) | (1u << 7) | (1u << 10) | (uint32_t(BN >> 3) << 17) | (uint32_t(256 >> 4) << 24);
};

template <int BN, int EPI>
__global__ void __launch_bounds__(kTcThreads, 1)
gemm_tc2_kernel(const __grid_constant__ CUtensorMap tmap_w, const __grid_constant__ CUtensorMap tmap_x,
                void* __restrict__ out, uint32_t n_tokens, uint32_t n_out, uint32_t K, uint32_t out_stride,
                uint32_t m_tiles /*256-row slabs*/, uint32_t t_tiles, uint32_t split_k, const TpPushRS tp) {
  using Cfg = Tc2Cfg<BN>;
  const TraceBuf tb = d_trace_tc2;
  unsigned long long tr0 = 0, tr1 = 0;
  if (tb.data && threadIdx.x == 0) tr0 = gtime_ns();
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");   // the next kernel may set itself up on freed SMs
  __shared__ uint8_t* s_peer_slot[kTpMaxRanks];   // kEpiPushRS: slot base of every rank
  if constexpr (EPI == kEpiPushRS) {
    if (threadIdx.x < tp.ctx.size) s_peer_slot[threadIdx.x] = tp.ctx.base[threadIdx.x] + tp.ctx.slot_off[tp.coll & 1];
  }
  extern __shared__ uint8_t smem_dyn[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_dyn) + 1023) & ~uintptr_t(1023));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + Cfg::kStages * Cfg::kStageBytes);
  uint64_t* full_bar = bars;
  uint64_t* empty_bar = bars + Cfg::kStages;
  uint64_t* tfull_bar = bars + 2 * Cfg::kStages;
  uint64_t* tempty_bar = tfull_bar + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);

  const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const bool leader = rank == 0;
  const uint32_t pair = blockIdx.x >> 1, n_pairs = gridDim.x >> 1;
  const uint32_t k_blocks_total = (K + kBK - 1) / kBK;
  const uint32_t k_per_split = (k_blocks_total + split_k - 1) / split_k;
  const uint32_t n_tiles = m_tiles * t_tiles * split_k;

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmap_w) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmap_x) : "memory");
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < Cfg::kStages; ++i) {
      mbar_init(full_bar + i, 2);
      mbar_init(empty_bar + i, 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(tfull_bar + i, 1);
      mbar_init(tempty_bar + i, 16);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                 "r"(uint32_t(Cfg::kTmemCols))
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  cluster_sync_all();  // peer barriers are initialised before anyone signals them
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  // programmatic dependent launch: barrier init, TMEM allocation and the tensor-map fetch above
  // overlapped the previous kernel's tail; its outputs (our activations) are needed from here on
  asm volatile("griddepcontrol.wait;" ::: "memory");
  if (tb.data && threadIdx.x == 0) tr1 = gtime_ns();

  auto decode_tile = [&](uint32_t tile, uint32_t& mt, uint32_t& tt, uint32_t& ks) {
    tt = tile % t_tiles;
    uint32_t r = tile / t_tiles;
    ks = r % split_k;
    mt = r / split_k;
  };

  if (warp == 0) {
    if (lane == 0) {  // ---- TMA producer (both CTAs) ----
      if (tp.wait_coll_plus1) tp_wait_ag_single(tp.ctx, tp.wait_coll_plus1 - 1);
      uint32_t stage = 0, phase = 0;
      for (uint32_t tile = pair; tile < n_tiles; tile += n_pairs) {
        uint32_t mt, tt, ks;
        decode_tile(tile, mt, tt, ks);
        const uint32_t kb0 = ks * k_per_split;
        const uint32_t kb1 = min(k_blocks_total, kb0 + k_per_split);
        for (uint32_t kb = kb0; kb < kb1; ++kb) {
          mbar_wait(empty_bar + stage, phase ^ 1);
          uint8_t* sa = smem + stage * Cfg::kStageBytes;
          uint8_t* sb = sa + kBM * kBK * 2;
          if (leader) mbar_expect_tx(full_bar + stage, 2 * Cfg::kStageBytes);  // both CTAs' bytes
          else mbar_arrive_leader(full_bar + stage);
          tma_load_2d_2sm(sa, &tmap_w, full_bar + stage, int32_t(kb * kBK), int32_t(mt * 256 + rank * kBM));
          tma_load_2d_2sm(sb, &tmap_x, full_bar + stage, int32_t(kb * kBK), int32_t(tt * BN + rank * Cfg::kHalfN));
          if (++stage == Cfg::kStages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    if (leader && lane == 0) {  // ---- MMA issuer for the pair ----
      uint32_t stage = 0, phase = 0, acc = 0, acc_phase = 0;
      for (uint32_t tile = pair; tile < n_tiles; tile += n_pairs) {
        uint32_t mt, tt, ks;
        decode_tile(tile, mt, tt, ks);
        const uint32_t kb0 = ks * k_per_split;
        const uint32_t kb1 = min(k_blocks_total, kb0 + k_per_split);
        mbar_wait(tempty_bar + acc, acc_phase ^ 1);
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + acc * BN;
        for (uint32_t kb = kb0; kb < kb1; ++kb) {
          mbar_wait(full_bar + stage, phase);
          tc_fence_after();
          const uint32_t sa = smem_u32(smem + stage * Cfg::kStageBytes);
          const uint32_t sb = sa + kBM * kBK * 2;
          const uint64_t adesc = make_sw128_desc(sa);
          const uint64_t bdesc = make_sw128_desc(sb);
#pragma unroll
          for (int k = 0; k < kBK / 16; ++k)
            tc_mma_2sm(tmem_d, adesc + uint64_t(k * 2), bdesc + uint64_t(k * 2), Cfg::kIdesc, (kb > kb0 || k > 0) ? 1u : 0u);
          tc_commit_2sm(empty_bar + stage);
          if (++stage == Cfg::kStages) { stage = 0; phase ^= 1; }
        }
        tc_commit_2sm(tfull_bar + acc);
        if (++acc == 2) { acc = 0; acc_phase ^= 1; }
      }
    }
  } else if (warp >= 4) {  // ---- epilogue (both CTAs, own TMEM lanes = own 128 weight rows) ----
    const uint32_t q = warp & 3;
    uint32_t acc = 0, acc_phase = 0;
    for (uint32_t tile = pair; tile < n_tiles; tile += n_pairs) {
      uint32_t mt, tt, ks;
      decode_tile(tile, mt, tt, ks);
      mbar_wait(tfull_bar + acc, acc_phase);
      tc_fence_after();
      const uint32_t n = mt * 256 + rank * kBM + q * 32 + lane;
      const uint32_t t0 = tt * BN;
      // two warps share a TMEM lane quarter: each takes half of the token columns
      constexpr uint32_t kColsPerWarp = (BN / 2 >= 16) ? BN / 2 : 16;
      const uint32_t c_begin = ((warp - 4) >> 2) * kColsPerWarp;
#pragma unroll 1
      for (uint32_t c = c_begin; c < c_begin + kColsPerWarp && c < BN; c += 16) {
        if (t0 + c >= n_tokens) break;
        uint32_t r[16];
        tc_ld16(tmem_base + ((q * 32) << 16) + acc * BN + c, r);
        tc_wait_ld();
        if constexpr (EPI == LLMLB_EPI_SILU_MUL) {
          __nv_bfloat16* o = reinterpret_cast<__nv_bfloat16*>(out);
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            const float v = __uint_as_float(r[j]);
            const float other = __shfl_xor_sync(0xffffffffu, v, 1);
            // lanes (2i, 2i+1) hold (gate_i, up_i); even lanes finish even columns, odd lanes odd ones
            if (((j ^ lane) & 1) == 0 && (n | 1) < n_out && t0 + c + j < n_tokens) {
              const float g = (lane & 1) ? other : v, u = (lane & 1) ? v : other;
              const float s = __fdividef(g, 1.f + __expf(-g));  // IEEE division was ~half of the epilogue's instructions
              o[size_t(t0 + c + j) * out_stride + (n >> 1)] = __float2bfloat16_rn(s * u);
            }
          }
        } else if (n < n_out) {
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            const uint32_t t = t0 + c + j;
            if (t < n_tokens) {
              const float v = __uint_as_float(r[j]);
              const size_t idx = size_t(t) * out_stride + n;
              if constexpr (EPI == LLMLB_EPI_STORE_BF16) reinterpret_cast<__nv_bfloat16*>(out)[idx] = __float2bfloat16_rn(v);
              else if constexpr (EPI == LLMLB_EPI_STORE_F32) reinterpret_cast<float*>(out)[idx] = v;
              else if constexpr (EPI == kEpiPartialF32) reinterpret_cast<float*>(out)[size_t(ks) * n_tokens * out_stride + idx] = v;
              else if constexpr (EPI == kEpiPushRS) {    // reduce-scatter by address into the row owner's slot
                const uint32_t owner = t / tp.rpr, tl = t - owner * tp.rpr;
                st_peer_bf16(reinterpret_cast<__nv_bfloat16*>(s_peer_slot[owner]) +
                                 (size_t(tp.ctx.rank * split_k + ks) * tp.rpr + tl) * out_stride + n, v);
              } else {
                if (split_k > 1) atomicAdd(reinterpret_cast<float*>(out) + idx, v);
                else reinterpret_cast<float*>(out)[idx] += v;
              }
            }
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_leader(tempty_bar + acc);  // leader's MMA thread reuses the accumulator
      if (++acc == 2) { acc = 0; acc_phase ^= 1; }
    }
  }

  tc_fence_before();
  cluster_sync_all();  // nobody frees TMEM / exits while the peer may still signal or read
  if (tb.data && threadIdx.x == 0)
    trace_emit(tb, (4ull << 60) | ((unsigned long long)EPI << 56) | ((unsigned long long)n_out << 32) | K, tr0, tr1, gtime_ns(), n_tokens);
  if (warp == 2) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(uint32_t(Cfg::kTmemCols))
                 : "memory");
  }
  if constexpr (EPI == kEpiPushRS) {
    const uint32_t slot = tp.coll & 1;
    tp_signal_when_grid_done(tp.ctx, &tp_flags(tp.ctx, tp.ctx.rank)->done[slot], gridDim.x, tp_epoch(tp.ctx, tp.coll),
                             [&](TpFlags* f) { return &f->push_flag[slot][tp.ctx.rank]; });
  }
}

template <int BN, int EPI>
static int launch_tc2(const CUtensorMap& tw, const CUtensorMap& tx_half, void* out, uint32_t n_tokens, uint32_t n_out,
                      uint32_t k, uint32_t out_stride, uint32_t split_k, cudaStream_t st, const TpPushRS* tpp = nullptr) {
  using Cfg = Tc2Cfg<BN>;
  auto kern = gemm_tc2_kernel<BN, EPI>;
  static bool configured = false;
  if (!configured) {
    LLMLB_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmemBytes));
    configured = true;
  }
  TpPushRS tp{};
  if (tpp) tp = *tpp;
  const uint32_t m_tiles = (n_out + 255) / 256, t_tiles = (n_tokens + BN - 1) / BN;
  const uint32_t tiles = m_tiles * t_tiles * split_k;
  uint32_t pairs = tiles < (uint32_t)(kNumSMs / 2) ? tiles : (uint32_t)(kNumSMs / 2);
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(pairs * 2);
  cfg.blockDim = dim3(kTcThreads);
  cfg.dynamicSmemBytes = Cfg::kSmemBytes;
  cfg.stream = st;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 2;
  LLMLB_CUDA_CHECK(cudaLaunchKernelEx(&cfg, kern, tw, tx_half, out, n_tokens, n_out, k, out_stride, m_tiles, t_tiles, split_k, tp));
  LLMLB_LAUNCH_CHECK();
  return LLMLB_OK;
}

// BN = 256 only (n_tokens > 128).  tx_half: activation tensor map with a 128-row box.
int gemm_tc2_launch(const CUtensorMap& tw, const CUtensorMap& tx_half, void* out, uint32_t n_tokens, uint32_t n_out,
                    uint32_t k, uint32_t epi, uint32_t out_stride, cudaStream_t st, uint32_t* n_parts,
                    const TpPushRS* tpp, uint32_t max_split) {
  uint32_t split_k = 1;
  if (epi == LLMLB_EPI_RESID_F32 || epi == (uint32_t)kEpiPartialF32 || epi == (uint32_t)kEpiPushRS) {
    uint32_t tiles = ((n_out + 255) / 256) * ((n_tokens + 255) / 256);
    uint32_t kblocks = (k + kBK - 1) / kBK;
    while (tiles * split_k * 2 <= (uint32_t)(kNumSMs / 2) && kblocks / (split_k * 2) >= 8 && split_k * 2 <= max_split) split_k *= 2;
  }
  if (n_parts) *n_parts = split_k;
  switch (epi) {
    case LLMLB_EPI_STORE_BF16: return launch_tc2<256, LLMLB_EPI_STORE_BF16>(tw, tx_half, out, n_tokens, n_out, k, out_stride, 1, st, tpp);
    case LLMLB_EPI_RESID_F32: return launch_tc2<256, LLMLB_EPI_RESID_F32>(tw, tx_half, out, n_tokens, n_out, k, out_stride, split_k, st);
    case LLMLB_EPI_SILU_MUL: return launch_tc2<256, LLMLB_EPI_SILU_MUL>(tw, tx_half, out, n_tokens, n_out, k, out_stride, 1, st, tpp);
    case LLMLB_EPI_STORE_F32: return launch_tc2<256, LLMLB_EPI_STORE_F32>(tw, tx_half, out, n_tokens, n_out, k, out_stride, 1, st, tpp);
    case kEpiPartialF32: return launch_tc2<256, kEpiPartialF32>(tw, tx_half, out, n_tokens, n_out, k, out_stride, split_k, st);
    case kEpiPushRS: return launch_tc2<256, kEpiPushRS>(tw, tx_half, out, n_tokens, n_out, k, out_stride, split_k, st, tpp);
  }
  set_error("gemm_tc2: unknown epilogue");
  return LLMLB_E_INVALID_ARG;
}

}  // namespace llmlb
