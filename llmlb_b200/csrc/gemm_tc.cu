// Prefill / batched-decode projections on the 5th-gen tensor cores (SURVEY §8 a2.3/8/9/10/11).
//
//   out[t, n] = sum_k X[t, k] * W[n, k]        X bf16 [T, K], W bf16 [N, K] (both K-major)
//
// "Weights-as-M" tiling: a CTA owns a 128-row slab of W as the MMA's M operand and BN tokens
// as the N operand (BN = 16..256 picked from T), so one kernel serves 16-token batched decode
// (HBM-bound: W streamed once through a deep TMA ring) and 512-token prefill (tensor-bound).
// Warp roles (384 threads, 1 CTA/SM, persistent over tiles):
//   warp 0 lane 0 : TMA producer   — cp.async.bulk.tensor 2D, 128B-swizzled 64-wide K slabs
//   warp 1 lane 0 : MMA issuer     — tcgen05.mma.cta_group::1.kind::f16, fp32 accum in TMEM
//   warp 2        : TMEM allocator — 2 accumulator stages (epilogue of tile i overlaps MMA of i+1)
//   warps 4..11   : epilogue       — tcgen05.ld 32x32b (two warps per TMEM lane quarter, half the
//                                    columns each), fused residual-add / SiLU*up / store
// Split-K (residual epilogue only) uses fp32 red.global.add.
#include <cuda.h>

#include "../../include/llmlb_b200.h"
#include "common.cuh"
#include "tc_common.cuh"

namespace llmlb {

static __device__ TraceBuf d_trace_tc;
void tc_set_trace(const TraceBuf& tb) { cudaMemcpyToSymbol(d_trace_tc, &tb, sizeof(tb)); }

template <int BN, int EPI>
__global__ void __launch_bounds__(kTcThreads, 1)
gemm_tc_kernel(const __grid_constant__ CUtensorMap tmap_w, const __grid_constant__ CUtensorMap tmap_x,
               void* __restrict__ out, uint32_t n_tokens, uint32_t n_out, uint32_t K,
               uint32_t out_stride, uint32_t m_tiles, uint32_t t_tiles, uint32_t split_k, uint32_t pdl,
               const TpPushRS tp) {
  using Cfg = TcCfg<BN>;
  __shared__ uint8_t* s_peer_slot[kTpMaxRanks];   // kEpiPushRS: slot base of every rank
  if constexpr (EPI == kEpiPushRS) {
    if (threadIdx.x < tp.ctx.size) s_peer_slot[threadIdx.x] = tp.ctx.base[threadIdx.x] + tp.ctx.slot_off[tp.coll & 1];
  }
  if constexpr (EPI == kEpiPushRSLL) {
    if (threadIdx.x < tp.ctx.size) s_peer_slot[threadIdx.x] = tp.ctx.base[threadIdx.x] + tp.ctx.rsll_off[tp.coll & 1];
  }
  // Programmatic dependent launch: the next kernel of the stream may be
  // scheduled as soon as SMs free up, and THIS kernel may have been scheduled before its
  // predecessor finished: until griddepcontrol.wait it touches nothing but weights.
  if (pdl) asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  extern __shared__ uint8_t smem_dyn[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_dyn) + 1023) &
                                             ~uintptr_t(1023));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + Cfg::kStages * Cfg::kStageBytes);
  uint64_t* full_bar = bars;
  uint64_t* empty_bar = bars + Cfg::kStages;
  uint64_t* tfull_bar = bars + 2 * Cfg::kStages;
  uint64_t* tempty_bar = tfull_bar + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);

  const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t k_blocks_total = (K + kBK - 1) / kBK;
  const uint32_t k_per_split = (k_blocks_total + split_k - 1) / split_k;
  const uint32_t n_tiles = m_tiles * t_tiles * split_k;

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmap_w) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmap_x) : "memory");
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < Cfg::kStages; ++i) {
      mbar_init(full_bar + i, 1);
      mbar_init(empty_bar + i, 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(tfull_bar + i, 1);
      mbar_init(tempty_bar + i, 8);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                     smem_u32(tmem_slot)),
                 "r"(uint32_t(Cfg::kTmemCols))
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  // debug timeline: cycles each role spent blocked (producer on free slots, MMA issuer on data,
  // epilogue on finished accumulators) — see tools/gemm_stalls.py
  const TraceBuf tb = d_trace_tc;
  __shared__ long long stall[4];
  const long long c_begin = clock64();
  long long c_wait = 0;
  const unsigned long long g_begin = tb.data ? gtime_ns() : 0ull;

  // tile -> (m_tile, t_tile, split): t fastest so consecutive CTAs share the W slab in L2
  auto decode_tile = [&](uint32_t tile, uint32_t& mt, uint32_t& tt, uint32_t& ks) {
    tt = tile % t_tiles;
    uint32_t r = tile / t_tiles;
    ks = r % split_k;
    mt = r / split_k;
  };

  if (warp == 0) {
    if (lane == 0) {
      uint32_t stage = 0, phase = 0;
      // L2 prefetch cursor: runs kPrefetchAhead K-slabs ahead of the smem loads (weights only —
      // the activation operand is small and L2-resident).  The smem ring holds 3 slabs in flight
      // (~1.5k MMA cycles); an HBM miss costs 3-4k, an L2 hit ~1k.
      // (a 512-byte-per-row prefetch view through a second, unswizzled map measured slower:
      // lm_head at 64 tokens 188 -> 203 us)
      constexpr uint32_t kPrefetchAhead = 12;
      uint32_t p_tile = blockIdx.x, p_kb = 0, p_kb1 = 0, p_mt = 0;
      auto p_load = [&]() {
        if (p_tile < n_tiles) {
          uint32_t tt, ks;
          decode_tile(p_tile, p_mt, tt, ks);
          p_kb = ks * k_per_split;
          p_kb1 = min(k_blocks_total, p_kb + k_per_split);
        }
      };
      auto p_step = [&]() {
        if (p_tile >= n_tiles) return;
        tma_prefetch_l2_2d(&tmap_w, int32_t(p_kb * kBK), int32_t(p_mt * kBM));
        if (++p_kb >= p_kb1) { p_tile += gridDim.x; p_load(); }
      };
      p_load();
      for (uint32_t i = 0; i < kPrefetchAhead; ++i) p_step();
      // pdl: the first ring of WEIGHT slabs is requested before the predecessor is known to be done;
      // the activation halves of those stages follow after griddepcontrol.wait (same full barrier,
      // its expect_tx already counts both)
      bool dep_ready = pdl == 0;
      if (dep_ready && tp.wait_coll_plus1) tp_wait_ag_single(tp.ctx, tp.wait_coll_plus1 - 1);
      uint32_t n_deferred = 0;
      uint32_t d_stage[Cfg::kStages], d_kb[Cfg::kStages], d_tt[Cfg::kStages];
      auto release_deferred = [&]() {
        asm volatile("griddepcontrol.wait;" ::: "memory");
        if (tp.wait_coll_plus1) tp_wait_ag_single(tp.ctx, tp.wait_coll_plus1 - 1);
        for (uint32_t i = 0; i < n_deferred; ++i)
          tma_load_2d(smem + d_stage[i] * Cfg::kStageBytes + kBM * kBK * 2, &tmap_x, full_bar + d_stage[i],
                      int32_t(d_kb[i] * kBK), int32_t(d_tt[i] * BN));
        dep_ready = true;
      };
      for (uint32_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        uint32_t mt, tt, ks;
        decode_tile(tile, mt, tt, ks);
        const uint32_t kb0 = ks * k_per_split;
        const uint32_t kb1 = min(k_blocks_total, kb0 + k_per_split);
        for (uint32_t kb = kb0; kb < kb1; ++kb) {
          p_step();
          if (!dep_ready && n_deferred == uint32_t(Cfg::kStages)) release_deferred();   // ring full of weights
          { const long long c0 = clock64(); mbar_wait(empty_bar + stage, phase ^ 1); c_wait += clock64() - c0; }
          uint8_t* sa = smem + stage * Cfg::kStageBytes;
          uint8_t* sb = sa + kBM * kBK * 2;
          mbar_expect_tx(full_bar + stage, Cfg::kStageBytes);
          tma_load_2d(sa, &tmap_w, full_bar + stage, int32_t(kb * kBK), int32_t(mt * kBM));
          if (dep_ready) {
            tma_load_2d(sb, &tmap_x, full_bar + stage, int32_t(kb * kBK), int32_t(tt * BN));
          } else {
            d_stage[n_deferred] = stage; d_kb[n_deferred] = kb; d_tt[n_deferred] = tt;
            ++n_deferred;
          }
          if (++stage == Cfg::kStages) { stage = 0; phase ^= 1; }
        }
      }
      if (!dep_ready) release_deferred();   // fewer K blocks than stages
    }
  } else if (warp == 1) {
    if (lane == 0) {
      uint32_t stage = 0, phase = 0, acc = 0, acc_phase = 0;
      for (uint32_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        uint32_t mt, tt, ks;
        decode_tile(tile, mt, tt, ks);
        const uint32_t kb0 = ks * k_per_split;
        const uint32_t kb1 = min(k_blocks_total, kb0 + k_per_split);
        mbar_wait(tempty_bar + acc, acc_phase ^ 1);
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + acc * BN;
        for (uint32_t kb = kb0; kb < kb1; ++kb) {
          { const long long c0 = clock64(); mbar_wait(full_bar + stage, phase); c_wait += clock64() - c0; }
          tc_fence_after();
          const uint32_t sa = smem_u32(smem + stage * Cfg::kStageBytes);
          const uint32_t sb = sa + kBM * kBK * 2;
          const uint64_t adesc = make_sw128_desc(sa);
          const uint64_t bdesc = make_sw128_desc(sb);
#pragma unroll
          for (int k = 0; k < kBK / 16; ++k) {
            // advance 32 B (16 bf16) inside the 128 B swizzle row: +2 in the 16-byte address field
            tc_mma(tmem_d, adesc + uint64_t(k * 2), bdesc + uint64_t(k * 2), Cfg::kIdesc,
                   (kb > kb0 || k > 0) ? 1u : 0u);
          }
          tc_commit(empty_bar + stage);  // frees the smem slot when these MMAs retire
          if (++stage == Cfg::kStages) { stage = 0; phase ^= 1; }
        }
        tc_commit(tfull_bar + acc);      // accumulator complete -> epilogue
        if (++acc == 2) { acc = 0; acc_phase ^= 1; }
      }
    }
  } else if (warp >= 4) {
    const uint32_t q = warp & 3;  // TMEM lane quarter this warp may read
    uint32_t acc = 0, acc_phase = 0;
    if (pdl) asm volatile("griddepcontrol.wait;" ::: "memory");   // outputs may alias what earlier kernels read
    uint32_t ep_ll = 0;
    if constexpr (EPI == kEpiPushRSLL) ep_ll = tp_epoch32(tp.ctx, tp.coll);   // the step counter is final after the wait
    for (uint32_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
      uint32_t mt, tt, ks;
      decode_tile(tile, mt, tt, ks);
      { const long long c0 = clock64(); mbar_wait(tfull_bar + acc, acc_phase); c_wait += clock64() - c0; }
      tc_fence_after();
      const uint32_t n = mt * kBM + q * 32 + lane;      // output feature of this thread
      const uint32_t t0 = tt * BN;
      // two warps share a TMEM lane quarter: each takes half of the token columns
      constexpr uint32_t kColsPerWarp = (BN / 2 >= 16) ? BN / 2 : 16;
      const uint32_t c_begin = ((warp - 4) >> 2) * kColsPerWarp;
      if constexpr (EPI == LLMLB_EPI_STORE_BF16 || EPI == LLMLB_EPI_SILU_MUL || EPI == LLMLB_EPI_STORE_F32) {
        if (split_k > 1) {
          // ---- in-kernel K-split: the split_k CTAs of an output tile each park their fp32 partial in the
          // workspace, meet at the tile's counter, and then each finishes every split_k-th 16-token column
          // group (sum over the parts in part order: deterministic), so the reduction itself is spread
          // over the CTAs that did the products.  All CTAs of the grid are co-resident (one tile per CTA,
          // grid <= SM count) and nobody waits before it has parked its own part.
          const uint32_t otile = mt * t_tiles + tt;
          float* wtile = tp.sk_ws + size_t(otile) * split_k * (BN * kBM);
          float* wmine = wtile + size_t(ks) * (BN * kBM);
#pragma unroll 1
          for (uint32_t c = c_begin; c < c_begin + kColsPerWarp && c < BN; c += 16) {
            if (t0 + c >= n_tokens) break;
            uint32_t r[16];
            tc_ld16(tmem_base + ((q * 32) << 16) + acc * BN + c, r);
            tc_wait_ld();
            float4* dst = reinterpret_cast<float4*>(wmine + (c >> 4) * (16 * kBM) + (q * 32 + lane) * 16);
#pragma unroll
            for (int j = 0; j < 4; ++j)
              dst[j] = make_float4(__uint_as_float(r[4 * j]), __uint_as_float(r[4 * j + 1]), __uint_as_float(r[4 * j + 2]), __uint_as_float(r[4 * j + 3]));
          }
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(tempty_bar + acc);
          epi_bar();
          if (threadIdx.x == 128) {
            __threadfence();                        // the CTA's parked part is performed device-wide before its arrival
            atomicAdd(tp.sk_cnt + otile, 1u);
            const unsigned long long w0 = gtime_ns();
            unsigned int spins = 0;
            while (ld_acquire_gpu_u32(tp.sk_cnt + otile) < split_k) {
              if ((++spins & 0xFFFu) == 0 && gtime_ns() - w0 > 2000000000ull) __trap();   // a part never arrived: fail, do not hang
            }
          }
          epi_bar();
          const uint32_t et = threadIdx.x - 128;    // 0..255
          const uint32_t n_groups = (min(uint32_t(BN), n_tokens - t0) + 15) >> 4;
          for (uint32_t grp = ks; grp < n_groups; grp += split_k) {
            const float* src = wtile + grp * (16 * kBM);
            if constexpr (EPI == LLMLB_EPI_SILU_MUL) {
              const uint32_t pr = et & 63, qt = et >> 6;           // rows (2pr, 2pr+1) = (gate, up); 4 tokens
              float4 g = make_float4(0.f, 0.f, 0.f, 0.f), u = g;
              for (uint32_t s2 = 0; s2 < split_k; ++s2) {
                const float4 a = __ldcg(reinterpret_cast<const float4*>(src + size_t(s2) * (BN * kBM) + (2 * pr) * 16 + qt * 4));
                const float4 b = __ldcg(reinterpret_cast<const float4*>(src + size_t(s2) * (BN * kBM) + (2 * pr + 1) * 16 + qt * 4));
                g.x += a.x; g.y += a.y; g.z += a.z; g.w += a.w;
                u.x += b.x; u.y += b.y; u.z += b.z; u.w += b.w;
              }
              const uint32_t nn = mt * kBM + 2 * pr;
              if (nn + 1 < n_out) {
                __nv_bfloat16* o = reinterpret_cast<__nv_bfloat16*>(out);
                const float gv[4] = {g.x, g.y, g.z, g.w}, uv[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                  const uint32_t t = t0 + grp * 16 + qt * 4 + j;
                  if (t < n_tokens) o[size_t(t) * out_stride + (nn >> 1)] = __float2bfloat16_rn(__fdividef(gv[j], 1.f + __expf(-gv[j])) * uv[j]);
                }
              }
            } else {
              const uint32_t row = et & 127, hf = et >> 7;         // one weight row, 8 tokens
              float4 a0 = make_float4(0.f, 0.f, 0.f, 0.f), a1 = a0;
              for (uint32_t s2 = 0; s2 < split_k; ++s2) {
                const float4* p4 = reinterpret_cast<const float4*>(src + size_t(s2) * (BN * kBM) + row * 16 + hf * 8);
                const float4 a = __ldcg(p4), b = __ldcg(p4 + 1);
                a0.x += a.x; a0.y += a.y; a0.z += a.z; a0.w += a.w;
                a1.x += b.x; a1.y += b.y; a1.z += b.z; a1.w += b.w;
              }
              const uint32_t nn = mt * kBM + row;
              if (nn < n_out) {
                const float v[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                  const uint32_t t = t0 + grp * 16 + hf * 8 + j;
                  if (t < n_tokens) {
                    const size_t idx = size_t(t) * out_stride + nn;
                    if constexpr (EPI == LLMLB_EPI_STORE_BF16) reinterpret_cast<__nv_bfloat16*>(out)[idx] = __float2bfloat16_rn(v[j]);
                    else reinterpret_cast<float*>(out)[idx] = v[j];
                  }
                }
              }
            }
          }
          // second pass over the counter: the CTA that sees every part gone through the meeting point zeroes it
          if (threadIdx.x == 128 && atomicAdd(tp.sk_cnt + otile, 1u) == 2 * split_k - 1) atomicExch(tp.sk_cnt + otile, 0u);
          if (++acc == 2) { acc = 0; acc_phase ^= 1; }
          continue;
        }
      }
#pragma unroll 1
      for (uint32_t c = c_begin; c < c_begin + kColsPerWarp && c < BN; c += 16) {
        if (t0 + c >= n_tokens) break;                  // warp-uniform
        uint32_t r[16];
        tc_ld16(tmem_base + ((q * 32) << 16) + acc * BN + c, r);
        tc_wait_ld();
        if constexpr (EPI == kEpiPushRSLL) {
          // lanes (2i, 2i+1) hold output features (n, n+1) of the same tokens: one 8-byte word {bf16 n, bf16 n+1, epoch}
          // per token; even lanes send the even token columns, odd lanes the odd ones
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            const float v = __uint_as_float(r[j]);
            const float other = __shfl_xor_sync(0xffffffffu, v, 1);
            const uint32_t t = t0 + c + j;
            if (((j ^ lane) & 1) == 0 && (n | 1) < n_out && t < n_tokens) {
              const float lo = (lane & 1) ? other : v, hi = (lane & 1) ? v : other;
              const uint32_t owner = t / tp.rpr, tl = t - owner * tp.rpr;
              uint2 w;
              w.x = pack_bf16(lo, hi);
              w.y = ep_ll;
              st_peer_u2(reinterpret_cast<uint2*>(s_peer_slot[owner]) +
                             (size_t(tp.ctx.rank * split_k + ks) * tp.rpr + tl) * (out_stride / 2) + (n >> 1), w);
            }
          }
        } else if constexpr (EPI == LLMLB_EPI_SILU_MUL) {
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
        } else {
          if (n < n_out) {
#pragma unroll
            for (int j = 0; j < 16; ++j) {
              const uint32_t t = t0 + c + j;
              if (t < n_tokens) {
                const float v = __uint_as_float(r[j]);
                const size_t idx = size_t(t) * out_stride + n;
                if constexpr (EPI == LLMLB_EPI_STORE_BF16)
                  reinterpret_cast<__nv_bfloat16*>(out)[idx] = __float2bfloat16_rn(v);
                else if constexpr (EPI == LLMLB_EPI_STORE_F32)
                  reinterpret_cast<float*>(out)[idx] = v;
                else if constexpr (EPI == kEpiPartialF32)  // deterministic split-K: slot ks of the workspace
                  reinterpret_cast<float*>(out)[size_t(ks) * n_tokens * out_stride + idx] = v;
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
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(tempty_bar + acc);
      if (++acc == 2) { acc = 0; acc_phase ^= 1; }
    }
  }

  if (tb.data) {
    if (warp == 0 && lane == 0) stall[0] = c_wait;
    if (warp == 1 && lane == 0) stall[1] = c_wait;
    if (warp == 4 && lane == 0) stall[2] = c_wait;  // epilogue warp 4: first column half
  }
  tc_fence_before();
  __syncthreads();
  if (tb.data && threadIdx.x == 0)
    trace_emit(tb, (6ull << 60) | ((unsigned long long)EPI << 56) | ((unsigned long long)n_out << 32) | K, g_begin, g_begin, gtime_ns(), n_tokens);
  if (tb.data && threadIdx.x == 0)
    trace_emit(tb, (2ull << 60) | ((unsigned long long)n_out << 32) | ((unsigned long long)EPI << 28) | K,
               (unsigned long long)(clock64() - c_begin), (unsigned long long)stall[0], (unsigned long long)stall[1],
               (unsigned long long)stall[2]);
  if (warp == 2) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base),
                 "r"(uint32_t(Cfg::kTmemCols))
                 : "memory");
  }
  if constexpr (EPI == kEpiPushRS) {
    const uint32_t slot = tp.coll & 1;
    tp_signal_when_grid_done(tp.ctx, &tp_flags(tp.ctx, tp.ctx.rank)->done[slot], gridDim.x, tp_epoch(tp.ctx, tp.coll),
                             [&](TpFlags* f) { return &f->push_flag[slot][tp.ctx.rank]; });
  }
}

// ----------------------------------------------------------------- host side ----------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*,
                                  const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                  const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) ==
            cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = (EncodeTiledFn)p;
  }
  return fn;
}

// 2D bf16 row-major [rows, cols]; box = {64 cols, box_rows}; 128B swizzle
int make_tmap_bf16(CUtensorMap* m, const void* base, uint64_t rows, uint64_t cols,
                   uint32_t box_rows) {
  EncodeTiledFn fn = get_encode_fn();
  if (!fn) {
    set_error("cuTensorMapEncodeTiled not available from the driver");
    return LLMLB_E_DEVICE;
  }
  cuuint64_t gdim[2] = {cols, rows};
  cuuint64_t gstr[1] = {cols * 2};
  cuuint32_t box[2] = {(cuuint32_t)kBK, box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), gdim, gstr, box,
                  estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                  CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed: " + std::to_string((int)r));
    return LLMLB_E_DEVICE;
  }
  return LLMLB_OK;
}

// general tiled map, bf16, 128B swizzle: dims / box innermost first, strides (bytes) of dims 1..rank-1
int make_tmap_nd(CUtensorMap* m, const void* base, uint32_t rank, const uint64_t* dims, const uint64_t* strides_bytes,
                 const uint32_t* box) {
  EncodeTiledFn fn = get_encode_fn();
  if (!fn) {
    set_error("cuTensorMapEncodeTiled not available from the driver");
    return LLMLB_E_DEVICE;
  }
  cuuint64_t gdim[5], gstr[4];
  cuuint32_t bx[5], estr[5];
  for (uint32_t i = 0; i < rank; ++i) { gdim[i] = dims[i]; bx[i] = box[i]; estr[i] = 1; }
  for (uint32_t i = 0; i + 1 < rank; ++i) gstr[i] = strides_bytes[i];
  CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, rank, const_cast<void*>(base), gdim, gstr, bx, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled (rank " + std::to_string(rank) + ") failed: " + std::to_string((int)r));
    return LLMLB_E_DEVICE;
  }
  return LLMLB_OK;
}

uint32_t tc_pick_bn(uint32_t n_tokens);
uint32_t tc_store_split(uint32_t n_tokens, uint32_t n_out, uint32_t k, const TpPushRS* tpp);

template <int BN, int EPI>
static int launch_tc(const CUtensorMap& tw, const CUtensorMap& tx, void* out, uint32_t n_tokens,
                     uint32_t n_out, uint32_t k, uint32_t out_stride, uint32_t split_k,
                     cudaStream_t st, const TpPushRS* tpp = nullptr) {
  using Cfg = TcCfg<BN>;
  auto kern = gemm_tc_kernel<BN, EPI>;
  static bool configured = false;
  if (!configured) {
    LLMLB_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                          Cfg::kSmemBytes));
    configured = true;
  }
  TpPushRS tp{};
  if (tpp) tp = *tpp;
  uint32_t m_tiles = (n_out + kBM - 1) / kBM;
  uint32_t t_tiles = (n_tokens + BN - 1) / BN;
  uint32_t tiles = m_tiles * t_tiles * split_k;
  uint32_t grid = tiles < (uint32_t)kNumSMs ? tiles : (uint32_t)kNumSMs;
  // programmatic dependent launch (64 streams: 12.5k -> 13.2k tok/s, 16 streams +8 %)
  constexpr bool pdl = true;
  if (!pdl) {
    kern<<<grid, kTcThreads, Cfg::kSmemBytes, st>>>(tw, tx, out, n_tokens, n_out, k, out_stride,
                                                    m_tiles, t_tiles, split_k, 0u, tp);
  } else {
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(kTcThreads);
    cfg.dynamicSmemBytes = Cfg::kSmemBytes;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    LLMLB_CUDA_CHECK(cudaLaunchKernelEx(&cfg, kern, tw, tx, out, n_tokens, n_out, k, out_stride, m_tiles, t_tiles, split_k, 1u, tp));
  }
  LLMLB_LAUNCH_CHECK();
  return LLMLB_OK;
}

template <int BN>
static int dispatch_tc_epi(uint32_t epi, const CUtensorMap& tw, const CUtensorMap& tx, void* out,
                           uint32_t n_tokens, uint32_t n_out, uint32_t k, uint32_t out_stride,
                           uint32_t split_k, cudaStream_t st, const TpPushRS* tpp) {
  switch (epi) {
    case LLMLB_EPI_STORE_BF16:
      return launch_tc<BN, LLMLB_EPI_STORE_BF16>(tw, tx, out, n_tokens, n_out, k, out_stride, split_k, st, tpp);
    case LLMLB_EPI_RESID_F32:
      return launch_tc<BN, LLMLB_EPI_RESID_F32>(tw, tx, out, n_tokens, n_out, k, out_stride,
                                                split_k, st);
    case LLMLB_EPI_SILU_MUL:
      return launch_tc<BN, LLMLB_EPI_SILU_MUL>(tw, tx, out, n_tokens, n_out, k, out_stride, split_k, st, tpp);
    case LLMLB_EPI_STORE_F32:
      return launch_tc<BN, LLMLB_EPI_STORE_F32>(tw, tx, out, n_tokens, n_out, k, out_stride, split_k, st, tpp);
    case kEpiPartialF32:
      return launch_tc<BN, kEpiPartialF32>(tw, tx, out, n_tokens, n_out, k, out_stride, split_k, st);
    case kEpiPushRS:
      return launch_tc<BN, kEpiPushRS>(tw, tx, out, n_tokens, n_out, k, out_stride, split_k, st, tpp);
    case kEpiPushRSLL:
      if constexpr (BN <= 128) return launch_tc<BN, kEpiPushRSLL>(tw, tx, out, n_tokens, n_out, k, out_stride, split_k, st, tpp);
      break;
  }
  set_error("gemm_tc: unknown epilogue");
  return LLMLB_E_INVALID_ARG;
}

// K-split of a store-epilogue GEMM (one 128 x BN tile per CTA, all co-resident): as many parts as keep the grid
// within the SM count, at least 4 K blocks each, every part non-empty.  1 = no split (no workspace, or enough tiles).
uint32_t tc_store_split(uint32_t n_tokens, uint32_t n_out, uint32_t k, const TpPushRS* tpp) {
  if (!tpp || !tpp->sk_ws || !tpp->sk_cnt) return 1;
  const uint32_t bn = tc_pick_bn(n_tokens);
  const uint32_t tiles = ((n_out + kBM - 1) / kBM) * ((n_tokens + bn - 1) / bn);
  const uint32_t kblocks = (k + kBK - 1) / kBK;
  if (tiles * 2 > (uint32_t)kNumSMs || tiles > kSkCounters) return 1;
  uint32_t s = (uint32_t)kNumSMs / tiles;
  if (s > 16) s = 16;
  if (s > kblocks / 4) s = kblocks / 4;
  if (s < 2) return 1;
  const uint32_t per = (kblocks + s - 1) / s;
  return (kblocks + per - 1) / per;
}

uint32_t tc_pick_bn(uint32_t n_tokens) {
  if (n_tokens <= 16) return 16;
  if (n_tokens <= 32) return 32;
  if (n_tokens <= 64) return 64;
  if (n_tokens <= 128) return 128;
  return 256;
}

// Launch with prebuilt tensor maps (the engine caches them: weights never move, activation
// buffers are fixed).  The X map's box rows must equal tc_pick_bn(n_tokens).
int gemm_tc2_launch(const CUtensorMap& tw, const CUtensorMap& tx_half, void* out, uint32_t n_tokens,
                    uint32_t n_out, uint32_t k, uint32_t epi, uint32_t out_stride, cudaStream_t st,
                    uint32_t* n_parts, const TpPushRS* tpp, uint32_t max_split);

// tx_half (optional): the activation map with a 128-row box; when given and the step is wide
// enough for 256-token tiles the CTA-pair kernel (gemm_tc2.cu) runs instead.
// K-split (kEpiPartialF32 / kEpiPushRS / RESID_F32 only) up to max_split parts; *n_parts = parts used.
// (A stream-K work split of the same pipeline was built and measured in round 1 — no better than
// slab tiles + K-split partials in either regime; it lives in tools/experiments/csrc/gemm_sk.cu.)
int gemm_tc_launch(const CUtensorMap& tw, const CUtensorMap& tx, void* out, uint32_t n_tokens,
                   uint32_t n_out, uint32_t k, uint32_t epi, uint32_t out_stride,
                   cudaStream_t st, const CUtensorMap* tx_half, uint32_t* n_parts,
                   const TpPushRS* tpp, uint32_t max_split) {
  const uint32_t bn = tc_pick_bn(n_tokens);
  if (n_parts) *n_parts = 1;
  // CTA pairs when there are enough 256 x 256 tiles to occupy most of the GPU; a narrow projection (tensor-
  // parallel shards: QKV at tp = 8 has 6 pair tiles) runs 128-row tiles with an in-kernel K-split instead
  const bool store_epi = epi == LLMLB_EPI_STORE_BF16 || epi == LLMLB_EPI_SILU_MUL || epi == LLMLB_EPI_STORE_F32;
  const uint32_t pair_ctas = 2 * ((n_out + 255) / 256) * ((n_tokens + 255) / 256);
  const bool narrow = store_epi && pair_ctas < 96 && tc_store_split(n_tokens, n_out, k, tpp) > 1;
  if (tx_half && bn == 256 && n_out >= 256 && !narrow)
    return gemm_tc2_launch(tw, *tx_half, out, n_tokens, n_out, k, epi, out_stride, st, n_parts, tpp, max_split);
  // split K for the residual epilogues when the tile count cannot fill the GPU
  uint32_t split_k = 1;
  if (epi == LLMLB_EPI_RESID_F32 || epi == (uint32_t)kEpiPartialF32 || epi == (uint32_t)kEpiPushRS || epi == (uint32_t)kEpiPushRSLL) {
    uint32_t tiles = ((n_out + kBM - 1) / kBM) * ((n_tokens + bn - 1) / bn);
    uint32_t kblocks = (k + kBK - 1) / kBK;
    while (tiles * split_k * 2 <= (uint32_t)kNumSMs && kblocks / (split_k * 2) >= 8 && split_k * 2 <= max_split) split_k *= 2;
  } else {
    split_k = tc_store_split(n_tokens, n_out, k, tpp);   // store epilogues: K-split reduced inside the kernel
  }
  if (n_parts) *n_parts = split_k;
  switch (bn) {
    case 16: return dispatch_tc_epi<16>(epi, tw, tx, out, n_tokens, n_out, k, out_stride, split_k, st, tpp);
    case 32: return dispatch_tc_epi<32>(epi, tw, tx, out, n_tokens, n_out, k, out_stride, split_k, st, tpp);
    case 64: return dispatch_tc_epi<64>(epi, tw, tx, out, n_tokens, n_out, k, out_stride, split_k, st, tpp);
    case 128: return dispatch_tc_epi<128>(epi, tw, tx, out, n_tokens, n_out, k, out_stride, split_k, st, tpp);
    default: return dispatch_tc_epi<256>(epi, tw, tx, out, n_tokens, n_out, k, out_stride, split_k, st, tpp);
  }
}

}  // namespace llmlb

using namespace llmlb;

// Kernel-level entry point of the tensor-core projections (parity tests, micro-benchmarks).
// impl 0 = tcgen05 + TMEM + TMA tiles.  The mma.sync baseline (1) and the stream-K split (2) of
// round 1 are no longer part of the library (tools/experiments/csrc/).
extern "C" int llmlb_op_gemm(const void* w, const void* x, void* out, uint32_t n_tokens,
                             uint32_t n_out, uint32_t k, uint32_t epilogue, uint32_t out_stride,
                             uint32_t impl, void* stream) {
  if (!w || !x || !out || n_out == 0 || k == 0 || k % 8 != 0) {
    set_error("llmlb_op_gemm: bad argument (k must be a multiple of 8)");
    return LLMLB_E_INVALID_ARG;
  }
  // tile counts are 32-bit: a dimension near 2^32 wraps them to zero (fuzzing the entry point over the fake CUDA runtime
  // divided by that zero); nothing the engine serves comes near these bounds
  if (n_tokens > (1u << 20) || n_out > (1u << 24) || k > (1u << 20)) {
    set_error("llmlb_op_gemm: dimension out of range (tokens <= 2^20, n_out <= 2^24, k <= 2^20)");
    return LLMLB_E_INVALID_ARG;
  }
  if (epilogue > LLMLB_EPI_STORE_F32) {
    set_error("llmlb_op_gemm: unknown epilogue");
    return LLMLB_E_INVALID_ARG;
  }
  if (epilogue == LLMLB_EPI_SILU_MUL && (n_out & 1)) {
    set_error("llmlb_op_gemm: SILU_MUL needs interleaved gate/up rows (even n_out)");
    return LLMLB_E_INVALID_ARG;
  }
  if (impl != 0) {
    set_error("llmlb_op_gemm: only impl 0 (tcgen05 tiles) is built into the library");
    return LLMLB_E_UNSUPPORTED;
  }
  if (n_tokens == 0) return LLMLB_OK;
  cudaStream_t st = (cudaStream_t)stream;
  CUtensorMap tw, tx, txh;
  int rc = make_tmap_bf16(&tw, w, n_out, k, 128);
  if (rc) return rc;
  rc = make_tmap_bf16(&tx, x, n_tokens, k, tc_pick_bn(n_tokens));
  if (rc) return rc;
  rc = make_tmap_bf16(&txh, x, n_tokens, k, 128);
  if (rc) return rc;
  // the kernel-level entry point owns one K-split workspace per process (callers are serialised tests / benches)
  static float* op_ws = nullptr;
  static unsigned int* op_cnt = nullptr;
  if (!op_ws) {
    LLMLB_CUDA_CHECK(cudaMalloc((void**)&op_ws, kSkWsBytes));
    LLMLB_CUDA_CHECK(cudaMalloc((void**)&op_cnt, kSkCounters * sizeof(unsigned int)));
    LLMLB_CUDA_CHECK(cudaMemset(op_cnt, 0, kSkCounters * sizeof(unsigned int)));
  }
  TpPushRS tpp{};
  tpp.sk_ws = op_ws; tpp.sk_cnt = op_cnt;
  return gemm_tc_launch(tw, tx, out, n_tokens, n_out, k, epilogue, out_stride, st, &txh, nullptr, &tpp, 8);
}

// Host-only (no launch, no device): the K-split a store-epilogue projection of this shape would run with, and the grid
// it implies — what tests/test_gemm_plan_cpu.py checks the co-residency invariants of the in-kernel K-split on.
// out = {tile rows BN (token tile), tiles, split_k, CTAs}
extern "C" int llmlb_debug_store_split(uint32_t n_tokens, uint32_t n_out, uint32_t k, uint32_t out[4]) {
  if (!out || n_tokens == 0 || n_out == 0 || k == 0) return LLMLB_E_INVALID_ARG;
  TpPushRS tpp{};
  tpp.sk_ws = reinterpret_cast<float*>(uintptr_t(1));          // "a workspace exists": never dereferenced here
  tpp.sk_cnt = reinterpret_cast<unsigned int*>(uintptr_t(1));
  const uint32_t bn = tc_pick_bn(n_tokens);
  const uint32_t tiles = ((n_out + kBM - 1) / kBM) * ((n_tokens + bn - 1) / bn);
  const uint32_t s = tc_store_split(n_tokens, n_out, k, &tpp);
  out[0] = bn; out[1] = tiles; out[2] = s; out[3] = tiles * s;
  return LLMLB_OK;
}
