// Decode GEMV, K-split variant (the one the engine's batch-1 decode runs).
//
// Why: with "a warp owns whole rows" the work quantum is a 4-row group, and 7168 groups over
// 2368 resident warps leaves some warps 4 trips and most 3 (25% tail), while N=4096 outputs only
// fill 64 CTAs.  Here the quantum is one row PAIR per CTA: rows are dealt to the 148 CTAs in
// contiguous, near-equal ranges and every warp of a CTA streams its own K slice of EVERY row of
// the CTA, so all SMs pull from HBM for the whole kernel regardless of N.
//   * CTA = 16 warps.  K is cut into 256-element chunks (one 16-byte load per lane); a "team" of
//     TW warps covers a row, each warp CW chunks (TW*CW*256 == K).  16/TW teams take alternate
//     row batches.
//   * The x slice of a lane never changes -> it lives in registers (fp32), RMSNorm fused: the CTA
//     reduces sum(x^2) once, each lane normalises only its own slice.
//   * Row batches of RB = 8/CW rows are software-pipelined: the next batch's 16-byte streaming
//     loads are issued before the current batch is reduced, so ~16 loads/lane stay in flight.
//   * Per batch: per-row warp shuffle tree -> partial[buf][row][warp] in smem -> team-scoped named
//     barrier -> team warp 0 finishes the sum and applies the epilogue (residual add / SiLU*up / ...).
// Algorithmic bytes: n_out * k * 2 per launch.
#include "../../include/llmlb_b200.h"
#include "common.cuh"
#include "tp_common.cuh"

namespace llmlb {

// Tensor-parallel decode (protocol A of tp_common.cuh), fused into this kernel:
//   TPM == 1  the RMSNorm prologue is the all-reduce's consumer: every CTA folds the N partial rows
//             of the slot into the replicated fp32 residual (rank order), spinning on the epoch of
//             each {value, epoch} pair, keeps the new residual in shared memory for the norm and
//             writes its share of it to x_out (the other residual buffer: other CTAs of this grid
//             still read x_in)
//   TPM == 2  the epilogue is the producer: every finished output element is stored with its epoch
//             into the slot of EVERY rank (no flag, no end-of-grid signal)
struct TpGemv {
  TpCtx ctx;
  uint32_t coll_in, coll_out;   // collective consumed by the prologue / produced by the epilogue
  float* x_out;                 // TPM == 1: residual after the fold
};

constexpr int kKsThreads = 512;
constexpr int kKsWarps = 16;
static __device__ TraceBuf d_trace_ks;
void ks_set_trace(const TraceBuf& tb) { cudaMemcpyToSymbol(d_trace_ks, &tb, sizeof(tb)); }

__device__ __forceinline__ void team_barrier(int id, int threads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(threads) : "memory");
}

template <int B, int EPI, bool NORM, int CW, int TPM>
__global__ void __launch_bounds__(kKsThreads)
gemv_ks_kernel(const __nv_bfloat16* __restrict__ W, const void* xin /* predecessor output: no restrict (PDL) */,
               const __nv_bfloat16* __restrict__ gain, float eps, void* __restrict__ out,
               uint32_t n_out, uint32_t K, uint32_t out_stride, uint32_t TW,
               const uint8_t* __restrict__ pf_ptr, uint32_t pf_bytes, const TpGemv tp) {
  static_assert(TPM == 0 || (TPM == 1 && NORM) || (TPM == 2 && !NORM && EPI == LLMLB_EPI_STORE_F32), "tp mode");
  extern __shared__ float ks_dyn[];   // TPM == 1: the folded residual, [B][K] fp32
  constexpr int RB = 8 / CW;  // rows per batch (even)
  __shared__ float partial[2][kKsWarps][RB * B];  // [buf][warp][row*B + b]
  __shared__ float red[B][kKsWarps];

  const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const uint32_t teams = kKsWarps / TW;
  const uint32_t team = warp / TW, wt = warp % TW;  // team index, warp within team
  const bool active = team < teams;                  // spare warps (16 % TW) only help the prologue

  // rows of this CTA, in row pairs so SiLU(gate)*up pairs never straddle CTAs
  const uint32_t n_pairs = (n_out + 1) / 2;
  const uint32_t row_begin = uint32_t((uint64_t(blockIdx.x) * n_pairs) / gridDim.x) * 2;
  const uint32_t row_end = min(n_out, uint32_t((uint64_t(blockIdx.x + 1) * n_pairs) / gridDim.x) * 2);
  const uint32_t n_batches = (row_end - row_begin + RB - 1) / RB;
  const uint32_t rows_base = row_begin, rows_lim = row_end;

  // element offset of this lane's chunk c: chunks are interleaved over the team's warps
  auto koff = [&](int c) { return (uint32_t(c) * TW + wt) * 256u + lane * 8u; };

  uint4 wf[RB][CW];
  auto load_batch = [&](uint32_t batch) {
#pragma unroll
    for (int r = 0; r < RB; ++r) {
      const uint32_t row = min(rows_base + batch * RB + r, n_out - 1);
      const __nv_bfloat16* p = W + size_t(row) * K;
#pragma unroll
      for (int c = 0; c < CW; ++c) wf[r][c] = ldg_stream(p + koff(c));
    }
  };
  const TraceBuf tb = d_trace_ks;
  unsigned long long tr0 = 0, tr1 = 0, tr2 = 0, tr_flag = 0;
  if (tb.data && threadIdx.x == 0) tr0 = gtime_ns();
  // PDL: let the next kernel in the stream start its own weight prefetch right away ...
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  // this CTA's batches: team, team+teams, ...  (a dynamically dealt variant was measured in round 1:
  // slower — the per-trip atomic + publish costs more than the ~6 % tail spread it removes)
  uint32_t batch = team;
  const uint32_t stride0 = teams;
  if (active && batch < n_batches) load_batch(batch);
  // ... and only now wait for the producer of x / out (weights above never depend on it)
  asm volatile("griddepcontrol.wait;" ::: "memory");
  if (tb.data && threadIdx.x == 0) tr1 = gtime_ns();
  uint32_t ep_out = 0;   // TPM == 2: the epoch every pushed value carries (step counter is final after the wait)
  if constexpr (TPM == 2) ep_out = tp_epoch32(tp.ctx, tp.coll_out);

  // ---- prologue: this lane's slice of x in fp32 registers (RMSNorm fused) ----
  float xr[B][CW][8];
  if constexpr (NORM) {
    const float* xf = reinterpret_cast<const float*>(xin);
    float ss[B];
#pragma unroll
    for (int b = 0; b < B; ++b) ss[b] = 0.f;
    if constexpr (TPM == 1) {
      const uint32_t slot = tp.coll_in & 1;
      TpFlags* mine = tp_flags(tp.ctx, tp.ctx.rank);
      const uint32_t ep32 = tp_epoch32(tp.ctx, tp.coll_in);
      const uint8_t* slot_base = tp.ctx.base[tp.ctx.rank] + tp.ctx.ll_off[slot];
      // x_in[b][4i..4i+3] + the N pushed partials, summed in rank order (identical sums on every rank); the loads
      // of up to four sources are issued together
      auto fold_one = [&](int b, uint32_t i) -> float4 {
        float4 v = reinterpret_cast<const float4*>(xf + size_t(b) * K)[i];
        for (uint32_t r0 = 0; r0 < tp.ctx.size; r0 += 4) {
          const uint4* pp[4];
          uint4 pa[4], pb[4];
#pragma unroll
          for (int q = 0; q < 4; ++q)
            if (r0 + q < tp.ctx.size) {
              pp[q] = reinterpret_cast<const uint4*>(slot_base) + ((size_t(r0 + q) * kTpSmallRows + b) * K + 4 * size_t(i)) / 2;
              pa[q] = ld_pairs(pp[q]); pb[q] = ld_pairs(pp[q] + 1);
            }
#pragma unroll
          for (int q = 0; q < 4; ++q)
            if (r0 + q < tp.ctx.size) {
              const float4 a = tp_take_pairs(mine, pp[q], pa[q], pb[q], ep32);
              v.x += a.x; v.y += a.y; v.z += a.z; v.w += a.w;
            }
        }
        return v;
      };
      // every CTA folds the whole residual itself (one L2 hop after the push lands)
      for (uint32_t i = threadIdx.x; i < K / 4; i += kKsThreads) {
#pragma unroll
        for (int b = 0; b < B; ++b) {
          const float4 v = fold_one(b, i);
          reinterpret_cast<float4*>(ks_dyn + size_t(b) * K)[i] = v;
          if (i % gridDim.x == blockIdx.x) reinterpret_cast<float4*>(tp.x_out + size_t(b) * K)[i] = v;
          ss[b] += v.x * v.x + v.y * v.y + v.z * v.z + v.w * v.w;
        }
      }
      if (tb.data && threadIdx.x == 0) tr_flag = gtime_ns();
      xf = ks_dyn;   // generic pointer into shared memory: the slices below come from the fold
    } else {
    for (uint32_t i = threadIdx.x; i < K / 4; i += kKsThreads) {
#pragma unroll
      for (int b = 0; b < B; ++b) {
        float4 v = reinterpret_cast<const float4*>(xf + size_t(b) * K)[i];
        ss[b] += v.x * v.x + v.y * v.y + v.z * v.z + v.w * v.w;
      }
    }
    }
#pragma unroll
    for (int b = 0; b < B; ++b) {
      float s = warp_sum(ss[b]);
      if (lane == 0) red[b][warp] = s;
    }
    __syncthreads();
#pragma unroll
    for (int b = 0; b < B; ++b) {
      float tot = 0.f;
#pragma unroll
      for (int w = 0; w < kKsWarps; ++w) tot += red[b][w];
      const float rs = rsqrtf(tot / float(K) + eps);
      if (active) {
#pragma unroll
        for (int c = 0; c < CW; ++c) {
          const uint32_t k0 = koff(c);
          const float4 v0 = *reinterpret_cast<const float4*>(xf + size_t(b) * K + k0);
          const float4 v1 = *reinterpret_cast<const float4*>(xf + size_t(b) * K + k0 + 4);
          const uint4 g = __ldg(reinterpret_cast<const uint4*>(gain + k0));
          // same rounding point as the standalone rmsnorm kernel: y is bf16
          xr[b][c][0] = __bfloat162float(__float2bfloat16_rn(v0.x * rs * bf16_lo(g.x)));
          xr[b][c][1] = __bfloat162float(__float2bfloat16_rn(v0.y * rs * bf16_hi(g.x)));
          xr[b][c][2] = __bfloat162float(__float2bfloat16_rn(v0.z * rs * bf16_lo(g.y)));
          xr[b][c][3] = __bfloat162float(__float2bfloat16_rn(v0.w * rs * bf16_hi(g.y)));
          xr[b][c][4] = __bfloat162float(__float2bfloat16_rn(v1.x * rs * bf16_lo(g.z)));
          xr[b][c][5] = __bfloat162float(__float2bfloat16_rn(v1.y * rs * bf16_hi(g.z)));
          xr[b][c][6] = __bfloat162float(__float2bfloat16_rn(v1.z * rs * bf16_lo(g.w)));
          xr[b][c][7] = __bfloat162float(__float2bfloat16_rn(v1.w * rs * bf16_hi(g.w)));
        }
      }
    }
  } else {
    if (active) {
      const __nv_bfloat16* xb = reinterpret_cast<const __nv_bfloat16*>(xin);
#pragma unroll
      for (int b = 0; b < B; ++b)
#pragma unroll
        for (int c = 0; c < CW; ++c) {
          const uint4 v = *reinterpret_cast<const uint4*>(xb + size_t(b) * K + koff(c));
          xr[b][c][0] = bf16_lo(v.x); xr[b][c][1] = bf16_hi(v.x);
          xr[b][c][2] = bf16_lo(v.y); xr[b][c][3] = bf16_hi(v.y);
          xr[b][c][4] = bf16_lo(v.z); xr[b][c][5] = bf16_hi(v.z);
          xr[b][c][6] = bf16_lo(v.w); xr[b][c][7] = bf16_hi(v.w);
        }
    }
  }
  if (tb.data && threadIdx.x == 0) tr2 = gtime_ns();
  // ---- main loop: this team's row batches ----
  uint32_t buf = 0;
  uint32_t next = batch + stride0;      // batch after the current one
  if (active)
  for (; batch < n_batches; buf ^= 1) {
    uint4 wc[RB][CW];
#pragma unroll
    for (int r = 0; r < RB; ++r)
#pragma unroll
      for (int c = 0; c < CW; ++c) wc[r][c] = wf[r][c];
    if (next < n_batches) load_batch(next);

    float acc[RB][B];
#pragma unroll
    for (int r = 0; r < RB; ++r) {
#pragma unroll
      for (int b = 0; b < B; ++b) acc[r][b] = 0.f;
#pragma unroll
      for (int c = 0; c < CW; ++c) {
        const uint4 w = wc[r][c];
        const float w0 = bf16_lo(w.x), w1 = bf16_hi(w.x), w2 = bf16_lo(w.y), w3 = bf16_hi(w.y);
        const float w4 = bf16_lo(w.z), w5 = bf16_hi(w.z), w6 = bf16_lo(w.w), w7 = bf16_hi(w.w);
#pragma unroll
        for (int b = 0; b < B; ++b) {
          float a = acc[r][b];
          a = fmaf(w0, xr[b][c][0], a); a = fmaf(w1, xr[b][c][1], a);
          a = fmaf(w2, xr[b][c][2], a); a = fmaf(w3, xr[b][c][3], a);
          a = fmaf(w4, xr[b][c][4], a); a = fmaf(w5, xr[b][c][5], a);
          a = fmaf(w6, xr[b][c][6], a); a = fmaf(w7, xr[b][c][7], a);
          acc[r][b] = a;
        }
      }
    }
#pragma unroll
    for (int r = 0; r < RB; ++r)
#pragma unroll
      for (int b = 0; b < B; ++b) {
        const float s = warp_sum(acc[r][b]);
        if (lane == 0) partial[buf][warp][r * B + b] = s;
      }
    team_barrier(1 + int(team), int(TW) * 32);
    if (wt == 0) {
      // lanes 0 .. RB*B-1: one (row, token) each; sum the team's partials in warp order
      const uint32_t r = lane / B, b = lane % B;
      float v = 0.f;
      if (lane < RB * B)
        for (uint32_t w = 0; w < TW; ++w) v += partial[buf][team * TW + w][lane];
      const uint32_t row = rows_base + batch * RB + r;
      if constexpr (EPI == LLMLB_EPI_SILU_MUL) {
        const float up = __shfl_down_sync(0xffffffffu, v, B);  // row r+1, same token
        if (lane < RB * B && (r & 1) == 0 && row + 1 < rows_lim) {
          const float s = v / (1.f + __expf(-v));
          reinterpret_cast<__nv_bfloat16*>(out)[size_t(b) * out_stride + (row >> 1)] =
              __float2bfloat16_rn(s * up);
        }
      } else if constexpr (TPM == 2) {
        if (lane < RB * B && row < rows_lim) {
          const size_t idx = (size_t(tp.ctx.rank) * kTpSmallRows + b) * out_stride + row;
          const uint32_t slot = tp.coll_out & 1;
          for (uint32_t r = 0; r < tp.ctx.size; ++r)
            st_peer_pair(reinterpret_cast<uint2*>(tp.ctx.base[r] + tp.ctx.ll_off[slot]) + idx, v, ep_out);
        }
      } else if (lane < RB * B && row < rows_lim) {
        const size_t idx = size_t(b) * out_stride + row;
        if constexpr (EPI == LLMLB_EPI_STORE_BF16)
          reinterpret_cast<__nv_bfloat16*>(out)[idx] = __float2bfloat16_rn(v);
        else if constexpr (EPI == LLMLB_EPI_RESID_F32)
          reinterpret_cast<float*>(out)[idx] += v;
        else
          reinterpret_cast<float*>(out)[idx] = v;
      }
    }
    batch = next;
    next += stride0;
  }
  // ---- tail: pull the head of the NEXT projection's weights into L2 while this kernel drains
  // and the next one launches (the boundary otherwise leaves HBM idle for ~2-3 us) ----
  for (uint32_t off = (blockIdx.x * kKsThreads + threadIdx.x) * 128u; off < pf_bytes; off += gridDim.x * kKsThreads * 128u)
    asm volatile("prefetch.global.L2 [%0];" ::"l"(pf_ptr + off));
  if (tb.data && threadIdx.x == 0) {
    trace_emit(tb, ((unsigned long long)TPM << 58) | ((unsigned long long)n_out << 32) | K, tr0, tr1, tr2, gtime_ns());
    if (TPM == 1) trace_emit(tb, (5ull << 60) | ((unsigned long long)n_out << 32) | K, tr1, tr_flag, tr2, 0);   // dependency wait -> fold done -> norm done
  }
}

// picks (TW, CW): TW*CW*256 == K, TW <= 16, CW in {1,2,4}, B*CW <= 4.  Returns false if none.
static bool ks_pick(uint32_t n_tokens, uint32_t K, uint32_t* tw, uint32_t* cw) {
  if (K % 256) return false;
  const uint32_t chunks = K / 256;
  for (uint32_t c : {1u, 2u, 4u}) {
    if (chunks % c) continue;
    uint32_t t = chunks / c;
    if (t <= 16 && n_tokens * c <= 4) { *tw = t; *cw = c; return true; }
  }
  return false;
}

template <int B, int EPI, bool NORM, int CW, int TPM = 0>
static int ks_launch(const void* w, const void* x, const void* gain, float eps, void* out,
                     uint32_t n_out, uint32_t k, uint32_t out_stride, uint32_t tw, cudaStream_t st,
                     const void* pf_ptr, uint32_t pf_bytes, const TpGemv* tp = nullptr) {
  uint32_t n_pairs = (n_out + 1) / 2;
  uint32_t grid = n_pairs < (uint32_t)kNumSMs ? n_pairs : (uint32_t)kNumSMs;
  auto kern = gemv_ks_kernel<B, EPI, NORM, CW, TPM>;
  size_t dyn = 0;
  if constexpr (TPM == 1) {
    dyn = size_t(B) * k * sizeof(float);
    static size_t configured = 0;
    if (dyn > configured) {
      LLMLB_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn));
      configured = dyn;
    }
  }
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(kKsThreads);
  cfg.dynamicSmemBytes = dyn;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;  // programmatic dependent launch
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  TpGemv tpv{};
  if (tp) tpv = *tp;
  LLMLB_CUDA_CHECK(cudaLaunchKernelEx(&cfg, kern, (const __nv_bfloat16*)w, x,
                                      (const __nv_bfloat16*)gain, eps, out, n_out, k, out_stride, tw,
                                      (const uint8_t*)pf_ptr, pf_bytes, tpv));
  LLMLB_LAUNCH_CHECK();
  return LLMLB_OK;
}

template <int B, int CW>
static int ks_dispatch(uint32_t epi, bool norm, const void* w, const void* x, const void* gain,
                       float eps, void* out, uint32_t n_out, uint32_t k, uint32_t out_stride,
                       uint32_t tw, cudaStream_t st, const void* pf, uint32_t pfb) {
#define KS_CASE(E)                                                                                       \
  case E:                                                                                                \
    return norm ? ks_launch<B, E, true, CW>(w, x, gain, eps, out, n_out, k, out_stride, tw, st, pf, pfb) \
                : ks_launch<B, E, false, CW>(w, x, gain, eps, out, n_out, k, out_stride, tw, st, pf, pfb);
  switch (epi) {
    KS_CASE(LLMLB_EPI_STORE_BF16)
    KS_CASE(LLMLB_EPI_RESID_F32)
    KS_CASE(LLMLB_EPI_SILU_MUL)
    KS_CASE(LLMLB_EPI_STORE_F32)
  }
#undef KS_CASE
  set_error("gemv_ks: unknown epilogue");
  return LLMLB_E_INVALID_ARG;
}

// returns LLMLB_E_UNSUPPORTED when the shape does not fit this variant (caller falls back)
int gemv_ks_try(const void* w, const void* x, const void* gain, float eps, void* out,
                uint32_t n_tokens, uint32_t n_out, uint32_t k, uint32_t epi, uint32_t out_stride,
                cudaStream_t st, const void* pf_ptr, uint32_t pf_bytes) {
  uint32_t tw = 0, cw = 0;
  if (n_tokens == 0 || n_tokens > 4 || !ks_pick(n_tokens, k, &tw, &cw)) return LLMLB_E_UNSUPPORTED;
  const bool norm = gain != nullptr;
#define KS_GO(BB, CC) return ks_dispatch<BB, CC>(epi, norm, w, x, gain, eps, out, n_out, k, out_stride, tw, st, pf_ptr, pf_bytes)
  if (n_tokens == 1) { if (cw == 1) KS_GO(1, 1); if (cw == 2) KS_GO(1, 2); KS_GO(1, 4); }
  if (n_tokens == 2) { if (cw == 1) KS_GO(2, 1); KS_GO(2, 2); }
  if (n_tokens == 3) KS_GO(3, 1);
  KS_GO(4, 1);
#undef KS_GO
}

// ---- tensor-parallel variants (protocol A of tp_common.cuh) ----
bool gemv_tp_shape_ok(uint32_t n_tokens, uint32_t k) {
  uint32_t tw, cw;
  return n_tokens >= 1 && n_tokens <= 4 && ks_pick(n_tokens, k, &tw, &cw);
}

// consumer: x_out = x_in + sum of the pushed partials of collective coll_in; out = epi(W . RMSNorm(x_out))
int gemv_tp_consume(const TpCtx& ctx, uint32_t coll_in, const void* w, const float* x_in, float* x_out,
                    const void* gain, float eps, void* out, uint32_t n_tokens, uint32_t n_out, uint32_t k,
                    uint32_t epi, uint32_t out_stride, cudaStream_t st) {
  uint32_t tw = 0, cw = 0;
  if (n_tokens == 0 || n_tokens > 4 || !gain || !ks_pick(n_tokens, k, &tw, &cw)) return LLMLB_E_UNSUPPORTED;
  TpGemv tp{};
  tp.ctx = ctx; tp.coll_in = coll_in; tp.x_out = x_out;
#define KS_TC(BB, CC)                                                                                                          \
  switch (epi) {                                                                                                               \
    case LLMLB_EPI_STORE_BF16: return ks_launch<BB, LLMLB_EPI_STORE_BF16, true, CC, 1>(w, x_in, gain, eps, out, n_out, k, out_stride, tw, st, nullptr, 0, &tp); \
    case LLMLB_EPI_SILU_MUL: return ks_launch<BB, LLMLB_EPI_SILU_MUL, true, CC, 1>(w, x_in, gain, eps, out, n_out, k, out_stride, tw, st, nullptr, 0, &tp);     \
    case LLMLB_EPI_STORE_F32: return ks_launch<BB, LLMLB_EPI_STORE_F32, true, CC, 1>(w, x_in, gain, eps, out, n_out, k, out_stride, tw, st, nullptr, 0, &tp);   \
    default: set_error("gemv_tp_consume: epilogue"); return LLMLB_E_INVALID_ARG;                                               \
  }
  if (n_tokens == 1) { if (cw == 1) { KS_TC(1, 1) } if (cw == 2) { KS_TC(1, 2) } KS_TC(1, 4) }
  if (n_tokens == 2) { if (cw == 1) { KS_TC(2, 1) } KS_TC(2, 2) }
  if (n_tokens == 3) { KS_TC(3, 1) }
  KS_TC(4, 1)
#undef KS_TC
}

// producer: partial = W . x (bf16 x) pushed into slot[coll_out & 1][my rank] of every rank (n_out = hidden)
int gemv_tp_push(const TpCtx& ctx, uint32_t coll_out, const void* w, const void* x_bf16, uint32_t n_tokens,
                 uint32_t n_out, uint32_t k, cudaStream_t st) {
  uint32_t tw = 0, cw = 0;
  if (n_tokens == 0 || n_tokens > 4 || !ks_pick(n_tokens, k, &tw, &cw)) return LLMLB_E_UNSUPPORTED;
  TpGemv tp{};
  tp.ctx = ctx; tp.coll_out = coll_out;
#define KS_TP(BB, CC) return ks_launch<BB, LLMLB_EPI_STORE_F32, false, CC, 2>(w, x_bf16, nullptr, 0.f, nullptr, n_out, k, n_out, tw, st, nullptr, 0, &tp)
  if (n_tokens == 1) { if (cw == 1) KS_TP(1, 1); if (cw == 2) KS_TP(1, 2); KS_TP(1, 4); }
  if (n_tokens == 2) { if (cw == 1) KS_TP(2, 1); KS_TP(2, 2); }
  if (n_tokens == 3) KS_TP(3, 1);
  KS_TP(4, 1);
#undef KS_TP
}

}  // namespace llmlb
