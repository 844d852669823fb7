// Tensor-parallel exchange kernels over NVLink peer memory (SURVEY §8 a2.13).  Layout and the two
// push protocols are described in tp_common.cuh.  This file holds
//   * tp_step_begin_kernel      bumps the step counter the epochs are derived from
//   * tp_reduce_norm_kernel     protocol B consumer: owned rows  x += sum(partials); y = RMSNorm(x)*g
//                               pushed as bf16 into every rank's y buffer (all-gather by address)
//   * tp_push_rows / tp_fold_rows   protocol A, unfused (for projection shapes the fused GEMV
//                               prologue / epilogue in gemv_ks.cu does not take)
//   * allgather_cols_kernel     vocab-sharded logits -> full rows on every rank (pull, barrier)
//   * allreduce_add_kernel      the standalone llmlb_op_allreduce (pull, barrier; parity tests)
#include "../../include/llmlb_b200.h"
#include "common.cuh"
#include "tp_common.cuh"

namespace llmlb {

constexpr int kArMaxBlocks = 148;
static __device__ TraceBuf d_trace_tp;
void tp_set_trace(const TraceBuf& tb) { cudaMemcpyToSymbol(d_trace_tp, &tb, sizeof(tb)); }

struct ArSignals {  // start of every rank's exchange region: barrier flags of the pull kernels
  uint32_t flag[kArMaxBlocks][kTpMaxRanks];  // flag[block][src_rank]: epoch written by src_rank's block
  uint32_t epoch[kArMaxBlocks];              // local only: last epoch this block used
};
constexpr size_t kArSignalBytes = (sizeof(ArSignals) + 255) & ~size_t(255);

size_t tp_region_prefix_bytes() { return kArSignalBytes + kTpFlagBytes; }

__device__ __forceinline__ void st_release_sys(uint32_t* p, uint32_t v) {
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}

// cross-GPU barrier for block blockIdx.x (pull kernels).  Epochs are compared wrap-safe.
__device__ __forceinline__ void ar_barrier(const TpCtx& P) {
  ArSignals* mine = reinterpret_cast<ArSignals*>(P.base[P.rank]);
  __shared__ uint32_t s_epoch;
  if (threadIdx.x == 0) {
    s_epoch = mine->epoch[blockIdx.x] + 1;
    mine->epoch[blockIdx.x] = s_epoch;
  }
  __syncthreads();
  const uint32_t ep = s_epoch;
  if (threadIdx.x < P.size) {
    ArSignals* peer = reinterpret_cast<ArSignals*>(P.base[threadIdx.x]);
    st_release_sys(&peer->flag[blockIdx.x][P.rank], ep);
    const unsigned long long t0 = gtime_ns();
    unsigned int spins = 0;
    while (int32_t(ld_acquire_sys(&mine->flag[blockIdx.x][threadIdx.x]) - ep) < 0) {
      if ((++spins & 0xFFFu) == 0 && gtime_ns() - t0 > 20000000000ull) {
        tp_flags(P, P.rank)->timed_out = 1;
        __threadfence_system();
        __trap();
      }
    }
  }
  __syncthreads();
}

__global__ void tp_step_begin_kernel(TpCtx c) {
  TpFlags* f = tp_flags(c, c.rank);
  f->step = f->step + 1;
}

// ---------------------------------------------------------------- protocol B consumer -------
// grid = max(1, owned rows); CTA b owns token row rank*rpr + b.
template <bool LL>
__global__ void __launch_bounds__(1024)
tp_reduce_norm_kernel(TpCtx c, uint32_t coll, float* __restrict__ x, const __nv_bfloat16* __restrict__ gain,
                      uint32_t n_tokens, uint32_t rpr, uint32_t n_own, uint32_t hidden, float eps, uint32_t n_parts,
                      uint32_t wait_ag) {
  __shared__ float red[32];
  const TraceBuf tb = d_trace_tp;
  unsigned long long tr0 = 0, tr1 = 0, tr2 = 0;
  if (tb.data && threadIdx.x == 0) tr0 = gtime_ns();
  // the projection GEMM that follows may start pulling its weights now (it waits for this grid
  // before it touches y)
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  const uint32_t slot = coll & 1;
  TpFlags* mine = tp_flags(c, c.rank);
  const unsigned long long epoch = tp_epoch(c, coll);
  const uint32_t ep32 = tp_epoch32(c, coll);
  if constexpr (!LL) tp_wait_flags(mine, mine->push_flag[slot], c.size, epoch);
  if (tb.data && threadIdx.x == 0) tr1 = gtime_ns();
  if (blockIdx.x < n_own) {
    const uint32_t t = c.rank * rpr + blockIdx.x;
    float4* xr = reinterpret_cast<float4*>(x + size_t(t) * hidden);
    const uint2* slot_row = reinterpret_cast<const uint2*>(c.base[c.rank] + c.slot_off[slot]) + size_t(blockIdx.x) * (hidden / 4);
    const size_t part_stride = size_t(rpr) * (hidden / 4);
    float ss = 0.f;
    // a thread's elements stay in registers between the two passes (hidden <= 2 * 4 * blockDim; more: re-read)
    float4 keep[2];
    uint32_t it = 0;
    for (uint32_t i = threadIdx.x; i < hidden / 4; i += blockDim.x, ++it) {
      float4 v;
      if constexpr (!LL) v = xr[i];
      // part = rank * split_k + ks, ascending: a fixed order; bf16 on the wire.  Eight loads are in flight
      // together (one dependent L2 round trip per eight parts instead of one per part)
      if constexpr (LL) {
        // narrow steps: every 8-byte word is {bf16 x 2, epoch}: spin on the words themselves (no flag round)
        const uint4* ll_row = reinterpret_cast<const uint4*>(c.base[c.rank] + c.rsll_off[slot]) + size_t(blockIdx.x) * (hidden / 4);
        // The residual row is read only after THIS rank's own words of the collective arrived.  This kernel has no
        // dependency wait and may be resident while the previous collective's reduce kernel (which writes x) is
        // still running (programmatic launches overlap whole kernels when grids are small); the local projection
        // GEMM's words prove it finished: words <- this rank's GEMM <- (its dependency wait) the GEMM before <-
        // that reduce kernel.  (Reading x first gave wrong tokens on 7-wide decode steps: tools/tp_check.py.)
        {
          const uint32_t split_k = n_parts / c.size;
          for (uint32_t ks = 0; ks < split_k; ++ks) {
            const uint4* w = ll_row + size_t(c.rank * split_k + ks) * part_stride + i;
            uint4 a0 = ld_pairs(w);
            if (a0.y != ep32 || a0.w != ep32) {
              const unsigned long long t0 = gtime_ns();
              unsigned int spins = 0;
              do {
                a0 = ld_pairs(w);
                if ((++spins & 0xFFFu) == 0 && gtime_ns() - t0 > 20000000000ull) { mine->timed_out = 1; __threadfence_system(); __trap(); }
              } while (a0.y != ep32 || a0.w != ep32);
            }
          }
          __threadfence();
          v = __ldcg(xr + i);
        }
        for (uint32_t r0 = 0; r0 < n_parts; r0 += 8) {
          uint4 a[8];
#pragma unroll
          for (int q = 0; q < 8; ++q)
            if (r0 + q < n_parts) a[q] = ld_pairs(ll_row + size_t(r0 + q) * part_stride + i);
#pragma unroll
          for (int q = 0; q < 8; ++q)
            if (r0 + q < n_parts) {
              if (a[q].y != ep32 || a[q].w != ep32) {
                const unsigned long long t0 = gtime_ns();
                unsigned int spins = 0;
                do {
                  a[q] = ld_pairs(ll_row + size_t(r0 + q) * part_stride + i);
                  if ((++spins & 0xFFFu) == 0 && gtime_ns() - t0 > 20000000000ull) { mine->timed_out = 1; __threadfence_system(); __trap(); }
                } while (a[q].y != ep32 || a[q].w != ep32);
              }
            }
#pragma unroll
          for (int q = 0; q < 8; ++q)
            if (r0 + q < n_parts) { v.x += bf16_lo(a[q].x); v.y += bf16_hi(a[q].x); v.z += bf16_lo(a[q].z); v.w += bf16_hi(a[q].z); }
        }
      } else {
      for (uint32_t r0 = 0; r0 < n_parts; r0 += 8) {
        uint2 a[8];
#pragma unroll
        for (int q = 0; q < 8; ++q)
          if (r0 + q < n_parts) a[q] = ld_pushed_u2(slot_row + size_t(r0 + q) * part_stride + i);
#pragma unroll
        for (int q = 0; q < 8; ++q)
          if (r0 + q < n_parts) { v.x += bf16_lo(a[q].x); v.y += bf16_hi(a[q].x); v.z += bf16_lo(a[q].y); v.w += bf16_hi(a[q].y); }
      }
      }
      xr[i] = v;
      if (it < 2) keep[it] = v;
      ss += v.x * v.x + v.y * v.y + v.z * v.z + v.w * v.w;
    }
    ss = warp_sum(ss);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = ss;
    __syncthreads();
    float tot = 0.f;
    for (uint32_t w = 0; w < (blockDim.x >> 5); ++w) tot += red[w];
    const float rs = rsqrtf(tot / float(hidden) + eps);
    const uint2* g2 = reinterpret_cast<const uint2*>(gain);
    it = 0;
    for (uint32_t i = threadIdx.x; i < hidden / 4; i += blockDim.x, ++it) {
      const float4 v = it < 2 ? keep[it] : xr[i];  // own writes, same thread
      const uint2 g = __ldg(g2 + i);
      uint2 o;
      o.x = pack_bf16(v.x * rs * bf16_lo(g.x), v.y * rs * bf16_hi(g.x));
      o.y = pack_bf16(v.z * rs * bf16_lo(g.y), v.w * rs * bf16_hi(g.y));
#pragma unroll
      for (uint32_t r = 0; r < uint32_t(kTpMaxRanks); ++r)
        if (r < c.size) st_peer_u2(reinterpret_cast<uint2*>(c.base[r] + c.y_off) + size_t(t) * (hidden / 4) + i, o);
    }
  }
  if (tb.data && threadIdx.x == 0) tr2 = gtime_ns();
  tp_signal_when_grid_done(c, &mine->done[2 + slot], gridDim.x, epoch,
                           [&](TpFlags* f) { return &f->ag_flag[slot][c.rank]; });
  // the grid (hence the kernel boundary the next GEMM waits on) outlives the arrival of every
  // owner's rows in MY y buffer
  if (wait_ag && blockIdx.x == 0) tp_wait_flags(mine, mine->ag_flag[slot], c.size, epoch);
  if (tb.data && threadIdx.x == 0) trace_emit(tb, (3ull << 60) | n_tokens, tr0, tr1, tr2, gtime_ns());   // start, partials in, rows pushed, end
}

// ---------------------------------------------------------------- protocol A, unfused -------
// partial [rows <= 4][hidden] fp32 (local) -> {value, epoch} pairs in slot[coll & 1][src = me] of every rank.
// A 16-byte store of two pairs is not one atomic unit, but each 8-byte pair is: enough.
__global__ void __launch_bounds__(256)
tp_push_rows_kernel(TpCtx c, uint32_t coll, const float* __restrict__ partial, uint32_t rows, uint32_t hidden) {
  const uint32_t slot = coll & 1;
  const uint32_t n4 = rows * hidden / 4;
  const uint32_t h4 = hidden / 4;
  const uint32_t ep32 = tp_epoch32(c, coll);
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += gridDim.x * blockDim.x) {
    const float4 v = reinterpret_cast<const float4*>(partial)[i];
    const uint32_t row = i / h4, col = i - row * h4;
    for (uint32_t r = 0; r < c.size; ++r) {
      uint4* dst = reinterpret_cast<uint4*>(c.base[r] + c.ll_off[slot]) + ((size_t(c.rank) * kTpSmallRows + row) * hidden + 4 * size_t(col)) / 2;
      asm volatile("st.relaxed.sys.global.v4.u32 [%0], {%1,%2,%3,%4};" ::"l"(dst), "r"(__float_as_uint(v.x)), "r"(ep32), "r"(__float_as_uint(v.y)), "r"(ep32) : "memory");
      asm volatile("st.relaxed.sys.global.v4.u32 [%0], {%1,%2,%3,%4};" ::"l"(dst + 1), "r"(__float_as_uint(v.z)), "r"(ep32), "r"(__float_as_uint(v.w)), "r"(ep32) : "memory");
    }
  }
}
// x_out = x_in + sum over src of slot[src]   (rows <= 4)
__global__ void __launch_bounds__(256)
tp_fold_rows_kernel(TpCtx c, uint32_t coll, const float* __restrict__ x_in, float* __restrict__ x_out,
                    uint32_t rows, uint32_t hidden) {
  const uint32_t slot = coll & 1;
  TpFlags* mine = tp_flags(c, c.rank);
  const uint32_t ep32 = tp_epoch32(c, coll);
  const uint32_t n4 = rows * hidden / 4, h4 = hidden / 4;
  const uint4* sb = reinterpret_cast<const uint4*>(c.base[c.rank] + c.ll_off[slot]);
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += gridDim.x * blockDim.x) {
    const uint32_t row = i / h4, col = i - row * h4;
    float4 v = reinterpret_cast<const float4*>(x_in)[i];
    for (uint32_t r = 0; r < c.size; ++r) {
      const uint4* pp = sb + ((size_t(r) * kTpSmallRows + row) * hidden + 4 * size_t(col)) / 2;
      const float4 a = tp_take_pairs(mine, pp, ld_pairs(pp), ld_pairs(pp + 1), ep32);
      v.x += a.x; v.y += a.y; v.z += a.z; v.w += a.w;
    }
    reinterpret_cast<float4*>(x_out)[i] = v;
  }
}

// ---------------------------------------------------------------- pull kernels ---------------
__device__ __forceinline__ float4 ld_peer_f4(const float4* p) { return ld_pushed_f4(p); }

// x[i] += sum_r region_r[off + i]   for i in [0, n)   (n multiple of 4)
__global__ void __launch_bounds__(512)
allreduce_add_kernel(TpCtx P, uint64_t off, float* __restrict__ x, uint64_t n) {
  ar_barrier(P);
  const uint64_t n4 = n / 4;
  for (uint64_t i = uint64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n4;
       i += uint64_t(gridDim.x) * blockDim.x) {
    float4 acc = reinterpret_cast<float4*>(x)[i];
#pragma unroll
    for (int r = 0; r < kTpMaxRanks; ++r) {
      if (r < int(P.size)) {
        float4 v = ld_peer_f4(reinterpret_cast<const float4*>(P.base[r] + off) + i);
        acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
      }
    }
    reinterpret_cast<float4*>(x)[i] = acc;
  }
}

// out[row, r*cols_local + c] = region_r[off][row, c]   (gathers vocab-sharded logits on every rank)
__global__ void __launch_bounds__(512)
allgather_cols_kernel(TpCtx P, uint64_t off, float* __restrict__ out, uint32_t rows, uint32_t cols_local) {
  ar_barrier(P);
  const uint32_t c4 = cols_local / 4;
  const uint64_t total = uint64_t(rows) * P.size * c4;
  for (uint64_t i = uint64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
       i += uint64_t(gridDim.x) * blockDim.x) {
    uint32_t c = uint32_t(i % c4);
    uint64_t t = i / c4;
    uint32_t r = uint32_t(t % P.size);
    uint32_t row = uint32_t(t / P.size);
    float4 v = ld_peer_f4(reinterpret_cast<const float4*>(P.base[r] + off) + size_t(row) * c4 + c);
    reinterpret_cast<float4*>(out + (size_t(row) * P.size + r) * cols_local)[c] = v;
  }
}

// ---------------------------------------------------------------- host side ------------------
int tp_step_begin(const TpCtx& c, cudaStream_t st) {
  tp_step_begin_kernel<<<1, 1, 0, st>>>(c);
  LLMLB_LAUNCH_CHECK();
  return LLMLB_OK;
}

int tp_reduce_norm(const TpCtx& c, uint32_t coll, float* x, const void* gain, uint32_t n_tokens, uint32_t hidden,
                   float eps, uint32_t split_k, bool wait_ag, bool ll, cudaStream_t st) {
  const uint32_t rpr = (n_tokens + c.size - 1) / c.size;
  const uint32_t lo = c.rank * rpr;
  const uint32_t n_own = lo >= n_tokens ? 0u : (n_tokens - lo < rpr ? n_tokens - lo : rpr);
  // programmatic dependent launch WITHOUT a dependency wait in the kernel: everything it reads arrives by
  // flag (the local rank's partials included), it writes nothing the producer GEMM or anything before it
  // still reads, and its done[] counters are its own — so it may sit on the SMs, polling, while the GEMM drains
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(n_own ? n_own : 1u);
  // one element group (4 values) per thread where the row allows it: every load of a row is in flight at once
  uint32_t threads = ((hidden / 4 + 31) / 32) * 32;
  if (threads > 1024) threads = 1024;
  if (threads < 64) threads = 64;
  cfg.blockDim = dim3(threads);
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  if (ll)
    LLMLB_CUDA_CHECK(cudaLaunchKernelEx(&cfg, tp_reduce_norm_kernel<true>, c, coll, x, (const __nv_bfloat16*)gain, n_tokens, rpr, n_own,
                                        hidden, eps, c.size * split_k, wait_ag ? 1u : 0u));
  else
    LLMLB_CUDA_CHECK(cudaLaunchKernelEx(&cfg, tp_reduce_norm_kernel<false>, c, coll, x, (const __nv_bfloat16*)gain, n_tokens, rpr, n_own,
                                        hidden, eps, c.size * split_k, wait_ag ? 1u : 0u));
  LLMLB_LAUNCH_CHECK();
  return LLMLB_OK;
}

int tp_push_rows(const TpCtx& c, uint32_t coll, const float* partial, uint32_t rows, uint32_t hidden, cudaStream_t st) {
  uint32_t blocks = (rows * hidden / 4 + 255) / 256;
  if (blocks > 32) blocks = 32;
  tp_push_rows_kernel<<<blocks, 256, 0, st>>>(c, coll, partial, rows, hidden);
  LLMLB_LAUNCH_CHECK();
  return LLMLB_OK;
}
int tp_fold_rows(const TpCtx& c, uint32_t coll, const float* x_in, float* x_out, uint32_t rows, uint32_t hidden, cudaStream_t st) {
  uint32_t blocks = (rows * hidden / 4 + 255) / 256;
  if (blocks > 32) blocks = 32;
  tp_fold_rows_kernel<<<blocks, 256, 0, st>>>(c, coll, x_in, x_out, rows, hidden);
  LLMLB_LAUNCH_CHECK();
  return LLMLB_OK;
}

int ar_allreduce_add(const TpCtx& P, uint64_t off, float* x, uint64_t n, cudaStream_t st) {
  uint32_t blocks = (uint32_t)((n / 4 + 511) / 512);
  if (blocks > (uint32_t)kArMaxBlocks) blocks = kArMaxBlocks;
  if (blocks < 1) blocks = 1;
  allreduce_add_kernel<<<blocks, 512, 0, st>>>(P, off, x, n);
  LLMLB_LAUNCH_CHECK();
  return LLMLB_OK;
}
int ar_allgather_cols(const TpCtx& P, uint64_t off, float* out, uint32_t rows, uint32_t cols_local, cudaStream_t st) {
  uint64_t total = uint64_t(rows) * P.size * (cols_local / 4);
  uint32_t blocks = (uint32_t)((total + 511) / 512);
  if (blocks > (uint32_t)kArMaxBlocks) blocks = kArMaxBlocks;
  if (blocks < 1) blocks = 1;
  allgather_cols_kernel<<<blocks, 512, 0, st>>>(P, off, out, rows, cols_local);
  LLMLB_LAUNCH_CHECK();
  return LLMLB_OK;
}

}  // namespace llmlb
