// Tensor-parallel exchange over NVLink peer memory: shared layout + device helpers (SURVEY §8 a2.13/e).
//
// Every rank owns ONE CUDA-IPC-shared exchange region, mapped into all peers:
//
//   [ ArSignals | TpFlags | slot 0 | slot 1 | pair slot 0 | pair slot 1 | rs-pair slot 0 | rs-pair slot 1 |
//     logits slot | y (bf16 activations, t_cap x hidden) ]
//
// Two protocols, both PUSH based (a producer stores into its peers' memory; nobody ever reads
// remote memory, so a consumer only pays local L2 latency once the data has landed):
//
//  A  "one-shot push", T <= 4 rows (decode).  The O / down projection GEMV stores every fp32
//     partial value together with the collective's 32-bit epoch as ONE 8-byte {value, epoch} pair
//     into pair slot[coll & 1][src = my rank] of EVERY rank.  8-byte stores are single-copy atomic,
//     so a consumer that reads a pair carrying its epoch has the value: no fence, no ticket, no
//     flag.  The CONSUMER is the next projection's RMSNorm prologue (gate/up, next QKV, lm_head):
//     every CTA spins on the epochs of the pairs, folds the N partials into the replicated fp32
//     residual in rank order (bit-identical on every rank) and normalises — no separate all-reduce
//     kernel, no barrier round trip.
//
//  B  "reduce-scatter + all-gather", T > 4 rows (prefill, batched decode).  Token rows are dealt
//     to owner ranks in chunks of rpr = ceil(T / N).  The O / down projection GEMM's epilogue
//     stores each partial tile row, as bf16, straight into the OWNER's slot (reduce-scatter by
//     address).  Wide steps (T > kTpLLTokens) write slot[.][part][row] and the last CTA raises
//     push_flag on every rank; narrow steps write {bf16 x 2, epoch} words into the rs-pair slot and
//     raise no flag.  tp_reduce_norm_kernel, one CTA per owned row: waits for the N flags (or the
//     words' epochs), x[row] += sum of the partials (the residual is row-sharded: only the owner
//     keeps it), RMSNorm, and stores the bf16 row into the `y` buffer of EVERY rank (all-gather by
//     address); the last CTA raises ag_flag everywhere.  The GEMM that consumes y waits for the
//     N ag_flags in its TMA producer (tp_wait_ag_single); for any other consumer the reduce kernel's
//     CTA 0 does not exit before all N ag_flags arrived, so the kernel boundary orders the loads.
//
// Flags hold 64-bit epochs, never reset: epoch = (step << 12) | (collective index within the step + 1),
// `step` is bumped by tp_step_begin_kernel at the start of every forward pass, identically on all
// ranks (they launch identical steps).  Pairs carry the 32-bit form (tp_epoch32).  Slots alternate
// per collective; a rank can never be more than one collective ahead of a peer (it needs the peer's
// push to finish its own consumer), so two slots suffice.  Slot 0 also serves the standalone pull
// all-reduce (llmlb_op_allreduce).
#pragma once
#include <stdint.h>

#include "common.cuh"

namespace llmlb {

constexpr int kTpMaxRanks = 8;
constexpr int kTpSlots = 2;
constexpr int kTpSmallRows = 4;       // protocol A rows per source in a slot

struct TpFlags {
  // written by peers (system-scope release stores), read locally with acquire loads
  unsigned long long push_flag[kTpSlots][kTpMaxRanks];  // [slot][src]: src finished pushing partials into my slot
  unsigned long long ag_flag[kTpSlots][kTpMaxRanks];    // [slot][owner]: owner finished pushing its y rows to me
  // local only
  unsigned long long step;          // forward passes started so far (tp_step_begin_kernel)
  unsigned int done[4];             // last-CTA counters: [coll & 1] producers, [2 + (coll & 1)] reduce_norm
  unsigned int timed_out;           // set before a spin gives up and traps (dead peer)
};
constexpr size_t kTpFlagBytes = (sizeof(TpFlags) + 255) & ~size_t(255);

struct TpCtx {                      // kernel parameter, by value
  uint8_t* base[kTpMaxRanks];       // exchange region of every rank (peer-mapped)
  uint32_t rank, size;
  uint64_t flags_off;               // TpFlags
  uint64_t slot_off[kTpSlots];      // protocol B, wide steps: bf16 partials of the reduce-scatter [part][row][hidden]
  uint64_t ll_off[kTpSlots];        // protocol A: {value, epoch} pairs [src][kTpSmallRows][hidden] (never written by
                                    // anything else, so a stale word can only be an older epoch)
  uint64_t rsll_off[kTpSlots];      // protocol B, narrow steps: {bf16 x 2, epoch} words of the reduce-scatter
                                    // [part][row of the owner][hidden / 2] (never written by anything else)
  uint64_t y_off;                   // bf16 [t_cap, hidden] normalised activations
  uint64_t slot_bytes;
};

#ifdef __CUDACC__
__device__ __forceinline__ void st_release_sys_u64(unsigned long long* p, unsigned long long v) {
  asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ld_acquire_sys_u64(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ unsigned long long ld_relaxed_sys_u64(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.relaxed.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
// data pushed by a peer: never through L1 (a stale line from the slot's previous use may sit there)
__device__ __forceinline__ float4 ld_pushed_f4(const float4* p) {
  float4 v;
  asm volatile("ld.relaxed.sys.global.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
               : "l"(p)
               : "memory");
  return v;
}
__device__ __forceinline__ void st_peer_bf16(__nv_bfloat16* p, float v) {   // reduce-scatter partials travel as bf16
  const unsigned short b = __bfloat16_as_ushort(__float2bfloat16_rn(v));
  asm volatile("st.relaxed.sys.global.u16 [%0], %1;" ::"l"(p), "h"(b) : "memory");
}
__device__ __forceinline__ uint2 ld_pushed_u2(const uint2* p) {
  uint2 v;
  asm volatile("ld.relaxed.sys.global.v2.u32 {%0,%1}, [%2];" : "=r"(v.x), "=r"(v.y) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_peer_u2(void* p, uint2 v) {
  asm volatile("st.relaxed.sys.global.v2.u32 [%0], {%1,%2};" ::"l"(p), "r"(v.x), "r"(v.y) : "memory");
}
// ---- protocol A: every pushed value travels with its epoch in ONE 8-byte store {value bits, epoch32}:
// the push is visible one NVLink flight after the producing lane computed it.  Costs 2x the (tiny)
// bytes on the wire.
__device__ __forceinline__ void st_peer_pair(void* p, float v, uint32_t epoch) {
  asm volatile("st.relaxed.sys.global.v2.u32 [%0], {%1,%2};" ::"l"(p), "r"(__float_as_uint(v)), "r"(epoch) : "memory");
}
__device__ __forceinline__ uint4 ld_pairs(const uint4* p) {   // two {value, epoch} pairs
  uint4 v;
  asm volatile("ld.relaxed.sys.global.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ TpFlags* tp_flags(const TpCtx& c, uint32_t r) {
  return reinterpret_cast<TpFlags*>(c.base[r] + c.flags_off);
}
// read AFTER the kernel's dependency wait: tp_step_begin_kernel of this step has completed
__device__ __forceinline__ unsigned long long tp_epoch(const TpCtx& c, uint32_t coll) {
  return (ld_relaxed_sys_u64(&tp_flags(c, c.rank)->step) << 12) | (unsigned long long)(coll + 1);
}
// never 0 (slots start zeroed); equality is the test, so wrap-around after 2^24 steps is harmless:
// a slot is rewritten every second collective
__device__ __forceinline__ uint32_t tp_epoch32(const TpCtx& c, uint32_t coll) {
  return (uint32_t(ld_relaxed_sys_u64(&tp_flags(c, c.rank)->step)) << 8) | (coll + 1);
}
// four values of one source row whose pairs sit at p[0], p[1]: spin until all four carry `epoch`
__device__ __forceinline__ float4 tp_take_pairs(TpFlags* mine, const uint4* p, uint4 a, uint4 b, uint32_t epoch) {
  if (a.y != epoch || a.w != epoch || b.y != epoch || b.w != epoch) {
    const unsigned long long t0 = gtime_ns();
    unsigned int spins = 0;
    do {
      a = ld_pairs(p); b = ld_pairs(p + 1);
      if ((++spins & 0xFFFu) == 0 && gtime_ns() - t0 > 20000000000ull) {
        mine->timed_out = 1;
        __threadfence_system();
        __trap();
      }
    } while (a.y != epoch || a.w != epoch || b.y != epoch || b.w != epoch);
  }
  return make_float4(__uint_as_float(a.x), __uint_as_float(a.z), __uint_as_float(b.x), __uint_as_float(b.z));
}
// Threads 0..size-1 of the CTA each wait for one flag; then the CTA barriers.  A peer that never
// arrives (crashed process) must not hang the GPU forever: after ~20 s the kernel records the
// fact and traps, which surfaces as a CUDA error in the engine instead of a dead device.
__device__ __forceinline__ void tp_wait_flags(TpFlags* mine, const unsigned long long* flags, uint32_t size,
                                              unsigned long long epoch) {
  if (threadIdx.x < size) {
    const unsigned long long* f = flags + threadIdx.x;
    if (ld_acquire_sys_u64(f) < epoch) {
      const unsigned long long t0 = gtime_ns();
      unsigned int spins = 0;
      while (ld_acquire_sys_u64(f) < epoch) {
        if ((++spins & 0xFFFu) == 0 && gtime_ns() - t0 > 20000000000ull) {
          mine->timed_out = 1;
          __threadfence_system();
          __trap();
        }
      }
    }
  }
  __syncthreads();
}
// ONE thread (the TMA producer of a GEMM that consumes y) waits until every owner's rows of
// collective `coll` have landed in this rank's y, then orders the tensor-map (async proxy) reads
// behind what it observed.
__device__ __forceinline__ void tp_wait_ag_single(const TpCtx& c, uint32_t coll) {
  TpFlags* mine = tp_flags(c, c.rank);
  const unsigned long long epoch = tp_epoch(c, coll);
  const unsigned long long t0 = gtime_ns();
  unsigned int spins = 0;
  // the N flag loads of one round are independent (relaxed) and in flight together: one L2 round trip per
  // round instead of N; the acquire is the fence after the last round
  for (;;) {
    bool all = true;
#pragma unroll
    for (uint32_t r = 0; r < uint32_t(kTpMaxRanks); ++r)
      if (r < c.size) all &= ld_relaxed_sys_u64(&mine->ag_flag[coll & 1][r]) >= epoch;
    if (all) break;
    if ((++spins & 0xFFFu) == 0 && gtime_ns() - t0 > 20000000000ull) {
      mine->timed_out = 1;
      __threadfence_system();
      __trap();
    }
  }
  asm volatile("fence.acq_rel.sys;" ::: "memory");
  asm volatile("fence.proxy.async.global;" ::: "memory");
}
// Every thread of every CTA of the grid calls this after its last push.  When the whole grid is
// through, threads 0..size-1 of the last CTA raise `flag_of(peer)` = epoch on every rank.
// (CTA barrier -> thread 0: fence.sys, ticket, fence.sys -> CTA barrier -> release stores: the
// pushes of all CTAs happen-before the flag at system scope.)
template <class FlagOf>
__device__ __forceinline__ void tp_signal_when_grid_done(const TpCtx& c, unsigned int* done, uint32_t n_ctas,
                                                         unsigned long long epoch, FlagOf flag_of) {
  __shared__ unsigned int s_last;
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence_system();         // this CTA's pushes are performed system-wide before its ticket is taken
    const unsigned int old = atomicAdd(done, 1u);
    const unsigned int last = (old == n_ctas - 1) ? 1u : 0u;
    if (last) *done = 0;            // the next user of this counter is ordered after this kernel
    s_last = last;
  }
  __syncthreads();
  // the release stores below are themselves fences for what the last CTA observed (the other CTAs'
  // tickets, each taken after that CTA's own system fence): no second full fence on every CTA
  if (s_last && threadIdx.x < c.size) st_release_sys_u64(flag_of(tp_flags(c, threadIdx.x)), epoch);
}
#endif

// ---- host-side entry points (tp_exchange.cu) ----
size_t tp_region_prefix_bytes();      // ArSignals + TpFlags
int tp_step_begin(const TpCtx& c, cudaStream_t st);
// fallbacks of protocol A for projection shapes the fused GEMV does not take
int tp_push_rows(const TpCtx& c, uint32_t coll, const float* partial, uint32_t rows, uint32_t hidden, cudaStream_t st);
int tp_fold_rows(const TpCtx& c, uint32_t coll, const float* x_in, float* x_out, uint32_t rows, uint32_t hidden, cudaStream_t st);
// protocol B consumer
// wait_ag: the grid does not end before every owner's rows arrived here (for consumers of y that are
// not tensor-core GEMMs; those wait for the flags themselves: TpPushRS::wait_coll_plus1)
int tp_reduce_norm(const TpCtx& c, uint32_t coll, float* x, const void* gain, uint32_t n_tokens, uint32_t hidden,
                   float eps, uint32_t split_k, bool wait_ag, bool ll, cudaStream_t st);

}  // namespace llmlb
