// RoPE + paged-KV append + attention (SURVEY §8 a2.4-a2.7).
//
// KV pages: K and V pools are [page][kv_head][64 tokens][128] bf16, so one (page, head) is a
// contiguous 16 KiB run — the unit the decode kernel streams and the prefill kernel stages.
// RoPE uses a precomputed fp32 (cos,sin) table [position][64] (HF rotate-half pairing i, i+64).
//
//  * rope_append_kernel       prefill: rotate q,k in place in the qkv activation, write k,v pages
//                             (prefill attention itself runs on tcgen05: attention_tc.cu)
//  * decode_attention_kernel  one new token per sequence: rotate q,k, append k,v, split-KV
//                             attention over the pages (HBM-bound: ctx*2*128*2 B per kv head),
//                             the cluster leader merges the splits through DSMEM
//  * decode_attention_mma_kernel  wide batches, no split: one warp per (sequence, head group),
//                             mma.sync m16n8k16 over K/V staged by cp.async
#include "../../include/llmlb_b200.h"
#include "common.cuh"

namespace llmlb {

constexpr float kLog2e = 1.4426950408889634f;

__global__ void rope_table_kernel(float2* __restrict__ table, uint32_t max_pos, double theta) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= max_pos * 64) return;
  uint32_t pos = i / 64, j = i % 64;
  double inv = pow(theta, -double(2 * j) / double(kHeadDim));
  double a = double(pos) * inv;
  table[i] = make_float2(float(cos(a)), float(sin(a)));
}

// ------------------------------------------------------------------ prefill rope + append ---
__global__ void __launch_bounds__(256)
rope_append_kernel(__nv_bfloat16* __restrict__ qkv, const int32_t* __restrict__ positions,
                   const int32_t* __restrict__ page_of_token, const float2* __restrict__ rope,
                   __nv_bfloat16* __restrict__ k_pages, __nv_bfloat16* __restrict__ v_pages,
                   uint32_t n_heads, uint32_t n_kv, uint32_t pdl) {
  // programmatic dependent launch: the attention kernel behind may set itself up now; this grid
  // may itself have been scheduled before the QKV projection finished
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  if (pdl) asm volatile("griddepcontrol.wait;" ::: "memory");
  const uint32_t t = blockIdx.x;
  const uint32_t width = (n_heads + 2 * n_kv) * kHeadDim;
  __nv_bfloat16* row = qkv + size_t(t) * width;
  const int32_t pos = positions[t];
  const int32_t page = page_of_token[t];
  const uint32_t slot = uint32_t(pos) % kPageTokens;
  const float2* cs = rope + size_t(pos) * 64;
  // rotate q heads then k heads: pair (i, i+64) within each head
  const uint32_t n_rot = (n_heads + n_kv) * 64;
  for (uint32_t p = threadIdx.x; p < n_rot; p += blockDim.x) {
    uint32_t h = p / 64, i = p % 64;
    float2 c = cs[i];
    __nv_bfloat16* hp = row + size_t(h) * kHeadDim;
    float a = __bfloat162float(hp[i]), b = __bfloat162float(hp[i + 64]);
    __nv_bfloat16 ra = __float2bfloat16_rn(a * c.x - b * c.y);
    __nv_bfloat16 rb = __float2bfloat16_rn(b * c.x + a * c.y);
    hp[i] = ra;
    hp[i + 64] = rb;
    if (h >= n_heads && page >= 0) {
      uint32_t kh = h - n_heads;
      __nv_bfloat16* dst =
          k_pages + ((size_t(page) * n_kv + kh) * kPageTokens + slot) * kHeadDim;
      dst[i] = ra;
      dst[i + 64] = rb;
    }
  }
  if (page >= 0) {
    const __nv_bfloat16* vrow = row + size_t(n_heads + n_kv) * kHeadDim;
    for (uint32_t p = threadIdx.x; p < n_kv * kHeadDim / 8; p += blockDim.x) {
      uint32_t kh = p / 16, c = p % 16;
      uint4 v = reinterpret_cast<const uint4*>(vrow + size_t(kh) * kHeadDim)[c];
      reinterpret_cast<uint4*>(v_pages +
                               ((size_t(page) * n_kv + kh) * kPageTokens + slot) * kHeadDim)[c] = v;
    }
  }
}

// ------------------------------------------------------------------ mma.sync / cp.async / DSMEM helpers ---
__device__ __forceinline__ void cp_async16(void* smem, const void* gmem, bool valid) {
  uint32_t s = (uint32_t)__cvta_generic_to_shared(smem);
  int sz = valid ? 16 : 0;
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(s), "l"(gmem), "r"(sz));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;" ::"n"(N));
}
__device__ __forceinline__ void ldmatrix_x4(uint32_t (&r)[4], const void* p) {
  uint32_t s = (uint32_t)__cvta_generic_to_shared(p);
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
               : "r"(s));
}
__device__ __forceinline__ void ldmatrix_x4_trans(uint32_t (&r)[4], const void* p) {
  uint32_t s = (uint32_t)__cvta_generic_to_shared(p);
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
               : "r"(s));
}
__device__ __forceinline__ void mma_bf16_16816(float (&c)[4], const uint32_t (&a)[4], uint32_t b0,
                                               uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, "
      "{%8,%9}, {%0,%1,%2,%3};"
      : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
// tile of 64 rows x 128 bf16 (256 B rows, 16 chunks of 16 B); chunk index xor (row & 7)
__device__ __forceinline__ uint32_t swz(uint32_t row, uint32_t chunk) {
  return row * 128 + ((chunk ^ (row & 7)) << 3);  // element offset
}

__device__ __forceinline__ uint32_t smem_addr_u32(const void* p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}
// read a float / float4 at shared-memory offset `addr` of cluster CTA `rank` (DSMEM)
__device__ __forceinline__ float ld_dsmem_f32(uint32_t addr, uint32_t rank) {
  uint32_t ra;
  float v;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(ra) : "r"(addr), "r"(rank));
  asm volatile("ld.shared::cluster.f32 %0, [%1];" : "=f"(v) : "r"(ra));
  return v;
}
__device__ __forceinline__ float4 ld_dsmem_f4(uint32_t addr, uint32_t rank) {
  uint32_t ra;
  float4 v;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(ra) : "r"(addr), "r"(rank));
  asm volatile("ld.shared::cluster.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
               : "r"(ra));
  return v;
}

__device__ __forceinline__ uint32_t dsmem_addr(uint32_t addr, uint32_t rank) {
  uint32_t ra;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(ra) : "r"(addr), "r"(rank));
  return ra;
}
__device__ __forceinline__ void st_dsmem_f4(uint32_t ra, float4 v) {
  asm volatile("st.shared::cluster.v4.f32 [%0], {%1,%2,%3,%4};" ::"r"(ra), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ void st_dsmem_f32(uint32_t ra, float v) {
  asm volatile("st.shared::cluster.f32 [%0], %1;" ::"r"(ra), "f"(v) : "memory");
}

// ------------------------------------------------------------------ decode attention --------
// One CTA per (sequence, group of 4 q heads, KV split); the n_splits CTAs of a (sequence, head
// group) form a thread-block CLUSTER: every CTA reduces its slice of the context to (m, l, o)
// in shared memory, then rank 0 pulls the partials of its peers through distributed shared
// memory and writes the bf16 output — no global workspace, no atomics, no second kernel.
// K/V rows are prefetched 64 tokens (one page) ahead: 16 x 16-byte loads per lane in flight.
constexpr int kDecHeads = 4;     // q heads per CTA (all share one kv head)
constexpr int kDecThreads = 128;

static __device__ TraceBuf d_trace_attn;
void attn_set_trace(const TraceBuf& tb) { cudaMemcpyToSymbol(d_trace_attn, &tb, sizeof(tb)); }

struct DecPartial {               // per-CTA result, read by the cluster leader
  float o[kDecHeads][kHeadDim];
  float m[kDecHeads];
  float l[kDecHeads];
};

__global__ void __launch_bounds__(kDecThreads)
decode_attention_kernel(const __nv_bfloat16* qkv /* NOT __restrict__: written by the predecessor grid while this one may
                                                           already be resident (programmatic launch) — with restrict + const
                                                           the compiler hoisted four q loads above griddepcontrol.wait as
                                                           LDG.CONSTANT (SASS, round 2) and the kernel read the previous
                                                           layer's rows */,
                        __nv_bfloat16* k_pages,
                        __nv_bfloat16* v_pages, const int32_t* __restrict__ block_tables,
                        uint32_t bt_stride, const int32_t* __restrict__ bt_rows,
                        const int32_t* __restrict__ seq_lens,
                        const float2* __restrict__ rope, __nv_bfloat16* __restrict__ out,
                        uint32_t n_heads, uint32_t n_kv, uint32_t n_splits) {
  __shared__ float q_s[kDecHeads][kHeadDim];
  __shared__ float kv_new[2][kHeadDim];  // rotated k and v of the new token (owner CTA only)
  __shared__ float mrg_o[4][kDecHeads][kHeadDim];
  __shared__ float mrg_ml[4][kDecHeads][2];
  __shared__ DecPartial parts[16];  // only the cluster leader's copy is filled (peers push into it)

  const TraceBuf tb = d_trace_attn;
  unsigned long long tr0 = 0, tr1 = 0, tr2 = 0;
  if (tb.data && threadIdx.x == 0) tr0 = gtime_ns();
  // PDL: the O-projection GEMV that follows may start prefetching its weights now
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  // cluster phase 1 (arrive now, wait just before the first DSMEM store): every CTA has started
  if (n_splits > 1) asm volatile("barrier.cluster.arrive.relaxed.aligned;" ::: "memory");
  const uint32_t z = blockIdx.x, hb = blockIdx.y, s = blockIdx.z;
  const uint32_t h0 = hb * kDecHeads, kvh = h0 / (n_heads / n_kv);
  const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const uint32_t width = (n_heads + 2 * n_kv) * kHeadDim;
  const int32_t L = seq_lens[s];  // includes the new token
  const int32_t* bt = block_tables + size_t(bt_rows ? bt_rows[s] : int32_t(s)) * bt_stride;
  const uint32_t pos = uint32_t(L - 1);
  const float2* cs = rope + size_t(pos) * 64;
  const __nv_bfloat16* row = qkv + size_t(s) * width;

  const uint32_t n_pages = (uint32_t(L) + kPageTokens - 1) / kPageTokens;
  const uint32_t pages_per_split = (n_pages + n_splits - 1) / n_splits;
  const uint32_t p_begin = z * pages_per_split;
  const uint32_t p_end = min(n_pages, p_begin + pages_per_split);
  const uint32_t t_begin = p_begin * kPageTokens;
  const uint32_t t_end = min(uint32_t(L), p_end * kPageTokens);
  // ---- before the dependency wait: everything that does not read this step's qkv ----
  // (seq_lens / block tables were written at the start of the step; old K/V long before)
  const uint32_t grp = lane >> 3, sub = lane & 7;
  int32_t page_next = (p_begin < p_end) ? bt[p_begin] : 0;
  uint4 kq[4][2], vq[4][2];
  auto load_page = [&](int32_t page) {
    const size_t pbase = (size_t(page) * n_kv + kvh) * kPageTokens * kHeadDim + sub * 16;
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      const size_t off = pbase + size_t(r * 16 + warp * 4 + grp) * kHeadDim;
      kq[r][0] = *reinterpret_cast<const uint4*>(k_pages + off);
      kq[r][1] = *reinterpret_cast<const uint4*>(k_pages + off + 8);
      vq[r][0] = *reinterpret_cast<const uint4*>(v_pages + off);
      vq[r][1] = *reinterpret_cast<const uint4*>(v_pages + off + 8);
    }
  };
  if (p_begin < p_end) load_page(page_next);   // 16 x 16-byte loads per lane in flight
  const float2 cs_lane0 = cs[tid & 63];        // rope row of the new position
  asm volatile("griddepcontrol.wait;" ::: "memory");

  // rotate q (4 heads x 64 pairs = 256 pairs over 128 threads), pre-scaled for exp2
  const float scale = rsqrtf(float(kHeadDim)) * kLog2e;
#pragma unroll
  for (uint32_t p = tid; p < kDecHeads * 64; p += kDecThreads) {
    uint32_t h = p / 64, i = p % 64;
    float2 c = cs_lane0;  // p % 64 == tid % 64 for both trips (128 threads, stride 128)
    const __nv_bfloat16* hp = row + size_t(h0 + h) * kHeadDim;
    float a = __bfloat162float(hp[i]), b = __bfloat162float(hp[i + 64]);
    // round through bf16 like the prefill path (q is stored as bf16 there)
    float ra = __bfloat162float(__float2bfloat16_rn(a * c.x - b * c.y));
    float rb = __bfloat162float(__float2bfloat16_rn(b * c.x + a * c.y));
    q_s[h][i] = ra * scale;
    q_s[h][i + 64] = rb * scale;
  }
  // the CTA whose range holds the new position rotates k and appends k,v; the values it uses
  // for that token come from shared memory (the page was prefetched before they existed)
  const bool owns_new = (t_begin <= pos && pos < t_end);
  if (owns_new) {
    const int32_t page = bt[pos / kPageTokens];
    const uint32_t slot = pos % kPageTokens;
    __nv_bfloat16* kd = k_pages + ((size_t(page) * n_kv + kvh) * kPageTokens + slot) * kHeadDim;
    __nv_bfloat16* vd = v_pages + ((size_t(page) * n_kv + kvh) * kPageTokens + slot) * kHeadDim;
    const __nv_bfloat16* kp = row + size_t(n_heads + kvh) * kHeadDim;
    const __nv_bfloat16* vp = row + size_t(n_heads + n_kv + kvh) * kHeadDim;
    if (tid < 64) {
      float2 c = cs_lane0;
      float a = __bfloat162float(kp[tid]), b = __bfloat162float(kp[tid + 64]);
      __nv_bfloat16 ra = __float2bfloat16_rn(a * c.x - b * c.y), rb = __float2bfloat16_rn(b * c.x + a * c.y);
      kd[tid] = ra; kd[tid + 64] = rb;
      kv_new[0][tid] = __bfloat162float(ra); kv_new[0][tid + 64] = __bfloat162float(rb);
    } else {
      uint32_t i = tid - 64;
      __nv_bfloat16 v0 = vp[i], v1 = vp[i + 64];
      vd[i] = v0; vd[i + 64] = v1;
      kv_new[1][i] = __bfloat162float(v0); kv_new[1][i + 64] = __bfloat162float(v1);
    }
  }
  __syncthreads();
  if (tb.data && threadIdx.x == 0) tr1 = gtime_ns();

  // each 8-lane group walks its own token stream; lane owns 16 dims
  float q_r[kDecHeads][16];
#pragma unroll
  for (int h = 0; h < kDecHeads; ++h)
#pragma unroll
    for (int d = 0; d < 16; ++d) q_r[h][d] = q_s[h][sub * 16 + d];
  float acc[kDecHeads][16];
  float m_r[kDecHeads], l_r[kDecHeads];
#pragma unroll
  for (int h = 0; h < kDecHeads; ++h) {
    m_r[h] = -INFINITY;
    l_r[h] = 0.f;
#pragma unroll
    for (int d = 0; d < 16; ++d) acc[h][d] = 0.f;
  }

  for (uint32_t pg = p_begin; pg < p_end; ++pg) {
    if (pg != p_begin) load_page(page_next);          // first page is already in registers
    if (pg + 1 < p_end) page_next = bt[pg + 1];
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      const uint32_t tok = pg * kPageTokens + r * 16 + warp * 4 + grp;
      const bool valid = tok < t_end;
      float kf[16], vf[16];
      if (tok == pos) {
#pragma unroll
        for (int d = 0; d < 16; ++d) { kf[d] = kv_new[0][sub * 16 + d]; vf[d] = kv_new[1][sub * 16 + d]; }
      } else {
        const uint32_t kw[8] = {kq[r][0].x, kq[r][0].y, kq[r][0].z, kq[r][0].w,
                                kq[r][1].x, kq[r][1].y, kq[r][1].z, kq[r][1].w};
        const uint32_t vw[8] = {vq[r][0].x, vq[r][0].y, vq[r][0].z, vq[r][0].w,
                                vq[r][1].x, vq[r][1].y, vq[r][1].z, vq[r][1].w};
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          kf[2 * i] = bf16_lo(kw[i]); kf[2 * i + 1] = bf16_hi(kw[i]);
          vf[2 * i] = bf16_lo(vw[i]); vf[2 * i + 1] = bf16_hi(vw[i]);
        }
      }
#pragma unroll
      for (int h = 0; h < kDecHeads; ++h) {
        float sc = 0.f;
#pragma unroll
        for (int d = 0; d < 16; ++d) sc = fmaf(q_r[h][d], kf[d], sc);
        sc += __shfl_xor_sync(0xffffffffu, sc, 1);
        sc += __shfl_xor_sync(0xffffffffu, sc, 2);
        sc += __shfl_xor_sync(0xffffffffu, sc, 4);
        if (valid) {
          float mn = fmaxf(m_r[h], sc);
          float corr = exp2f(m_r[h] - mn);
          float p = exp2f(sc - mn);
          m_r[h] = mn;
          l_r[h] = l_r[h] * corr + p;
#pragma unroll
          for (int d = 0; d < 16; ++d) acc[h][d] = fmaf(p, vf[d], acc[h][d] * corr);
        }
      }
    }
  }

  if (tb.data && threadIdx.x == 0) tr2 = gtime_ns();
  // merge the 4 token groups of the warp (lanes with equal `sub`)
#pragma unroll
  for (int h = 0; h < kDecHeads; ++h) {
#pragma unroll
    for (int step = 8; step <= 16; step <<= 1) {
      float mo = __shfl_xor_sync(0xffffffffu, m_r[h], step);
      float lo = __shfl_xor_sync(0xffffffffu, l_r[h], step);
      float mn = fmaxf(m_r[h], mo);
      float ca = (m_r[h] == -INFINITY) ? 0.f : exp2f(m_r[h] - mn);
      float cb = (mo == -INFINITY) ? 0.f : exp2f(mo - mn);
#pragma unroll
      for (int d = 0; d < 16; ++d) {
        float ao = __shfl_xor_sync(0xffffffffu, acc[h][d], step);
        acc[h][d] = acc[h][d] * ca + ao * cb;
      }
      l_r[h] = l_r[h] * ca + lo * cb;
      m_r[h] = mn;
    }
  }
  if (grp == 0) {
#pragma unroll
    for (int h = 0; h < kDecHeads; ++h) {
#pragma unroll
      for (int d = 0; d < 16; ++d) mrg_o[warp][h][sub * 16 + d] = acc[h][d];
      if (sub == 0) {
        mrg_ml[warp][h][0] = m_r[h];
        mrg_ml[warp][h][1] = l_r[h];
      }
    }
  }
  __syncthreads();
  // merge the 4 warps: thread -> (head = tid/32, 4 dims)
  const uint32_t h = tid >> 5, d0 = (tid & 31) * 4;
  float mn = -INFINITY;
#pragma unroll
  for (int w = 0; w < 4; ++w) mn = fmaxf(mn, mrg_ml[w][h][0]);
  float l = 0.f, ov[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
  for (int w = 0; w < 4; ++w) {
    float mw = mrg_ml[w][h][0];
    float c = (mw == -INFINITY) ? 0.f : exp2f(mw - mn);
    l += mrg_ml[w][h][1] * c;
#pragma unroll
    for (int d = 0; d < 4; ++d) ov[d] += mrg_o[w][h][d0 + d] * c;
  }
  __nv_bfloat16* dst = out + size_t(s) * n_heads * kHeadDim + size_t(h0 + h) * kHeadDim + d0;
  if (n_splits == 1) {
    float inv = 1.f / l;
    uint2 o2;
    o2.x = pack_bf16(ov[0] * inv, ov[1] * inv);
    o2.y = pack_bf16(ov[2] * inv, ov[3] * inv);
    *reinterpret_cast<uint2*>(dst) = o2;
    return;
  }
  // push this CTA's partial into the LEADER's shared memory, one cluster barrier, peers leave
  asm volatile("barrier.cluster.wait.aligned;" ::: "memory");  // phase 1: leader's smem is live
  {
    const uint32_t slot = dsmem_addr(smem_addr_u32(&parts[z]), 0);
    st_dsmem_f4(slot + offsetof(DecPartial, o) + (h * kHeadDim + d0) * 4, make_float4(ov[0], ov[1], ov[2], ov[3]));
    if ((tid & 31) == 0) {
      st_dsmem_f32(slot + offsetof(DecPartial, m) + h * 4, mn);
      st_dsmem_f32(slot + offsetof(DecPartial, l) + h * 4, l);
    }
  }
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  if (z != 0) {
    if (tb.data && threadIdx.x == 0) trace_emit(tb, 1ull, tr0, tr1, tr2, gtime_ns());
    return;
  }
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
  {
    float gm = -INFINITY;
    for (uint32_t r = 0; r < n_splits; ++r) gm = fmaxf(gm, parts[r].m[h]);
    float gl = 0.f, go[4] = {0.f, 0.f, 0.f, 0.f};
    for (uint32_t r = 0; r < n_splits; ++r) {
      const float pm = parts[r].m[h];
      const float c = (pm == -INFINITY) ? 0.f : exp2f(pm - gm);
      gl += parts[r].l[h] * c;
      const float4 po = *reinterpret_cast<const float4*>(&parts[r].o[h][d0]);
      go[0] += po.x * c; go[1] += po.y * c; go[2] += po.z * c; go[3] += po.w * c;
    }
    const float inv = 1.f / gl;
    uint2 o2;
    o2.x = pack_bf16(go[0] * inv, go[1] * inv);
    o2.y = pack_bf16(go[2] * inv, go[3] * inv);
    *reinterpret_cast<uint2*>(dst) = o2;
  }
  if (tb.data && threadIdx.x == 0) trace_emit(tb, 1ull, tr0, tr1, tr2, gtime_ns());
}

}  // namespace llmlb

using namespace llmlb;

extern "C" int llmlb_op_rope_table(float* table, uint32_t max_pos, float theta, void* stream) {
  if (!table || max_pos == 0) {
    set_error("llmlb_op_rope_table: bad argument");
    return LLMLB_E_INVALID_ARG;
  }
  uint32_t n = max_pos * 64;
  rope_table_kernel<<<(n + 255) / 256, 256, 0, (cudaStream_t)stream>>>((float2*)table, max_pos,
                                                                       (double)theta);
  LLMLB_LAUNCH_CHECK();
  return LLMLB_OK;
}

namespace llmlb {
int rope_append_launch(void* qkv, const int32_t* positions, const int32_t* page_of_token, const float* rope_table,
                       void* k_pages, void* v_pages, uint32_t n_tokens, uint32_t n_heads, uint32_t n_kv, bool pdl,
                       cudaStream_t st) {
  if (n_tokens == 0) return LLMLB_OK;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(n_tokens);
  cfg.blockDim = dim3(256);
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl ? 1 : 0;
  LLMLB_CUDA_CHECK(cudaLaunchKernelEx(&cfg, rope_append_kernel, (__nv_bfloat16*)qkv, positions, page_of_token,
                                      (const float2*)rope_table, (__nv_bfloat16*)k_pages, (__nv_bfloat16*)v_pages, n_heads, n_kv,
                                      pdl ? 1u : 0u));
  LLMLB_LAUNCH_CHECK();
  return LLMLB_OK;
}
}  // namespace llmlb

extern "C" int llmlb_op_rope_append(void* qkv, const int32_t* positions,
                                    const int32_t* page_of_token, const float* rope_table,
                                    void* k_pages, void* v_pages, uint32_t n_tokens,
                                    uint32_t n_heads, uint32_t n_kv, void* stream) {
  if (!qkv || !positions || !page_of_token || !rope_table || !k_pages || !v_pages) {
    set_error("llmlb_op_rope_append: null argument");
    return LLMLB_E_INVALID_ARG;
  }
  return rope_append_launch(qkv, positions, page_of_token, rope_table, k_pages, v_pages, n_tokens, n_heads, n_kv, false,
                            (cudaStream_t)stream);
}

extern "C" size_t llmlb_op_decode_attention_ws(uint32_t, uint32_t, uint32_t) {
  return 256;  // kept for ABI stability: the split merge now happens in cluster shared memory
}

namespace llmlb {

// ------------------------------------------------------------------ decode attention, batched ---
// Wide batches (no KV split): one WARP per (sequence, group of 4 q heads).  The 4 heads are rows
// 0..3 of a 16-row mma.sync tile (rows 4..15 are zero), K/V pages are staged by cp.async into a
// double-buffered shared-memory ring (next page in flight while the tensor cores work on this
// one), so the kernel is bound by the K/V stream instead of by SIMT dot products
// (round-1 profile at 64 streams: SIMT kernel 69 us/layer for 136 MB of K/V = 2 TB/s).
constexpr int kDamThreads = 32;
// K/V move through a 3-stage ring of 32-token half pages: 48 KiB + q per CTA, so FOUR one-warp CTAs
// share an SM and the 512 CTAs of a 64-stream step are resident at once (with whole pages and
// two stages only three fit: a second, mostly empty wave doubled the kernel's time — ncu,
// profiles/r1_decode_attn_mma_ncu_full.txt)
constexpr int kDamChunk = 32;
constexpr int kDamStages = 3;
constexpr int kDamSmem = kDamStages * 2 * kDamChunk * kHeadDim * 2 + kDecHeads * kHeadDim * 2;

__global__ void __launch_bounds__(kDamThreads)
decode_attention_mma_kernel(const __nv_bfloat16* __restrict__ qkv, __nv_bfloat16* k_pages,
                            __nv_bfloat16* v_pages, const int32_t* __restrict__ block_tables,
                            uint32_t bt_stride, const int32_t* __restrict__ bt_rows,
                            const int32_t* __restrict__ seq_lens, const float2* __restrict__ rope,
                            __nv_bfloat16* __restrict__ out, uint32_t n_heads, uint32_t n_kv, uint32_t trigger) {
  extern __shared__ __align__(128) uint8_t dam_smem[];
  // a PDL-launched successor (the O projection) may take the SMs this grid frees and start on its weights
  if (trigger) asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  __nv_bfloat16* sk = reinterpret_cast<__nv_bfloat16*>(dam_smem);            // [3][32][128] swizzled
  __nv_bfloat16* sv = sk + kDamStages * kDamChunk * kHeadDim;                // [3][32][128] swizzled
  __nv_bfloat16* sq = sv + kDamStages * kDamChunk * kHeadDim;                // [4][128] rotated q (bf16)
  __shared__ __align__(16) __nv_bfloat16 s_knew[kHeadDim];
  __shared__ __align__(16) __nv_bfloat16 s_vnew[kHeadDim];

  const uint32_t hb = blockIdx.x, s = blockIdx.y, lane = threadIdx.x;
  const uint32_t h0 = hb * kDecHeads, kvh = h0 / (n_heads / n_kv);
  const uint32_t width = (n_heads + 2 * n_kv) * kHeadDim;
  const int32_t L = seq_lens[s];
  const int32_t* bt = block_tables + size_t(bt_rows ? bt_rows[s] : int32_t(s)) * bt_stride;
  const uint32_t pos = uint32_t(L - 1);
  const float2* cs = rope + size_t(pos) * 64;
  const __nv_bfloat16* row = qkv + size_t(s) * width;
  const uint32_t n_chunks = (uint32_t(L) + kDamChunk - 1) / kDamChunk;
  const uint32_t g = lane >> 2, t4 = lane & 3;
  constexpr uint32_t kChunksPerPage = kPageTokens / kDamChunk;

  auto load_chunk = [&](uint32_t c, uint32_t buf) {
    const int32_t page = bt[c / kChunksPerPage];
    const size_t base = ((size_t(page) * n_kv + kvh) * kPageTokens + (c % kChunksPerPage) * kDamChunk) * kHeadDim;
    const __nv_bfloat16* kg = k_pages + base;
    const __nv_bfloat16* vg = v_pages + base;
    __nv_bfloat16* dk = sk + buf * kDamChunk * kHeadDim;
    __nv_bfloat16* dv = sv + buf * kDamChunk * kHeadDim;
    const uint32_t rows = min(uint32_t(kDamChunk), uint32_t(L) - c * kDamChunk);
#pragma unroll 4
    for (uint32_t i = 0; i < kDamChunk / 2; ++i) {
      const uint32_t x = lane + i * 32;  // 512 16-byte pieces per tile
      const uint32_t r = x >> 4, ch = x & 15;
      const bool valid = r < rows;
      cp_async16(dk + swz(r, ch), kg + r * kHeadDim + ch * 8, valid);
      cp_async16(dv + swz(r, ch), vg + r * kHeadDim + ch * 8, valid);
    }
  };
  load_chunk(0, 0);
  cp_async_commit();
  if (n_chunks > 1) load_chunk(1, 1);
  cp_async_commit();

  // rotate q (4 heads x 64 pairs), rotate + append the new k, append v
  for (uint32_t p = lane; p < kDecHeads * 64; p += 32) {
    const uint32_t h = p / 64, i = p % 64;
    const float2 c = cs[i];
    const __nv_bfloat16* hp = row + size_t(h0 + h) * kHeadDim;
    const float a = __bfloat162float(hp[i]), b = __bfloat162float(hp[i + 64]);
    sq[h * kHeadDim + i] = __float2bfloat16_rn(a * c.x - b * c.y);
    sq[h * kHeadDim + i + 64] = __float2bfloat16_rn(b * c.x + a * c.y);
  }
  {
    const int32_t page = bt[pos / kPageTokens];
    const uint32_t slot = pos % kPageTokens;
    __nv_bfloat16* kd = k_pages + ((size_t(page) * n_kv + kvh) * kPageTokens + slot) * kHeadDim;
    __nv_bfloat16* vd = v_pages + ((size_t(page) * n_kv + kvh) * kPageTokens + slot) * kHeadDim;
    const __nv_bfloat16* kp = row + size_t(n_heads + kvh) * kHeadDim;
    const __nv_bfloat16* vp = row + size_t(n_heads + n_kv + kvh) * kHeadDim;
    for (uint32_t i = lane; i < 64; i += 32) {
      const float2 c = cs[i];
      const float a = __bfloat162float(kp[i]), b = __bfloat162float(kp[i + 64]);
      const __nv_bfloat16 ra = __float2bfloat16_rn(a * c.x - b * c.y), rb = __float2bfloat16_rn(b * c.x + a * c.y);
      kd[i] = ra; kd[i + 64] = rb; s_knew[i] = ra; s_knew[i + 64] = rb;
      const __nv_bfloat16 v0 = vp[i], v1 = vp[i + 64];
      vd[i] = v0; vd[i + 64] = v1; s_vnew[i] = v0; s_vnew[i + 64] = v1;
    }
  }
  __syncwarp();

  // A fragments of Q: rows 0..3 real (lanes with g < 4), rows 8..15 zero
  uint32_t qf[8][4];
#pragma unroll
  for (int ks = 0; ks < 8; ++ks) {
    qf[ks][1] = 0; qf[ks][3] = 0;
    if (g < kDecHeads) {
      qf[ks][0] = *reinterpret_cast<const uint32_t*>(sq + g * kHeadDim + ks * 16 + t4 * 2);
      qf[ks][2] = *reinterpret_cast<const uint32_t*>(sq + g * kHeadDim + ks * 16 + 8 + t4 * 2);
    } else {
      qf[ks][0] = 0; qf[ks][2] = 0;
    }
  }
  float o[16][4];
#pragma unroll
  for (int i = 0; i < 16; ++i) o[i][0] = o[i][1] = o[i][2] = o[i][3] = 0.f;
  float m_run = -INFINITY, l_run = 0.f;   // row g (rows g+8 are padding)
  const float scale = rsqrtf(float(kHeadDim)) * kLog2e;

  for (uint32_t c = 0; c < n_chunks; ++c) {
    const uint32_t buf = c % kDamStages;
    if (c + 2 < n_chunks) load_chunk(c + 2, (c + 2) % kDamStages);   // the buffer chunk c-1 just left
    cp_async_commit();
    cp_async_wait<2>();
    __syncwarp();
    __nv_bfloat16* tk = sk + buf * kDamChunk * kHeadDim;
    __nv_bfloat16* tv = sv + buf * kDamChunk * kHeadDim;
    if (c == pos / kDamChunk) {  // the new token's row was fetched before it was written: patch it
      const uint32_t r = pos % kDamChunk;
      for (uint32_t ch = lane; ch < 16; ch += 32) {
        *reinterpret_cast<uint4*>(tk + swz(r, ch)) = *reinterpret_cast<const uint4*>(s_knew + ch * 8);
        *reinterpret_cast<uint4*>(tv + swz(r, ch)) = *reinterpret_cast<const uint4*>(s_vnew + ch * 8);
      }
      __syncwarp();
    }
    float sc[kDamChunk / 8][4];
#pragma unroll
    for (int nb = 0; nb < kDamChunk / 8; ++nb) {
      sc[nb][0] = sc[nb][1] = sc[nb][2] = sc[nb][3] = 0.f;
#pragma unroll
      for (int kp = 0; kp < 4; ++kp) {
        uint32_t kb[4];
        const uint32_t m = lane >> 3;
        ldmatrix_x4(kb, tk + swz(nb * 8 + (lane & 7), kp * 4 + m));
        mma_bf16_16816(sc[nb], qf[kp * 2], kb[0], kb[1]);
        mma_bf16_16816(sc[nb], qf[kp * 2 + 1], kb[2], kb[3]);
      }
    }
    const uint32_t kv0 = c * kDamChunk;
    float m_new = m_run;
#pragma unroll
    for (int nb = 0; nb < kDamChunk / 8; ++nb)
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        float v = sc[nb][e] * scale;
        if (kv0 + nb * 8 + t4 * 2 + e >= uint32_t(L)) v = -INFINITY;
        sc[nb][e] = v;
        m_new = fmaxf(m_new, v);
      }
    m_new = fmaxf(m_new, __shfl_xor_sync(0xffffffffu, m_new, 1));
    m_new = fmaxf(m_new, __shfl_xor_sync(0xffffffffu, m_new, 2));
    const float corr = exp2f(m_run - m_new);
    m_run = m_new;
    float rsum = 0.f;
#pragma unroll
    for (int nb = 0; nb < kDamChunk / 8; ++nb) {
      const float p0 = exp2f(sc[nb][0] - m_new), p1 = exp2f(sc[nb][1] - m_new);
      sc[nb][0] = p0; sc[nb][1] = p1;
      rsum += p0 + p1;
    }
    l_run = l_run * corr + rsum;
#pragma unroll
    for (int nb = 0; nb < 16; ++nb) { o[nb][0] *= corr; o[nb][1] *= corr; }
#pragma unroll
    for (int ks = 0; ks < kDamChunk / 16; ++ks) {
      uint32_t pa[4];
      pa[0] = pack_bf16(sc[2 * ks][0], sc[2 * ks][1]);
      pa[1] = 0;
      pa[2] = pack_bf16(sc[2 * ks + 1][0], sc[2 * ks + 1][1]);
      pa[3] = 0;
#pragma unroll
      for (int np = 0; np < 8; ++np) {
        uint32_t vb[4];
        const uint32_t m = lane >> 3;
        ldmatrix_x4_trans(vb, tv + swz(ks * 16 + (m & 1) * 8 + (lane & 7), np * 2 + (m >> 1)));
        mma_bf16_16816(o[np * 2], pa, vb[0], vb[1]);
        mma_bf16_16816(o[np * 2 + 1], pa, vb[2], vb[3]);
      }
    }
    __syncwarp();
  }
  cp_async_wait<0>();
  l_run += __shfl_xor_sync(0xffffffffu, l_run, 1);
  l_run += __shfl_xor_sync(0xffffffffu, l_run, 2);
  if (g < kDecHeads) {
    const float inv = 1.f / l_run;
    __nv_bfloat16* dst = out + size_t(s) * n_heads * kHeadDim + size_t(h0 + g) * kHeadDim;
#pragma unroll
    for (int nb = 0; nb < 16; ++nb)
      *reinterpret_cast<uint32_t*>(dst + nb * 8 + t4 * 2) = pack_bf16(o[nb][0] * inv, o[nb][1] * inv);
  }
}

// pdl: launch with programmatic stream serialization (the kernel prefetches its first K/V page
// and then waits on the producer of qkv).  Only safe when everything the prologue reads
// (seq_lens, block tables, old K/V) was written by kernels that are already complete: the engine
// uses it for layers >= 1 of a decode step.
int decode_attention_launch(const void* qkv, void* k_pages, void* v_pages, const int32_t* block_tables,
                            uint32_t bt_stride, const int32_t* bt_rows, const int32_t* seq_lens, uint32_t n_seqs,
                            void* out, uint32_t n_heads, uint32_t n_kv, const float* rope_table, uint32_t n_splits,
                            bool pdl, cudaStream_t st) {
  if (!qkv || !k_pages || !v_pages || !block_tables || !seq_lens || !out || !rope_table ||
      n_kv == 0 || n_heads % n_kv || n_heads % kDecHeads || (n_heads / n_kv) % kDecHeads ||
      n_splits == 0) {
    set_error("llmlb_op_decode_attention: bad argument (GQA group must be a multiple of 4)");
    return LLMLB_E_INVALID_ARG;
  }
  if (n_seqs == 0) return LLMLB_OK;
  static bool configured = false, allow16 = false;
  if (!configured) {
    allow16 = cudaFuncSetAttribute(decode_attention_kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 1) == cudaSuccess;
    cudaGetLastError();
    configured = true;
  }
  // splits form a cluster: round down to a supported cluster size
  uint32_t sp = (n_splits >= 16 && allow16) ? 16 : n_splits >= 8 ? 8 : n_splits >= 4 ? 4 : n_splits >= 2 ? 2 : 1;
  if (sp == 1) {  // wide batch: one warp per (sequence, head group), tensor cores + cp.async ring
    static bool dam_configured = false;
    if (!dam_configured) {
      LLMLB_CUDA_CHECK(cudaFuncSetAttribute(decode_attention_mma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kDamSmem));
      dam_configured = true;
    }
    decode_attention_mma_kernel<<<dim3(n_heads / kDecHeads, n_seqs), kDamThreads, kDamSmem, st>>>(
        (const __nv_bfloat16*)qkv, (__nv_bfloat16*)k_pages, (__nv_bfloat16*)v_pages, block_tables, bt_stride, bt_rows,
        seq_lens, (const float2*)rope_table, (__nv_bfloat16*)out, n_heads, n_kv, 1u);
    LLMLB_LAUNCH_CHECK();
    return LLMLB_OK;
  }
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(sp, n_heads / kDecHeads, n_seqs);
  cfg.blockDim = dim3(kDecThreads);
  cfg.dynamicSmemBytes = 0;
  cfg.stream = st;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = sp;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl ? 2 : 1;
  LLMLB_CUDA_CHECK(cudaLaunchKernelEx(
      &cfg, decode_attention_kernel, (const __nv_bfloat16*)qkv, (__nv_bfloat16*)k_pages,
      (__nv_bfloat16*)v_pages, block_tables, bt_stride, bt_rows, seq_lens,
      (const float2*)rope_table, (__nv_bfloat16*)out, n_heads, n_kv, sp));
  LLMLB_LAUNCH_CHECK();
  return LLMLB_OK;
}
}  // namespace llmlb

extern "C" int llmlb_op_decode_attention(const void* qkv, void* k_pages, void* v_pages,
                                         const int32_t* block_tables, uint32_t bt_stride,
                                         const int32_t* bt_rows, const int32_t* seq_lens,
                                         uint32_t n_seqs, void* out, uint32_t n_heads,
                                         uint32_t n_kv, const float* rope_table,
                                         uint32_t n_splits, uint32_t, void*, void* stream) {
  return decode_attention_launch(qkv, k_pages, v_pages, block_tables, bt_stride, bt_rows, seq_lens, n_seqs, out,
                                 n_heads, n_kv, rope_table, n_splits, false, (cudaStream_t)stream);
}
