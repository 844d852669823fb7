// Shared helpers for the sm_100a kernels of llmlb_b200.
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <atomic>
#include <string>

namespace llmlb {

constexpr int kHeadDim = 128;        // Llama-3 head width (the only one the kernels accept)
constexpr int kPageTokens = 64;      // tokens per KV page
constexpr int kNumSMs = 148;         // B200

// thread-local error text behind llmlb_last_error()
void set_error(const std::string& s);
extern std::atomic<uint64_t> g_kernel_launches;

#define LLMLB_CUDA_CHECK(expr)                                                            \
  do {                                                                                    \
    cudaError_t _e = (expr);                                                              \
    if (_e != cudaSuccess) {                                                              \
      ::llmlb::set_error(std::string(#expr) + ": " + cudaGetErrorString(_e));             \
      return LLMLB_E_DEVICE;                                                              \
    }                                                                                     \
  } while (0)

#define LLMLB_LAUNCH_CHECK()                                                              \
  do {                                                                                    \
    ::llmlb::g_kernel_launches.fetch_add(1, std::memory_order_relaxed);                   \
    cudaError_t _e = cudaGetLastError();                                                  \
    if (_e != cudaSuccess) {                                                              \
      ::llmlb::set_error(std::string("kernel launch: ") + cudaGetErrorString(_e));        \
      return LLMLB_E_DEVICE;                                                              \
    }                                                                                     \
  } while (0)

// ---- synthetic weights: integer hash -> Irwin-Hall(4) -> bf16, bit-reproducible on CPU ----
__host__ __device__ __forceinline__ uint64_t mix64(uint64_t z) {
  z += 0x9E3779B97F4A7C15ull;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}
// sum of four 16-bit lanes, centred; std of the sum is 2*65536/sqrt(12)*sqrt(1-2^-32) ~ 37837.2
constexpr float kSynthSumStd = 37837.22f;
__host__ __device__ __forceinline__ float synth_value(uint64_t seed, uint32_t tensor_id,
                                                      uint64_t idx, float scale) {
  uint64_t h = mix64(mix64(seed * 0xD1342543DE82EF95ull + tensor_id) + idx);
  int s = int(h & 0xFFFF) + int((h >> 16) & 0xFFFF) + int((h >> 32) & 0xFFFF) +
          int((h >> 48) & 0xFFFF) - 131070;
  return float(s) * scale;
}

// ---- optional in-kernel timeline (debug): thread 0 of a CTA appends one record ----
struct TraceBuf {
  unsigned long long* data;  // records of 6 u64: tag, blockIdx|smid<<32, t0..t3 (globaltimer ns)
  unsigned int* count;
  unsigned int cap;
};

#ifdef __CUDACC__
__device__ __forceinline__ unsigned int ld_acquire_gpu_u32(const unsigned int* p) {
  unsigned int v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ unsigned long long gtime_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
__device__ __forceinline__ void trace_emit(const TraceBuf& tb, unsigned long long tag, unsigned long long t0,
                                           unsigned long long t1, unsigned long long t2, unsigned long long t3) {
  if (!tb.data) return;
  unsigned int smid;
  asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
  unsigned int i = atomicAdd(tb.count, 1u);
  if (i < tb.cap) {
    unsigned long long* r = tb.data + size_t(i) * 6;
    r[0] = tag; r[1] = (unsigned long long)blockIdx.x | ((unsigned long long)smid << 32) | ((unsigned long long)blockIdx.y << 16);
    r[2] = t0; r[3] = t1; r[4] = t2; r[5] = t3;
  }
}
__device__ __forceinline__ float bf16_lo(uint32_t v) { return __uint_as_float(v << 16); }
__device__ __forceinline__ float bf16_hi(uint32_t v) { return __uint_as_float(v & 0xFFFF0000u); }
__device__ __forceinline__ uint32_t pack_bf16(float a, float b) {
  __nv_bfloat162 p = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&p);
}
__device__ __forceinline__ uint4 ldg_stream(const void* p) {  // streamed-once weights
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.L2::256B.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
               : "l"(p));
  return r;
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
#endif

}  // namespace llmlb
