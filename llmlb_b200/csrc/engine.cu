// llmlb_engine: the in-process replacement for the gateway's HTTP hop to an inference endpoint
// (reference boundary: llmlb/src/api/openai.rs:995-1005, llmlb/src/api/proxy.rs:372-401).
//
// One engine per GPU rank.  Host side (this file): weights + paged-KV pool + sequence slots, an
// iteration-level continuous-batching scheduler on its own thread (SURVEY §8 a2.14), per-request
// token-event queues for non-blocking submit/poll/cancel.  Device side: the kernels in the
// sibling .cu files, chained on one stream; decode steps are captured into CUDA graphs per batch
// width and all per-sequence decode state (length, last token, sampler counters) lives in HBM so
// the GPU never waits for the host between tokens — the host reads tokens `lookahead` steps late.
#include <cuda.h>

#include <algorithm>
#include <chrono>
#include <condition_variable>
#include <cstdlib>
#include <cstring>
#include <deque>
#include <map>
#include <memory>
#include <mutex>
#include <thread>
#include <unordered_map>
#include <vector>

#include <fcntl.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>

#include "../../include/llmlb_b200.h"
#include "common.cuh"
#include "tc_common.cuh"
#include "tp_common.cuh"

namespace llmlb {

// ---- pieces defined in the other translation units ----
int make_tmap_bf16(CUtensorMap* m, const void* base, uint64_t rows, uint64_t cols,
                   uint32_t box_rows);
uint32_t tc_pick_bn(uint32_t n_tokens);
int gemm_tc_launch(const CUtensorMap& tw, const CUtensorMap& tx, void* out, uint32_t n_tokens,
                   uint32_t n_out, uint32_t k, uint32_t epi, uint32_t out_stride, cudaStream_t st,
                   const CUtensorMap* tx_half = nullptr, uint32_t* n_parts = nullptr,
                   const TpPushRS* tpp = nullptr, uint32_t max_split = 8);

int rmsnorm_parts_launch(float* x, const float* parts, uint32_t n_parts, size_t part_stride, const void* gain,
                         void* y, uint32_t n_tokens, uint32_t hidden, float eps, cudaStream_t st);
int gemv_decode(const void* w, const void* x, const void* gain, float eps, void* out, uint32_t n_tokens,
                uint32_t n_out, uint32_t k, uint32_t epi, uint32_t out_stride, cudaStream_t st);
int decode_attention_launch(const void* qkv, void* k_pages, void* v_pages, const int32_t* block_tables,
                            uint32_t bt_stride, const int32_t* bt_rows, const int32_t* seq_lens, uint32_t n_seqs,
                            void* out, uint32_t n_heads, uint32_t n_kv, const float* rope_table, uint32_t n_splits,
                            bool pdl, cudaStream_t st);
void ks_set_trace(const TraceBuf& tb);
void tc_set_trace(const TraceBuf& tb);
void attn_set_trace(const TraceBuf& tb);
void tp_set_trace(const TraceBuf& tb);
void tc2_set_trace(const TraceBuf& tb);

// tensor parallel (tp_common.cuh): fused GEMV consumer / producer of protocol A, pull kernels
int gemv_tp_consume(const TpCtx& ctx, uint32_t coll_in, const void* w, const float* x_in, float* x_out,
                    const void* gain, float eps, void* out, uint32_t n_tokens, uint32_t n_out, uint32_t k,
                    uint32_t epi, uint32_t out_stride, cudaStream_t st);
int gemv_tp_push(const TpCtx& ctx, uint32_t coll_out, const void* w, const void* x_bf16, uint32_t n_tokens,
                 uint32_t n_out, uint32_t k, cudaStream_t st);
int ar_allreduce_add(const TpCtx& P, uint64_t off, float* x, uint64_t n, cudaStream_t st);
int ar_allgather_cols(const TpCtx& P, uint64_t off, float* out, uint32_t rows, uint32_t cols_local, cudaStream_t st);
constexpr uint32_t kTpMaxSplit = 4;   // K-split parts a push-RS GEMM may use (slot capacity)
// prefill attention on tcgen05 (attention_tc.cu)
int make_tmap_attn_q(CUtensorMap* m, const void* qkv, uint64_t n_tokens, uint64_t width);
int make_tmap_attn_kv(CUtensorMap* m, const void* pool, uint64_t n_layers, uint64_t n_pages, uint64_t n_kv);
int prefill_attention_tc_launch(const CUtensorMap& mq, const CUtensorMap& mk, const CUtensorMap& mv, uint32_t layer,
                                const int32_t* block_tables, uint32_t bt_stride, const int32_t* tiles, uint32_t n_tiles,
                                void* out, uint32_t n_heads, uint32_t n_kv, bool pdl, cudaStream_t st);
int rope_append_launch(void* qkv, const int32_t* positions, const int32_t* page_of_token, const float* rope_table,
                       void* k_pages, void* v_pages, uint32_t n_tokens, uint32_t n_heads, uint32_t n_kv, bool pdl,
                       cudaStream_t st);

static thread_local std::string g_err;
void set_error(const std::string& s) { g_err = s; }
std::atomic<uint64_t> g_kernel_launches{0};

#define RC(expr)                 \
  do {                           \
    int _rc = (expr);            \
    if (_rc != LLMLB_OK) return _rc; \
  } while (0)

// ------------------------------------------------------------------ small device kernels ----
__global__ void fill_bf16_kernel(__nv_bfloat16* p, uint64_t n, float v) {
  for (uint64_t i = uint64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n;
       i += uint64_t(gridDim.x) * blockDim.x)
    p[i] = __float2bfloat16_rn(v);
}
__global__ void synth_strided_kernel(__nv_bfloat16* __restrict__ out, uint64_t rows, uint64_t cols,
                                     uint64_t out_ld, uint64_t row0, uint64_t col0, uint64_t ld,
                                     uint64_t seed, uint32_t tensor_id, float scale) {
  const uint64_t n = rows * cols;
  for (uint64_t i = uint64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n;
       i += uint64_t(gridDim.x) * blockDim.x) {
    uint64_t r = i / cols, c = i - r * cols;
    out[r * out_ld + c] =
        __float2bfloat16_rn(synth_value(seed, tensor_id, (row0 + r) * ld + (col0 + c), scale));
  }
}

struct SlotState {  // per-sequence decode state, device resident
  int32_t* seq_len;     // tokens whose K/V are in the cache
  int32_t* last_token;  // next input token
  float* temperature;
  float* top_p;
  int32_t* top_k;
  uint64_t* seed;
  uint64_t* step;
};
struct BatchView {  // compact per-step arrays
  int32_t* slots;     // batch position -> slot
  int32_t* ids;
  int32_t* seq_lens;  // including the new token
  float* temperature;
  float* top_p;
  int32_t* top_k;
  uint64_t* seed;
  uint64_t* step;
  int32_t* out_ids;
};

// decode: pull the per-slot state into the compact batch arrays and advance the lengths
__global__ void decode_prepare_kernel(SlotState S, BatchView B, uint32_t n) {
  uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= n) return;
  int32_t slot = B.slots[b];
  B.ids[b] = S.last_token[slot];
  int32_t L = S.seq_len[slot] + 1;
  S.seq_len[slot] = L;
  B.seq_lens[b] = L;
  B.temperature[b] = S.temperature[slot];
  B.top_p[b] = S.top_p[slot];
  B.top_k[b] = S.top_k[slot];
  B.seed[b] = S.seed[slot];
  B.step[b] = S.step[slot];
}
// first token after prefill: only the sampler state is gathered
__global__ void sample_prepare_kernel(SlotState S, BatchView B, uint32_t n) {
  uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= n) return;
  int32_t slot = B.slots[b];
  B.temperature[b] = S.temperature[slot];
  B.top_p[b] = S.top_p[slot];
  B.top_k[b] = S.top_k[slot];
  B.seed[b] = S.seed[slot];
  B.step[b] = S.step[slot];
}
__global__ void step_finish_kernel(SlotState S, BatchView B, uint32_t n) {
  uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= n) return;
  int32_t slot = B.slots[b];
  S.last_token[slot] = B.out_ids[b];
  S.step[slot] += 1;
}
// y_last[r, :] = x[rows[r], :]  (fp32 -> fp32 gather of the rows that need logits)
__global__ void gather_rows_kernel(const float* __restrict__ x, const int32_t* __restrict__ rows,
                                   float* __restrict__ out, uint32_t hidden) {
  const float4* src = reinterpret_cast<const float4*>(x + size_t(rows[blockIdx.x]) * hidden);
  float4* dst = reinterpret_cast<float4*>(out + size_t(blockIdx.x) * hidden);
  for (uint32_t i = threadIdx.x; i < hidden / 4; i += blockDim.x) dst[i] = src[i];
}

// ------------------------------------------------------------------ host structures ---------
struct Request {
  uint64_t id = 0;
  std::vector<int32_t> prompt;
  llmlb_sampling s{};
  std::vector<int32_t> stop_ids;
  int slot = -1;
  std::vector<int32_t> pages;
  uint32_t prefilled = 0;   // context tokens whose KV is (being) written
  uint32_t launched = 0;    // generated tokens whose computation has been launched
  uint32_t harvested = 0;   // generated tokens seen by the host
  // `prompt` is the context to prefill: the client's prompt, plus — after a preemption — the tokens
  // generated so far (recompute instead of swapping KV out)
  uint32_t n_prompt0 = 0;   // the client's prompt length (usage accounting, context arithmetic)
  std::vector<int32_t> gen; // harvested generated tokens
  uint32_t gen_in_prompt = 0;
  uint32_t pages_published = 0;   // entries of `pages` already in the device block table
  uint32_t preempted = 0;
  bool admitted_once = false;
  bool finished = false;
  bool cancel = false;
  uint32_t cancel_reason = LLMLB_FINISH_CANCELLED;
  bool client_released = false;
  uint32_t finish_reason = LLMLB_FINISH_NONE;
  std::deque<llmlb_token_event> events;
  std::chrono::steady_clock::time_point t_submit;
};
using ReqPtr = std::shared_ptr<Request>;

struct InflightStep {
  cudaEvent_t ev_start = nullptr, ev_end = nullptr;
  int32_t* host_ids = nullptr;        // pinned
  std::vector<ReqPtr> reqs;           // batch position -> request
  bool is_prefill = false;
  uint32_t n_tokens = 0;
};

// ---- tensor-parallel plan channel ------------------------------------------------------------
// Rank 0 owns the request queue and the scheduler.  Everything that changes scheduler state —
// submit, cancel/release, pause, one scheduling iteration, one harvest — is appended, in the order
// rank 0 applied it, to a byte ring in POSIX shared memory; the follower ranks replay the same
// calls in the same order, so every rank holds the same slots, pages and batches and launches the
// same steps (the collectives inside a step need exactly that).  Sampling is identical on every
// rank (all-gathered logits, per-request seeds), so finishes are reproduced, not transmitted.
struct PlanHeader {
  std::atomic<uint64_t> head;        // bytes ever written
  std::atomic<uint64_t> tail[8];     // bytes consumed per rank (rank 0 unused)
  std::atomic<uint32_t> magic;       // set last by the leader
  uint32_t n_ranks;
  uint64_t ring_bytes;
};
enum PlanEvent : uint32_t { kPlanSubmit = 1, kPlanCancel = 2, kPlanRelease = 3, kPlanPause = 4, kPlanSched = 5, kPlanHarvest = 6, kPlanStop = 7,
                            kPlanExpire = 8 /* id + finish reason: a time-based decision of rank 0's clock */ };
constexpr uint32_t kPlanMagic = 0x4C4C5031u;   // "LLP1"
constexpr size_t kPlanHeaderBytes = 4096, kPlanRingBytes = size_t(8) << 20;
constexpr long long kPlanStallMs = 30000;   // a follower that has not drained an 8 MiB ring for this long is gone

struct PlanChannel {
  PlanHeader* h = nullptr;
  uint8_t* ring = nullptr;
  uint32_t rank = 0;
  std::string name;
  bool leader = false;

  int open(const std::string& shm_name, uint32_t my_rank, uint32_t n_ranks) {
    name = shm_name[0] == '/' ? shm_name : "/" + shm_name;
    rank = my_rank;
    leader = my_rank == 0;
    const size_t total = kPlanHeaderBytes + kPlanRingBytes;
    int fd = -1;
    if (leader) {
      shm_unlink(name.c_str());
      fd = shm_open(name.c_str(), O_CREAT | O_EXCL | O_RDWR, 0600);
      if (fd < 0 || ftruncate(fd, off_t(total)) != 0) { if (fd >= 0) close(fd); set_error("plan channel: cannot create " + name); return LLMLB_E_INTERNAL; }
    } else {
      for (int tries = 0; tries < 3000 && fd < 0; ++tries) {   // the leader may still be creating it
        fd = shm_open(name.c_str(), O_RDWR, 0600);
        struct stat sb;
        if (fd >= 0 && (fstat(fd, &sb) != 0 || size_t(sb.st_size) < total)) { close(fd); fd = -1; }
        if (fd < 0) usleep(10000);
      }
      if (fd < 0) { set_error("plan channel: " + name + " did not appear (rank 0 calls llmlb_engine_tp_plan_channel first)"); return LLMLB_E_TIMEOUT; }
    }
    void* p = mmap(nullptr, total, PROT_READ | PROT_WRITE, MAP_SHARED, fd, 0);
    close(fd);
    if (p == MAP_FAILED) { set_error("plan channel: mmap failed"); return LLMLB_E_INTERNAL; }
    h = static_cast<PlanHeader*>(p);
    ring = static_cast<uint8_t*>(p) + kPlanHeaderBytes;
    if (leader) {
      h->head.store(0);
      for (auto& t : h->tail) t.store(0);
      h->n_ranks = n_ranks;
      h->ring_bytes = kPlanRingBytes;
      h->magic.store(kPlanMagic, std::memory_order_release);
    } else {
      for (int tries = 0; tries < 3000 && h->magic.load(std::memory_order_acquire) != kPlanMagic; ++tries) usleep(10000);
      if (h->magic.load(std::memory_order_acquire) != kPlanMagic) { set_error("plan channel: header never initialised"); return LLMLB_E_TIMEOUT; }
    }
    return LLMLB_OK;
  }
  void close_channel() {
    if (h) munmap(h, kPlanHeaderBytes + kPlanRingBytes);
    if (leader && !name.empty()) shm_unlink(name.c_str());
    h = nullptr;
  }
  void copy_in(uint64_t pos, const void* src, size_t n) {
    const size_t off = size_t(pos % kPlanRingBytes), first = std::min(n, kPlanRingBytes - off);
    memcpy(ring + off, src, first);
    if (n > first) memcpy(ring, static_cast<const uint8_t*>(src) + first, n - first);
  }
  void copy_out(uint64_t pos, void* dst, size_t n) const {
    const size_t off = size_t(pos % kPlanRingBytes), first = std::min(n, kPlanRingBytes - off);
    memcpy(dst, ring + off, first);
    if (n > first) memcpy(static_cast<uint8_t*>(dst) + first, ring, n - first);
  }
  // leader: record = [u32 payload bytes][u32 type][payload, padded to 8]
  // false: a follower stopped reading (ring full for kPlanStallMs) — the caller holds the scheduler mutex, so the wait is
  // bounded and the engine is failed instead of wedging submit / poll / health behind a dead rank
  bool write(uint32_t type, const void* payload, uint32_t len) {
    const uint32_t padded = (len + 7u) & ~7u;
    const uint64_t need = 8 + padded;
    uint64_t head = h->head.load(std::memory_order_relaxed);
    const auto t0 = std::chrono::steady_clock::now();
    for (uint32_t spins = 0;; ++spins) {   // back-pressure: never overwrite what the slowest follower has not read
      uint64_t lo = head;
      for (uint32_t r = 1; r < h->n_ranks; ++r) lo = std::min(lo, h->tail[r].load(std::memory_order_acquire));
      if (head + need - lo <= kPlanRingBytes) break;
      if ((spins & 0x3FFu) == 0x3FFu &&
          std::chrono::duration_cast<std::chrono::milliseconds>(std::chrono::steady_clock::now() - t0).count() > kPlanStallMs) return false;
      usleep(50);
    }
    const uint32_t hdr[2] = {len, type};
    copy_in(head, hdr, 8);
    if (len) copy_in(head + 8, payload, len);
    h->head.store(head + need, std::memory_order_release);
    return true;
  }
  // follower: blocks until the next record is there (0 = aborted by engine destroy)
  uint32_t read(std::vector<uint8_t>* payload, const std::atomic<bool>& abort) {
    const uint64_t tail = h->tail[rank].load(std::memory_order_relaxed);
    for (uint32_t spins = 0; h->head.load(std::memory_order_acquire) == tail; ++spins) {
      if (abort.load(std::memory_order_relaxed)) return 0;
      if (spins > 2000) usleep(20); else std::this_thread::yield();
    }
    uint32_t hdr[2];
    copy_out(tail, hdr, 8);
    payload->resize(hdr[0]);
    if (hdr[0]) copy_out(tail + 8, payload->data(), hdr[0]);
    h->tail[rank].store(tail + 8 + ((hdr[0] + 7u) & ~7u), std::memory_order_release);
    return hdr[1];
  }
};

struct LayerW {
  __nv_bfloat16 *wqkv, *wo, *wgu, *wdown, *attn_norm, *ffn_norm;
  CUtensorMap m_wqkv, m_wo, m_wgu, m_wdown;
};

}  // namespace llmlb

using namespace llmlb;

struct llmlb_engine {
  llmlb_engine_config cfg{};
  llmlb_model_config M{};
  // derived geometry (per rank)
  uint32_t tp = 1, rank = 0;
  uint32_t nq_l = 0, nkv_l = 0, ffn_l = 0, vocab_l = 0, qkv_w = 0;
  uint32_t t_cap = 0;             // activation rows
  uint32_t pages_per_seq = 0, n_pages = 0;
  uint32_t lookahead = 2;
  cudaStream_t st = nullptr;

  // weights
  __nv_bfloat16* embed = nullptr;
  __nv_bfloat16* final_norm = nullptr;
  __nv_bfloat16* lm_head = nullptr;
  CUtensorMap m_lm_head{};
  std::vector<LayerW> layers;
  uint64_t param_bytes = 0;

  // KV pool [layer][page][kv_head][64][128]
  __nv_bfloat16 *k_pool = nullptr, *v_pool = nullptr;
  size_t layer_pool_elems = 0;
  float* rope = nullptr;
  int32_t* d_block_tables = nullptr;  // [max_seqs][pages_per_seq]
  std::vector<int32_t> free_pages;
  std::vector<int32_t> free_slots;

  // activations
  float* x = nullptr;
  __nv_bfloat16 *y = nullptr, *qkv = nullptr, *attn = nullptr, *h = nullptr;
  float* logits = nullptr;       // [max_seqs][vocab]
  float* logits_l = nullptr;     // [max_seqs][vocab_l] local slice when tp > 1
  float* x_last = nullptr;       // [max_seqs][hidden]
  void* attn_ws = nullptr;
  CUtensorMap m_y[5]{}, m_attn[5]{}, m_h[5]{};  // box rows 16,32,64,128,256
  CUtensorMap m_attn_q{}, m_kpool{}, m_vpool{};  // tcgen05 prefill attention: q rows of qkv, the K / V pools (5-D)
  static constexpr uint32_t kPfTile = 128;        // q rows per prefill-attention tile (UMMA M of attention_tc.cu)

  // per-step metadata (device) + pinned staging ring
  int32_t *d_ids = nullptr, *d_pos = nullptr, *d_page_of_tok = nullptr, *d_tiles = nullptr,
          *d_last_rows = nullptr;
  SlotState S{};
  BatchView B{};
  static constexpr int kRing = 8;
  uint8_t* h_stage[kRing] = {};
  size_t stage_bytes = 0;
  uint64_t stage_seq = 0;
  int32_t* h_out[kRing] = {};
  uint64_t out_seq = 0;
  std::vector<cudaEvent_t> ev_pool;

  // TP exchange (tp_common.cuh): one IPC-shared region per rank
  uint8_t* xchg = nullptr;
  size_t xchg_bytes = 0;
  TpCtx tpc{};
  uint64_t logits_slot_off = 0, pull_slot_off = 0, pull_slot_bytes = 0;
  bool tp_ready = false;
  uint32_t tp_coll = 0;              // collectives issued so far in the current forward pass
  float* xb = nullptr;               // second residual buffer (protocol A ping-pong)
  float* tp_stage = nullptr;         // [4][hidden] fp32: partial rows of projections the fused GEMV does not take
  __nv_bfloat16* ylast = nullptr;    // [max_seqs][hidden] normalised rows that need logits (protocol B)
  CUtensorMap m_ylast[5]{};

  // decode graphs by batch width
  std::unordered_map<uint32_t, cudaGraphExec_t> graphs;
  std::unordered_map<uint32_t, uint64_t> graph_nodes;  // kernels per captured step
  bool paused = false;
  std::string fatal_error;
  float* part_ws = nullptr;         // [8 splits][t_cap][hidden] fp32: K-split partials of O / down (tp == 1)
  float* sk_ws = nullptr;           // in-kernel K-split of the store-epilogue GEMMs: parked fp32 tiles (tc_common.cuh)
  unsigned int* sk_cnt = nullptr;   //   and one arrival counter per output tile
  int warmup();
  std::vector<int32_t> cur_batch_slots;  // what d B.slots currently holds

  // scheduler
  std::mutex mu;               // requests / queues / events
  std::condition_variable cv_sched, cv_events;
  std::mutex step_mu;          // held while a step (or a debug call) uses the GPU state
  std::thread worker;
  bool stop = false;
  PlanChannel plan;               // attached by llmlb_engine_tp_plan_channel (tp > 1)
  bool plan_on = false;           // mu: leader logs / follower replays
  std::atomic<bool> plan_abort{false};   // engine destroy: wakes a follower blocked on the log
  uint64_t next_id = 1;
  std::map<uint64_t, ReqPtr> requests;
  std::deque<ReqPtr> waiting;
  std::vector<ReqPtr> running;   // have a slot; prefilling or decoding
  std::deque<InflightStep> inflight;
  // stats
  std::atomic<uint64_t> steps_prefill{0}, steps_decode{0}, tokens_prefill{0}, tokens_decode{0};
  double gpu_ms_prefill = 0, gpu_ms_decode = 0;  // under mu
  int debug_slot = -1;
  std::vector<int32_t> debug_pages;
  uint32_t debug_len = 0;

  // ---- helpers ----
  __nv_bfloat16* kpool(uint32_t l) { return k_pool + size_t(l) * layer_pool_elems; }
  __nv_bfloat16* vpool(uint32_t l) { return v_pool + size_t(l) * layer_pool_elems; }
  static int bn_index(uint32_t bn) { return bn == 16 ? 0 : bn == 32 ? 1 : bn == 64 ? 2 : bn == 128 ? 3 : 4; }

  int init();
  int alloc_all();
  int gen_weights();
  // where a forward pass left the final hidden state
  struct FwdState {
    float* xres = nullptr;     // fp32 residual rows (complete unless `pending`)
    float* xother = nullptr;   // tp, protocol A: the other residual buffer
    bool pending = false;      // tp, protocol A: collective `pending_coll` is pushed but not folded into xres
    uint32_t pending_coll = 0;
    bool y_final = false;      // tp, protocol B: y holds RMSNorm(x) * final_norm for all rows (bf16)
  };
  int proj(const CUtensorMap& mw, const void* w, const void* xin, const CUtensorMap* mx, void* out, uint32_t T,
           uint32_t n_out, uint32_t k, uint32_t epi, uint32_t out_stride, int wait_coll = -1);
  int layer_stack_decode(uint32_t nb);
  int launch_decode_step(uint32_t nb);
  int forward_tokens(uint32_t T, bool decode, uint32_t nb, uint32_t n_tiles, FwdState* fs);
  int forward_small_tp(uint32_t T, bool decode, uint32_t nb, uint32_t n_tiles, FwdState* fs);
  int forward_big_tp(uint32_t T, bool decode, uint32_t nb, uint32_t n_tiles, FwdState* fs);
  int attention_block(uint32_t l, uint32_t T, bool decode, uint32_t nb, uint32_t n_tiles, bool pdl);
  int finish_small_tp(FwdState* fs, uint32_t T);                     // fold a pending collective: xres complete
  int logits_from_x(const float* src, uint32_t R);                   // fp32 rows, final norm applied here
  int logits_from_y(const __nv_bfloat16* src, const CUtensorMap* maps, uint32_t R);   // rows already normalised
  int logits_tp_consume(FwdState* fs, uint32_t R);                   // protocol A: lm_head consumes the pending collective
  int logits_gather(uint32_t R);                                     // tp > 1: vocab slices -> full rows
  int logits_after_forward(FwdState* fs, uint32_t R, bool decode);   // rows = x[0..R) (decode) or gathered last rows
  float* logits_dst() { return tp == 1 ? logits : reinterpret_cast<float*>(xchg + logits_slot_off); }
  int run_prefill(const std::vector<ReqPtr>& reqs, const std::vector<uint32_t>& take);
  int run_decode(const std::vector<ReqPtr>& batch);
  void harvest_one();
  void loop();
  void loop_follower();
  bool sched_iteration(std::unique_lock<std::mutex>& lk);   // one scheduling decision + launch; lk held on entry, released inside
  // the log has ONE writer at a time: every append happens with mu held
  void plan_log(uint32_t type, const void* payload = nullptr, uint32_t len = 0) {
    if (plan_on && plan.leader && !plan.write(type, payload, len)) {
      plan_on = false;   // no further appends; submits are refused from here on (fatal_error), running requests end with an error
      if (fatal_error.empty()) fatal_error = "tensor-parallel follower stopped reading the plan channel";
    }
  }
  void plan_log_locked(uint32_t type) { if (plan_on && plan.leader) { std::lock_guard<std::mutex> lk(mu); plan_log(type); } }
  // by value: callers pass elements of `running` / `waiting`, and these functions erase from those containers — a reference
  // would dangle, and for a request the client already released the container holds the LAST owner (found by ASan over the
  // fake CUDA runtime: heap-use-after-free in finish_request on cancel of a released, running request)
  void finish_request(ReqPtr r, uint32_t reason);
  void release_resources(ReqPtr r);
  void preempt(ReqPtr r);
  void expire_requests();     // leader / single rank: queue timeouts and request deadlines (time-based)
  std::atomic<uint64_t> preemptions{0};
  cudaEvent_t get_event();
  uint8_t* next_stage() { return h_stage[(stage_seq++) % kRing]; }
  uint32_t decode_splits(uint32_t nb) const {
    uint32_t ctas = nb * (nq_l / 4);
    // batched steps with enough (sequence, head group) pairs: the tensor-core kernel, one warp per pair, no KV split
    // (tp = 2, 64 streams: the 2-way split SIMT kernel took 45 us per layer for 75 MB of K/V)
    if (nb > 4 && ctas >= 96) return 1;
    uint32_t sp = (2 * kNumSMs + ctas - 1) / ctas;
    if (sp > 16) sp = 16;
    if (sp < 1) sp = 1;
    return sp;
  }
  int resolve_tensor(const std::string& name, __nv_bfloat16** base, uint64_t* rows, uint64_t* cols,
                     uint64_t* ld, uint64_t* full_rows, uint64_t* full_cols, uint64_t* row0,
                     uint64_t* col0);
};

extern "C" int llmlb_op_rope_table(float* table, uint32_t max_pos, float theta, void* stream);
extern "C" int llmlb_op_rope_append(void* qkv, const int32_t* positions,
                                    const int32_t* page_of_token, const float* rope_table,
                                    void* k_pages, void* v_pages, uint32_t n_tokens,
                                    uint32_t n_heads, uint32_t n_kv, void* stream);
extern "C" int llmlb_op_decode_attention(const void* qkv, void* k_pages, void* v_pages,
                                         const int32_t* block_tables, uint32_t bt_stride,
                                         const int32_t* bt_rows, const int32_t* seq_lens,
                                         uint32_t n_seqs, void* out, uint32_t n_heads,
                                         uint32_t n_kv, const float* rope_table, uint32_t n_splits,
                                         uint32_t ws_seqs, void* workspace, void* stream);

static inline uint32_t ceil_div(uint32_t a, uint32_t b) { return (a + b - 1) / b; }

// ------------------------------------------------------------------ creation ----------------
int llmlb_engine::init() {
  M = cfg.model;
  tp = cfg.tp_size ? cfg.tp_size : 1;
  rank = cfg.tp_rank;
  if (cfg.abi_version != LLMLB_ABI_VERSION) { set_error("abi_version mismatch"); return LLMLB_E_INVALID_ARG; }
  if (M.head_dim != (uint32_t)kHeadDim) { set_error("head_dim must be 128"); return LLMLB_E_INVALID_ARG; }
  if (cfg.kv_block_tokens != 0 && cfg.kv_block_tokens != (uint32_t)kPageTokens) {
    set_error("kv_block_tokens must be 64"); return LLMLB_E_INVALID_ARG;
  }
  if (!(tp == 1 || tp == 2 || tp == 4 || tp == 8) || rank >= tp) { set_error("bad tp_size/tp_rank"); return LLMLB_E_INVALID_ARG; }
  if (cfg.gemm_impl != 0) { set_error("gemm_impl: only 0 (tcgen05 tiles) is built into the library"); return LLMLB_E_INVALID_ARG; }
  if (cfg.attn_impl != 0) { set_error("attn_impl: only 0 (tcgen05 prefill attention) is built into the library"); return LLMLB_E_INVALID_ARG; }
  if (cfg.tp_proto != 0) { set_error("tp_proto: only 0 ({value, epoch} pairs, every CTA folds) is built into the library"); return LLMLB_E_INVALID_ARG; }
  if (M.n_kv_heads == 0 || M.n_heads % M.n_kv_heads || M.n_kv_heads % tp || M.ffn % tp || M.vocab % tp ||
      ((M.n_heads / M.n_kv_heads) % 4) || M.hidden % 8 || (M.ffn / tp) % 8 || (M.vocab / tp) % 4 ||
      M.n_layers == 0 || M.vocab == 0) {
    set_error("unsupported model geometry (GQA group must be a multiple of 4; dims divisible by tp)");
    return LLMLB_E_INVALID_ARG;
  }
  // the 32-bit exchange epoch keeps the collective's index (+1) in its low 8 bits (tp_common.cuh tp_epoch32): two collectives
  // per layer, so a deeper stack would carry into the step bits and a stale word of the NEXT step could pass for a fresh one
  if (tp > 1 && 2ull * M.n_layers + 1 > 255) {
    set_error("tensor parallel: at most 127 layers (two exchange collectives per layer are numbered in 8 bits)");
    return LLMLB_E_INVALID_ARG;
  }
  if (cfg.max_seqs == 0 || cfg.max_ctx == 0) { set_error("max_seqs/max_ctx must be > 0"); return LLMLB_E_INVALID_ARG; }
  nq_l = M.n_heads / tp; nkv_l = M.n_kv_heads / tp; ffn_l = M.ffn / tp; vocab_l = M.vocab / tp;
  qkv_w = (nq_l + 2 * nkv_l) * kHeadDim;
  uint32_t mst = cfg.max_step_tokens ? cfg.max_step_tokens : 2048;
  t_cap = std::max(mst, cfg.max_seqs);
  t_cap = ceil_div(t_cap, 64) * 64;
  cfg.max_step_tokens = mst;
  pages_per_seq = ceil_div(cfg.max_ctx, kPageTokens);
  n_pages = cfg.kv_pages ? cfg.kv_pages : cfg.max_seqs * pages_per_seq;
  lookahead = cfg.lookahead ? cfg.lookahead : 2;
  if (lookahead > 4) lookahead = 4;
  LLMLB_CUDA_CHECK(cudaSetDevice(cfg.device));
  LLMLB_CUDA_CHECK(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
  RC(alloc_all());
  RC(gen_weights());
  LLMLB_CUDA_CHECK(cudaStreamSynchronize(st));
  if (tp == 1) RC(warmup());
  for (int32_t p = int32_t(n_pages) - 1; p >= 0; --p) free_pages.push_back(p);
  for (int32_t s = int32_t(cfg.max_seqs) - 1; s >= 0; --s) free_slots.push_back(s);
  worker = std::thread([this] { this->loop(); });
  return LLMLB_OK;
}

// NOTE: zero-fill must be ordered with the engine's (non-blocking) stream: a cudaMemset on the
// legacy default stream is NOT ordered with it and raced with the first kernels (rope table).
static thread_local cudaStream_t g_alloc_stream = nullptr;
template <class T>
static int dmalloc(T** p, size_t n_elems, bool zero = true) {
  size_t bytes = n_elems * sizeof(T);
  if (bytes == 0) bytes = sizeof(T);
  cudaError_t e = cudaMalloc((void**)p, bytes);
  if (e != cudaSuccess) {
    set_error(std::string("cudaMalloc(") + std::to_string(bytes) + "): " + cudaGetErrorString(e));
    return LLMLB_E_DEVICE;
  }
  if (zero) cudaMemsetAsync(*p, 0, bytes, g_alloc_stream);
  return LLMLB_OK;
}

int llmlb_engine::alloc_all() {
  const size_t H = M.hidden;
  g_alloc_stream = st;
  RC(dmalloc(&embed, size_t(M.vocab) * H, false));
  RC(dmalloc(&final_norm, H, false));
  RC(dmalloc(&lm_head, size_t(vocab_l) * H, false));
  param_bytes = size_t(vocab_l) * H * 2;
  layers.resize(M.n_layers);
  for (auto& L : layers) {
    RC(dmalloc(&L.wqkv, size_t(qkv_w) * H, false));
    RC(dmalloc(&L.wo, H * size_t(nq_l) * kHeadDim, false));
    RC(dmalloc(&L.wgu, size_t(2) * ffn_l * H, false));
    RC(dmalloc(&L.wdown, H * size_t(ffn_l), false));
    RC(dmalloc(&L.attn_norm, H, false));
    RC(dmalloc(&L.ffn_norm, H, false));
    param_bytes += (size_t(qkv_w) * H + H * size_t(nq_l) * kHeadDim + size_t(2) * ffn_l * H + H * size_t(ffn_l)) * 2;
    RC(make_tmap_bf16(&L.m_wqkv, L.wqkv, qkv_w, H, 128));
    RC(make_tmap_bf16(&L.m_wo, L.wo, H, size_t(nq_l) * kHeadDim, 128));
    RC(make_tmap_bf16(&L.m_wgu, L.wgu, 2 * ffn_l, H, 128));
    RC(make_tmap_bf16(&L.m_wdown, L.wdown, H, ffn_l, 128));
  }
  RC(make_tmap_bf16(&m_lm_head, lm_head, vocab_l, H, 128));

  layer_pool_elems = size_t(n_pages) * nkv_l * kPageTokens * kHeadDim;
  RC(dmalloc(&k_pool, layer_pool_elems * M.n_layers));
  RC(dmalloc(&v_pool, layer_pool_elems * M.n_layers));
  RC(make_tmap_attn_kv(&m_kpool, k_pool, M.n_layers, n_pages, nkv_l));
  RC(make_tmap_attn_kv(&m_vpool, v_pool, M.n_layers, n_pages, nkv_l));
  RC(dmalloc(&rope, size_t(cfg.max_ctx) * 64 * 2));
  RC(llmlb_op_rope_table(rope, cfg.max_ctx, M.rope_theta, st));
  RC(dmalloc(&d_block_tables, size_t(cfg.max_seqs) * pages_per_seq));

  RC(dmalloc(&x, size_t(t_cap) * H));
  RC(dmalloc(&sk_ws, kSkWsBytes / 4, false));
  RC(dmalloc(&sk_cnt, kSkCounters));
  if (tp > 1) {
    // the exchange region (tp_common.cuh): [pull barrier flags | TpFlags | slots | pair slots | rs-pair slots | logits | y]
    const size_t al = 1024;
    auto up = [&](size_t v) { return (v + al - 1) & ~(al - 1); };
    const size_t slot = up(std::max(size_t(kTpMaxSplit) * (t_cap + kTpMaxRanks) * H * 4, size_t(kTpMaxRanks) * kTpSmallRows * H * 4));
    const size_t lslot = up(size_t(cfg.max_seqs) * vocab_l * 4);
    size_t off = up(tp_region_prefix_bytes());
    tpc.flags_off = tp_region_prefix_bytes() - kTpFlagBytes;
    tpc.slot_off[0] = off; off += slot;
    tpc.slot_off[1] = off; off += slot;
    tpc.slot_bytes = slot;
    const size_t llslot = up(size_t(kTpMaxRanks) * kTpSmallRows * H * 8);
    tpc.ll_off[0] = off; off += llslot;
    tpc.ll_off[1] = off; off += llslot;
    const size_t rsslot = up(size_t(kTpMaxSplit) * (kTpLLTokens + kTpMaxRanks) * H * 4);   // parts x rows-per-owner <= split x (T + N)
    tpc.rsll_off[0] = off; off += rsslot;
    tpc.rsll_off[1] = off; off += rsslot;
    logits_slot_off = off; off += lslot;
    tpc.y_off = off; off += up(size_t(t_cap) * H * 2);
    xchg_bytes = off;
    RC(dmalloc(&xchg, xchg_bytes));
    y = reinterpret_cast<__nv_bfloat16*>(xchg + tpc.y_off);
    tpc.rank = rank; tpc.size = tp;
    for (auto& b : tpc.base) b = nullptr;
    tpc.base[rank] = xchg;
    // llmlb_op_allreduce (standalone pull all-reduce of the parity tests) borrows slot 0
    pull_slot_off = tpc.slot_off[0]; pull_slot_bytes = slot;
    RC(dmalloc(&xb, size_t(kTpSmallRows) * H));
    RC(dmalloc(&tp_stage, size_t(kTpSmallRows) * H));
    RC(dmalloc(&ylast, size_t(cfg.max_seqs) * H));
  } else {
    RC(dmalloc(&y, size_t(t_cap) * H));
  }
  RC(dmalloc(&qkv, size_t(t_cap) * qkv_w));
  RC(make_tmap_attn_q(&m_attn_q, qkv, t_cap, qkv_w));
  RC(dmalloc(&attn, size_t(t_cap) * nq_l * kHeadDim));
  RC(dmalloc(&h, size_t(t_cap) * ffn_l));
  RC(dmalloc(&logits, size_t(cfg.max_seqs) * M.vocab));
  RC(dmalloc(&x_last, size_t(cfg.max_seqs) * H));
  size_t ws = llmlb_op_decode_attention_ws(cfg.max_seqs, nq_l, 16);
  RC(dmalloc((uint8_t**)&attn_ws, ws));
  {
    const uint32_t boxes[5] = {16, 32, 64, 128, 256};
    for (int i = 0; i < 5; ++i) {
      RC(make_tmap_bf16(&m_y[i], y, t_cap, H, boxes[i]));
      RC(make_tmap_bf16(&m_attn[i], attn, t_cap, size_t(nq_l) * kHeadDim, boxes[i]));
      RC(make_tmap_bf16(&m_h[i], h, t_cap, ffn_l, boxes[i]));
      if (tp > 1) RC(make_tmap_bf16(&m_ylast[i], ylast, cfg.max_seqs, H, boxes[i]));
    }
  }
  RC(dmalloc(&d_ids, t_cap));
  RC(dmalloc(&d_pos, t_cap));
  RC(dmalloc(&d_page_of_tok, t_cap));
  RC(dmalloc(&d_tiles, size_t(t_cap / 64 + cfg.max_seqs + 1) * 4));
  RC(dmalloc(&d_last_rows, cfg.max_seqs));
  const size_t ms = cfg.max_seqs;
  RC(dmalloc(&S.seq_len, ms)); RC(dmalloc(&S.last_token, ms)); RC(dmalloc(&S.temperature, ms));
  RC(dmalloc(&S.top_p, ms)); RC(dmalloc(&S.top_k, ms)); RC(dmalloc(&S.seed, ms)); RC(dmalloc(&S.step, ms));
  RC(dmalloc(&B.slots, ms)); RC(dmalloc(&B.ids, ms)); RC(dmalloc(&B.seq_lens, ms));
  RC(dmalloc(&B.temperature, ms)); RC(dmalloc(&B.top_p, ms)); RC(dmalloc(&B.top_k, ms));
  RC(dmalloc(&B.seed, ms)); RC(dmalloc(&B.step, ms)); RC(dmalloc(&B.out_ids, ms));
  // run_prefill's layout: ids, positions, pages [t_cap each] | tiles [tiles_cap x 4] | rows, slots, lens [max_seqs each]
  stage_bytes = size_t(t_cap) * 4 * 3 + size_t(t_cap / 64 + ms + 1) * 16 + ms * 4 * 3 + 256;
  for (int i = 0; i < kRing; ++i) {
    LLMLB_CUDA_CHECK(cudaHostAlloc((void**)&h_stage[i], stage_bytes, cudaHostAllocDefault));
    LLMLB_CUDA_CHECK(cudaHostAlloc((void**)&h_out[i], ms * 4, cudaHostAllocDefault));
  }
  if (tp == 1) RC(dmalloc(&part_ws, size_t(8) * t_cap * H, false));
  return LLMLB_OK;
}

static int synth(__nv_bfloat16* out, uint64_t rows, uint64_t cols, uint64_t out_ld, uint64_t row0,
                 uint64_t col0, uint64_t ld, uint64_t seed, uint32_t id, float std, cudaStream_t st) {
  uint64_t n = rows * cols;
  if (n == 0) return LLMLB_OK;
  uint32_t grid = (uint32_t)std::min<uint64_t>((n + 255) / 256, uint64_t(kNumSMs) * 16);
  synth_strided_kernel<<<grid, 256, 0, st>>>(out, rows, cols, out_ld, row0, col0, ld, seed, id,
                                             std / kSynthSumStd);
  LLMLB_LAUNCH_CHECK();
  return LLMLB_OK;
}
static int fill(__nv_bfloat16* p, uint64_t n, float v, cudaStream_t st) {
  fill_bf16_kernel<<<(uint32_t)std::min<uint64_t>((n + 255) / 256, 1024), 256, 0, st>>>(p, n, v);
  LLMLB_LAUNCH_CHECK();
  return LLMLB_OK;
}

// tensor ids: layer*16 + kind (0 q,1 k,2 v,3 o,4 gate,5 up,6 down); globals 0xFFFF0000+{0 embed,2 lm_head}
int llmlb_engine::gen_weights() {
  const uint64_t H = M.hidden, seed = cfg.synthetic_seed;
  const float sd = 0.02f;
  RC(synth(embed, M.vocab, H, H, 0, 0, H, seed, 0xFFFF0000u, sd, st));
  RC(fill(final_norm, H, 1.0f, st));
  RC(synth(lm_head, vocab_l, H, H, uint64_t(rank) * vocab_l, 0, H, seed, 0xFFFF0002u, sd, st));
  for (uint32_t l = 0; l < M.n_layers; ++l) {
    LayerW& L = layers[l];
    const uint32_t id = l * 16;
    const uint64_t qr = uint64_t(nq_l) * kHeadDim, kr = uint64_t(nkv_l) * kHeadDim;
    RC(synth(L.wqkv, qr, H, H, rank * qr, 0, H, seed, id + 0, sd, st));
    RC(synth(L.wqkv + qr * H, kr, H, H, rank * kr, 0, H, seed, id + 1, sd, st));
    RC(synth(L.wqkv + (qr + kr) * H, kr, H, H, rank * kr, 0, H, seed, id + 2, sd, st));
    RC(synth(L.wo, H, qr, qr, 0, rank * qr, uint64_t(M.n_heads) * kHeadDim, seed, id + 3, sd, st));
    RC(synth(L.wgu, ffn_l, H, 2 * H, uint64_t(rank) * ffn_l, 0, H, seed, id + 4, sd, st));      // even rows
    RC(synth(L.wgu + H, ffn_l, H, 2 * H, uint64_t(rank) * ffn_l, 0, H, seed, id + 5, sd, st));  // odd rows
    RC(synth(L.wdown, H, ffn_l, ffn_l, 0, uint64_t(rank) * ffn_l, M.ffn, seed, id + 6, sd, st));
    RC(fill(L.attn_norm, H, 1.0f, st));
    RC(fill(L.ffn_norm, H, 1.0f, st));
  }
  return LLMLB_OK;
}

// ------------------------------------------------------------------ forward passes ----------
// y[r, :] = src[rows[r], :]  (bf16 gather of the normalised rows that need logits; protocol B)
__global__ void gather_rows_bf16_kernel(const __nv_bfloat16* __restrict__ src, const int32_t* __restrict__ rows,
                                        __nv_bfloat16* __restrict__ out, uint32_t hidden) {
  const uint4* s4 = reinterpret_cast<const uint4*>(src + size_t(rows[blockIdx.x]) * hidden);
  uint4* d4 = reinterpret_cast<uint4*>(out + size_t(blockIdx.x) * hidden);
  for (uint32_t i = threadIdx.x; i < hidden / 8; i += blockDim.x) d4[i] = s4[i];
}

// One tensor-core projection of bf16 activations (T > 4).
int llmlb_engine::proj(const CUtensorMap& mw, const void*, const void*, const CUtensorMap* mx, void* out, uint32_t T,
                       uint32_t n_out, uint32_t k, uint32_t epi, uint32_t out_stride, int wait_coll) {
  TpPushRS tpp{};
  tpp.sk_ws = sk_ws; tpp.sk_cnt = sk_cnt;   // narrow projections K-split inside the kernel
  if (wait_coll >= 0) {   // tensor parallel: the activation operand is y of that collective (its all-gather flags gate the loads)
    tpp.ctx = tpc; tpp.wait_coll_plus1 = uint32_t(wait_coll) + 1;
  }
  return gemm_tc_launch(mw, mx[bn_index(tc_pick_bn(T))], out, T, n_out, k, epi, out_stride, st, &mx[bn_index(128)], nullptr, &tpp);
}

// RoPE + KV append + attention of layer l over the rows in qkv -> attn
int llmlb_engine::attention_block(uint32_t l, uint32_t T, bool decode, uint32_t nb, uint32_t n_tiles, bool pdl) {
  if (decode)
    return decode_attention_launch(qkv, kpool(l), vpool(l), d_block_tables, pages_per_seq, B.slots, B.seq_lens, nb,
                                   attn, nq_l, nkv_l, rope, decode_splits(nb), pdl, st);
  // both kernels are programmatic dependents: their set-up overlaps the tail of the kernel before
  RC(rope_append_launch(qkv, d_pos, d_page_of_tok, rope, kpool(l), vpool(l), T, nq_l, nkv_l, true, st));
  return prefill_attention_tc_launch(m_attn_q, m_kpool, m_vpool, l, d_block_tables, pages_per_seq, d_tiles, n_tiles, attn,
                                     nq_l, nkv_l, true, st);
}

// Runs the layer stack over T rows already embedded in x.  decode: rows are one new token per
// sequence (nb of them); else rows are prefill tokens described by d_pos/d_page_of_tok/d_tiles.
int llmlb_engine::forward_tokens(uint32_t T, bool decode, uint32_t nb, uint32_t n_tiles, FwdState* fs) {
  const uint32_t H = M.hidden;
  *fs = FwdState{};
  fs->xres = x;
  const bool small = T <= 4;
  if (tp > 1) {
    if (!tp_ready) { set_error("tensor-parallel engine: import the peer handles first (llmlb_engine_tp_import)"); return LLMLB_E_UNSUPPORTED; }
    RC(tp_step_begin(tpc, st));
    tp_coll = 0;
    return small ? forward_small_tp(T, decode, nb, n_tiles, fs) : forward_big_tp(T, decode, nb, n_tiles, fs);
  }
  // T > 4: the O / down projections write fp32 K-split partials into part_ws and the NEXT
  // normalisation folds them into the residual in slot order (deterministic; no atomics)
  const size_t part_stride = size_t(T) * H;
  uint32_t pending = 0;  // partial slots of the previous down projection not yet folded into x
  auto big_proj_parts = [&](const CUtensorMap& mw, const CUtensorMap* mx, uint32_t k, uint32_t* n_parts) -> int {
    return gemm_tc_launch(mw, mx[bn_index(tc_pick_bn(T))], part_ws, T, H, k, kEpiPartialF32, H, st,
                          &mx[bn_index(128)], n_parts);
  };
  for (uint32_t l = 0; l < M.n_layers; ++l) {
    LayerW& L = layers[l];
    const uint32_t ko = nq_l * kHeadDim;
    // --- attention block ---
    if (small) {
      RC(gemv_decode(L.wqkv, x, L.attn_norm, M.rms_eps, qkv, T, qkv_w, H, LLMLB_EPI_STORE_BF16, qkv_w, st));
    } else {
      RC(rmsnorm_parts_launch(x, part_ws, pending, part_stride, L.attn_norm, y, T, H, M.rms_eps, st));
      pending = 0;
      RC(proj(L.m_wqkv, L.wqkv, y, m_y, qkv, T, qkv_w, H, LLMLB_EPI_STORE_BF16, qkv_w));
    }
    // decode, layers >= 1: PDL launch (its K/V prefetch overlaps the QKV GEMV's tail); layer 0 is a
    // plain launch so that decode_prepare (seq_lens) is complete before any early prologue
    RC(attention_block(l, T, decode, nb, n_tiles, l > 0 && small));
    uint32_t n_o = 0;
    if (small) RC(gemv_decode(L.wo, attn, nullptr, M.rms_eps, x, T, H, ko, LLMLB_EPI_RESID_F32, H, st));
    else RC(big_proj_parts(L.m_wo, m_attn, ko, &n_o));
    // --- feed-forward block ---
    if (small) {
      RC(gemv_decode(L.wgu, x, L.ffn_norm, M.rms_eps, h, T, 2 * ffn_l, H, LLMLB_EPI_SILU_MUL, ffn_l, st));
      RC(gemv_decode(L.wdown, h, nullptr, M.rms_eps, x, T, H, ffn_l, LLMLB_EPI_RESID_F32, H, st));
    } else {
      RC(rmsnorm_parts_launch(x, part_ws, n_o, part_stride, L.ffn_norm, y, T, H, M.rms_eps, st));
      RC(proj(L.m_wgu, L.wgu, y, m_y, h, T, 2 * ffn_l, H, LLMLB_EPI_SILU_MUL, ffn_l));
      RC(big_proj_parts(L.m_wdown, m_h, ffn_l, &pending));
    }
  }
  // the last down projection's partials: fold into x (no normalisation: the logits path has its own)
  if (!small && pending) RC(rmsnorm_parts_launch(x, part_ws, pending, part_stride, nullptr, nullptr, T, H, M.rms_eps, st));
  return LLMLB_OK;
}

// Tensor parallel, T <= 4 (protocol A of tp_common.cuh): the O / down GEMVs push their partial rows
// to every rank, the NEXT projection's RMSNorm prologue folds them into the replicated residual.
// 5 launches per layer, all PDL-chained; no all-reduce kernel.
int llmlb_engine::forward_small_tp(uint32_t T, bool decode, uint32_t nb, uint32_t n_tiles, FwdState* fs) {
  const uint32_t H = M.hidden, ko = nq_l * kHeadDim;
  float* cur = x;
  float* oth = xb;
  int pending = -1;   // collective pushed but not yet folded into `cur`
  auto consume = [&](const void* w, const __nv_bfloat16* gain, void* out, uint32_t n_out, uint32_t epi, uint32_t out_stride) -> int {
    if (pending >= 0) {
      int rc = gemv_tp_consume(tpc, uint32_t(pending), w, cur, oth, gain, M.rms_eps, out, T, n_out, H, epi, out_stride, st);
      if (rc == LLMLB_E_UNSUPPORTED) {   // odd shape: fold with its own kernel, then the plain projection
        RC(tp_fold_rows(tpc, uint32_t(pending), cur, oth, T, H, st));
        rc = gemv_decode(w, oth, gain, M.rms_eps, out, T, n_out, H, epi, out_stride, st);
      }
      RC(rc);
      std::swap(cur, oth);
      pending = -1;
      return LLMLB_OK;
    }
    return gemv_decode(w, cur, gain, M.rms_eps, out, T, n_out, H, epi, out_stride, st);
  };
  auto push = [&](const void* w, const void* xin_bf16, uint32_t k) -> int {
    const uint32_t c = tp_coll++;
    int rc = gemv_tp_push(tpc, c, w, xin_bf16, T, H, k, st);
    if (rc == LLMLB_E_UNSUPPORTED) {
      RC(llmlb_op_gemv(w, xin_bf16, nullptr, M.rms_eps, tp_stage, T, H, k, LLMLB_EPI_STORE_F32, H, st));
      rc = tp_push_rows(tpc, c, tp_stage, T, H, st);
    }
    RC(rc);
    pending = int(c);
    return LLMLB_OK;
  };
  for (uint32_t l = 0; l < M.n_layers; ++l) {
    LayerW& L = layers[l];
    RC(consume(L.wqkv, L.attn_norm, qkv, qkv_w, LLMLB_EPI_STORE_BF16, qkv_w));
    RC(attention_block(l, T, decode, nb, n_tiles, l > 0));
    RC(push(L.wo, attn, ko));
    RC(consume(L.wgu, L.ffn_norm, h, 2 * ffn_l, LLMLB_EPI_SILU_MUL, ffn_l));
    RC(push(L.wdown, h, ffn_l));
  }
  fs->xres = cur; fs->xother = oth;
  fs->pending = true; fs->pending_coll = uint32_t(pending);
  return LLMLB_OK;
}

int llmlb_engine::finish_small_tp(FwdState* fs, uint32_t T) {
  if (!fs->pending) return LLMLB_OK;
  RC(tp_fold_rows(tpc, fs->pending_coll, fs->xres, fs->xother, T, M.hidden, st));
  std::swap(fs->xres, fs->xother);
  fs->pending = false;
  return LLMLB_OK;
}

// Tensor parallel, T > 4 (protocol B): the O / down GEMM epilogues reduce-scatter their fp32 tiles by
// address into the row owners' slots; tp_reduce_norm folds the owned rows into the (row-sharded)
// residual, normalises and all-gathers the bf16 rows into every rank's y.
int llmlb_engine::forward_big_tp(uint32_t T, bool decode, uint32_t nb, uint32_t n_tiles, FwdState* fs) {
  const uint32_t H = M.hidden, ko = nq_l * kHeadDim;
  const uint32_t rpr = ceil_div(T, tp);
  // returns the collective's index; last: the consumers of y behind it are not tensor-core GEMMs of
  // this loop, so the reduce kernel itself waits for the all-gather
  auto push_rs = [&](const CUtensorMap& mw, const CUtensorMap* mx, uint32_t k, const __nv_bfloat16* next_gain, bool last, int* coll) -> int {
    TpPushRS tpp{};
    tpp.ctx = tpc; tpp.coll = tp_coll++; tpp.rpr = rpr;
    *coll = int(tpp.coll);
    uint32_t n_parts = 1;
    const bool ll = T <= kTpLLTokens;   // narrow steps: {value, epoch} words, no flag round
    RC(gemm_tc_launch(mw, mx[bn_index(tc_pick_bn(T))], nullptr, T, H, k, ll ? kEpiPushRSLL : kEpiPushRS, H, st, &mx[bn_index(128)], &n_parts,
                      &tpp, kTpMaxSplit));
    return tp_reduce_norm(tpc, tpp.coll, x, next_gain, T, H, M.rms_eps, n_parts, last, ll, st);
  };
  // layer 0: the embedding rows are complete on every rank
  RC(llmlb_op_rmsnorm(x, layers[0].attn_norm, y, T, H, M.rms_eps, st));
  int c_prev = -1;   // collective whose all-gathered y the next projection consumes
  for (uint32_t l = 0; l < M.n_layers; ++l) {
    LayerW& L = layers[l];
    RC(proj(L.m_wqkv, L.wqkv, y, m_y, qkv, T, qkv_w, H, LLMLB_EPI_STORE_BF16, qkv_w, c_prev));
    RC(attention_block(l, T, decode, nb, n_tiles, false));
    RC(push_rs(L.m_wo, m_attn, ko, L.ffn_norm, false, &c_prev));
    RC(proj(L.m_wgu, L.wgu, y, m_y, h, T, 2 * ffn_l, H, LLMLB_EPI_SILU_MUL, ffn_l, c_prev));
    const bool last = l + 1 == M.n_layers;
    RC(push_rs(L.m_wdown, m_h, ffn_l, last ? final_norm : layers[l + 1].attn_norm, last, &c_prev));
  }
  fs->y_final = true;
  return LLMLB_OK;
}

// ---- logits ----
int llmlb_engine::logits_gather(uint32_t R) {
  if (tp == 1) return LLMLB_OK;
  return ar_allgather_cols(tpc, logits_slot_off, logits, R, vocab_l, st);
}
// logits[r, :] for R fp32 residual rows at src (final RMSNorm applied here)
int llmlb_engine::logits_from_x(const float* src, uint32_t R) {
  const uint32_t H = M.hidden;
  float* dst = logits_dst();
  if (R <= 4) {
    RC(llmlb_op_gemv(lm_head, src, final_norm, M.rms_eps, dst, R, vocab_l, H, LLMLB_EPI_STORE_F32, vocab_l, st));
  } else {
    RC(llmlb_op_rmsnorm(src, final_norm, y, R, H, M.rms_eps, st));
    RC(gemm_tc_launch(m_lm_head, m_y[bn_index(tc_pick_bn(R))], dst, R, vocab_l, H, LLMLB_EPI_STORE_F32, vocab_l, st, &m_y[bn_index(128)]));
  }
  return logits_gather(R);
}
// rows already normalised (bf16): the lm_head projection alone
int llmlb_engine::logits_from_y(const __nv_bfloat16* src, const CUtensorMap* maps, uint32_t R) {
  const uint32_t H = M.hidden;
  float* dst = logits_dst();
  if (R <= 4) RC(llmlb_op_gemv(lm_head, src, nullptr, M.rms_eps, dst, R, vocab_l, H, LLMLB_EPI_STORE_F32, vocab_l, st));
  else RC(gemm_tc_launch(m_lm_head, maps[bn_index(tc_pick_bn(R))], dst, R, vocab_l, H, LLMLB_EPI_STORE_F32, vocab_l, st, &maps[bn_index(128)]));
  return logits_gather(R);
}
// protocol A, decode: the lm_head GEMV's prologue consumes the last down projection's collective
int llmlb_engine::logits_tp_consume(FwdState* fs, uint32_t R) {
  int rc = gemv_tp_consume(tpc, fs->pending_coll, lm_head, fs->xres, fs->xother, final_norm, M.rms_eps, logits_dst(), R,
                           vocab_l, M.hidden, LLMLB_EPI_STORE_F32, vocab_l, st);
  if (rc == LLMLB_E_UNSUPPORTED) {
    RC(finish_small_tp(fs, R));
    return logits_from_x(fs->xres, R);
  }
  RC(rc);
  std::swap(fs->xres, fs->xother);
  fs->pending = false;
  return logits_gather(R);
}
// decode: logits of rows 0..R of the step; prefill: logits of the rows listed in d_last_rows
int llmlb_engine::logits_after_forward(FwdState* fs, uint32_t R, bool decode) {
  if (fs->y_final) {
    if (decode) return logits_from_y(y, m_y, R);
    gather_rows_bf16_kernel<<<R, 128, 0, st>>>(y, d_last_rows, ylast, M.hidden);
    LLMLB_LAUNCH_CHECK();
    return logits_from_y(ylast, m_ylast, R);
  }
  if (decode) {
    if (fs->pending) return logits_tp_consume(fs, R);
    return logits_from_x(fs->xres, R);
  }
  return LLMLB_E_INTERNAL;   // prefill with fp32 residual: run_prefill gathers the rows itself
}

int llmlb_engine::layer_stack_decode(uint32_t nb) {
  decode_prepare_kernel<<<ceil_div(nb, 128), 128, 0, st>>>(S, B, nb);
  LLMLB_LAUNCH_CHECK();
  RC(llmlb_op_embed(embed, B.ids, x, nb, M.hidden, M.vocab, st));
  FwdState fs;
  RC(forward_tokens(nb, true, nb, 0, &fs));
  RC(logits_after_forward(&fs, nb, true));
  RC(llmlb_op_sample(logits, nb, M.vocab, B.temperature, B.top_p, B.top_k, B.seed, B.step, B.out_ids, st));
  step_finish_kernel<<<ceil_div(nb, 128), 128, 0, st>>>(S, B, nb);
  LLMLB_LAUNCH_CHECK();
  return LLMLB_OK;
}

int llmlb_engine::launch_decode_step(uint32_t nb) {
  if (!cfg.use_cuda_graphs) return layer_stack_decode(nb);
  auto it = graphs.find(nb);
  if (it == graphs.end()) {
    // kernel attributes (max dynamic smem) were set by the eager warm-up in init()
    cudaGraph_t g = nullptr;
    uint64_t launches_before = g_kernel_launches.load();
    LLMLB_CUDA_CHECK(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
    int rc = layer_stack_decode(nb);
    cudaError_t ce = cudaStreamEndCapture(st, &g);
    if (rc != LLMLB_OK) { if (g) cudaGraphDestroy(g); return rc; }
    if (ce != cudaSuccess) { set_error(std::string("graph capture: ") + cudaGetErrorString(ce)); return LLMLB_E_DEVICE; }
    cudaGraphExec_t ge = nullptr;
    LLMLB_CUDA_CHECK(cudaGraphInstantiate(&ge, g, 0));
    cudaGraphDestroy(g);
    graphs[nb] = ge;
    graph_nodes[nb] = g_kernel_launches.load() - launches_before;
    g_kernel_launches.store(launches_before);  // capture did not execute anything
    it = graphs.find(nb);
  }
  LLMLB_CUDA_CHECK(cudaGraphLaunch(it->second, st));
  g_kernel_launches.fetch_add(graph_nodes[nb]);
  return LLMLB_OK;
}

// ------------------------------------------------------------------ steps -------------------
__global__ void iota_kernel(int32_t* p, uint32_t n) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = int32_t(i);
}
__global__ void slot_init_kernel(SlotState S, int32_t slot, float temperature, float top_p,
                                 int32_t top_k, uint64_t seed, uint64_t step0) {
  S.seq_len[slot] = 0;
  S.last_token[slot] = 0;
  S.temperature[slot] = temperature;
  S.top_p[slot] = top_p;
  S.top_k[slot] = top_k;
  S.seed[slot] = seed;
  S.step[slot] = step0;   // a preempted sequence resumes its sampler stream where it stopped
}
__global__ void prefill_finish_kernel(SlotState S, BatchView B, uint32_t n) {
  uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= n) return;
  S.seq_len[B.slots[b]] = B.seq_lens[b];  // tokens now in the cache
}

cudaEvent_t llmlb_engine::get_event() {
  if (!ev_pool.empty()) {
    cudaEvent_t e = ev_pool.back();
    ev_pool.pop_back();
    return e;
  }
  cudaEvent_t e = nullptr;
  cudaEventCreate(&e);
  return e;
}

// reqs[i] contributes take[i] prompt tokens starting at reqs[i]->prefilled
int llmlb_engine::run_prefill(const std::vector<ReqPtr>& reqs, const std::vector<uint32_t>& take) {
  uint32_t T = 0;
  for (uint32_t t : take) T += t;
  uint8_t* stg = next_stage();
  int32_t* s_ids = reinterpret_cast<int32_t*>(stg);
  int32_t* s_pos = s_ids + t_cap;
  int32_t* s_page = s_pos + t_cap;
  int32_t* s_tiles = s_page + t_cap;
  const uint32_t tiles_cap = t_cap / 64 + cfg.max_seqs + 1;
  int32_t* s_rows = s_tiles + size_t(tiles_cap) * 4;
  int32_t* s_slots = s_rows + cfg.max_seqs;
  int32_t* s_lens = s_slots + cfg.max_seqs;

  InflightStep step;
  step.is_prefill = true;
  step.n_tokens = T;
  uint32_t row = 0, n_tiles = 0, R = 0;
  for (size_t i = 0; i < reqs.size(); ++i) {
    Request& r = *reqs[i];
    if (r.prefilled == 0) {  // first chunk: publish block table + sampler state
      LLMLB_CUDA_CHECK(cudaMemcpyAsync(d_block_tables + size_t(r.slot) * pages_per_seq, r.pages.data(),
                                       r.pages.size() * 4, cudaMemcpyHostToDevice, st));
      slot_init_kernel<<<1, 1, 0, st>>>(S, r.slot, r.s.temperature, r.s.top_p, (int32_t)r.s.top_k, r.s.seed, uint64_t(r.harvested));
      LLMLB_LAUNCH_CHECK();
      r.pages_published = uint32_t(r.pages.size());
    }
    const uint32_t p0 = r.prefilled;
    for (uint32_t j = 0; j < take[i]; ++j) {
      uint32_t pos = p0 + j;
      s_ids[row + j] = r.prompt[pos];
      s_pos[row + j] = int32_t(pos);
      s_page[row + j] = r.pages[pos / kPageTokens];
    }
    for (uint32_t j = 0; j < take[i]; j += kPfTile) {
      s_tiles[n_tiles * 4 + 0] = int32_t(row + j);
      s_tiles[n_tiles * 4 + 1] = int32_t(std::min<uint32_t>(kPfTile, take[i] - j));
      s_tiles[n_tiles * 4 + 2] = int32_t(p0 + j);
      s_tiles[n_tiles * 4 + 3] = r.slot;
      ++n_tiles;
    }
    if (p0 + take[i] == r.prompt.size()) {
      s_rows[R] = int32_t(row + take[i] - 1);
      s_slots[R] = r.slot;
      s_lens[R] = int32_t(r.prompt.size());
      step.reqs.push_back(reqs[i]);
      ++R;
    }
    row += take[i];
  }
  // note: r.pages.data() above is pageable host memory: the async copy is staged by the driver
  LLMLB_CUDA_CHECK(cudaMemcpyAsync(d_ids, s_ids, T * 4, cudaMemcpyHostToDevice, st));
  LLMLB_CUDA_CHECK(cudaMemcpyAsync(d_pos, s_pos, T * 4, cudaMemcpyHostToDevice, st));
  LLMLB_CUDA_CHECK(cudaMemcpyAsync(d_page_of_tok, s_page, T * 4, cudaMemcpyHostToDevice, st));
  LLMLB_CUDA_CHECK(cudaMemcpyAsync(d_tiles, s_tiles, n_tiles * 16, cudaMemcpyHostToDevice, st));
  if (R) {
    LLMLB_CUDA_CHECK(cudaMemcpyAsync(d_last_rows, s_rows, R * 4, cudaMemcpyHostToDevice, st));
    LLMLB_CUDA_CHECK(cudaMemcpyAsync(B.slots, s_slots, R * 4, cudaMemcpyHostToDevice, st));
    LLMLB_CUDA_CHECK(cudaMemcpyAsync(B.seq_lens, s_lens, R * 4, cudaMemcpyHostToDevice, st));
    cur_batch_slots.clear();  // B.slots no longer holds a decode batch
  }
  step.ev_start = get_event();
  step.ev_end = get_event();
  LLMLB_CUDA_CHECK(cudaEventRecord(step.ev_start, st));
  RC(llmlb_op_embed(embed, d_ids, x, T, M.hidden, M.vocab, st));
  FwdState fs;
  RC(forward_tokens(T, false, 0, n_tiles, &fs));
  if (!fs.y_final) RC(finish_small_tp(&fs, T));   // tp, T <= 4: every rank folds the last collective (also when R == 0)
  if (R) {
    if (fs.y_final) {
      RC(logits_after_forward(&fs, R, false));
    } else {
      gather_rows_kernel<<<R, 256, 0, st>>>(fs.xres, d_last_rows, x_last, M.hidden);
      LLMLB_LAUNCH_CHECK();
      RC(logits_from_x(x_last, R));
    }
    sample_prepare_kernel<<<ceil_div(R, 128), 128, 0, st>>>(S, B, R);
    LLMLB_LAUNCH_CHECK();
    RC(llmlb_op_sample(logits, R, M.vocab, B.temperature, B.top_p, B.top_k, B.seed, B.step, B.out_ids, st));
    step_finish_kernel<<<ceil_div(R, 128), 128, 0, st>>>(S, B, R);
    LLMLB_LAUNCH_CHECK();
    prefill_finish_kernel<<<ceil_div(R, 128), 128, 0, st>>>(S, B, R);
    LLMLB_LAUNCH_CHECK();
    step.host_ids = h_out[(out_seq++) % kRing];
    LLMLB_CUDA_CHECK(cudaMemcpyAsync(step.host_ids, B.out_ids, R * 4, cudaMemcpyDeviceToHost, st));
  }
  LLMLB_CUDA_CHECK(cudaEventRecord(step.ev_end, st));
  {
    // bookkeeping that API threads read (health counters; `inflight` in the debug hooks and the plan-channel attach) is
    // written under mu — ThreadSanitizer over the fake CUDA runtime flagged the deque (step_mu alone is held here)
    std::lock_guard<std::mutex> lk(mu);
    for (size_t i = 0; i < reqs.size(); ++i) {
      reqs[i]->prefilled += take[i];
      if (reqs[i]->prefilled == reqs[i]->prompt.size()) reqs[i]->launched = reqs[i]->harvested + 1;
    }
    steps_prefill++;
    tokens_prefill += T;
    inflight.push_back(std::move(step));
  }
  return LLMLB_OK;
}

int llmlb_engine::run_decode(const std::vector<ReqPtr>& batch) {
  const uint32_t nb = (uint32_t)batch.size();
  std::vector<int32_t> slots(nb);
  for (uint32_t b = 0; b < nb; ++b) slots[b] = batch[b]->slot;
  if (slots != cur_batch_slots) {
    int32_t* stg = reinterpret_cast<int32_t*>(next_stage());
    memcpy(stg, slots.data(), nb * 4);
    LLMLB_CUDA_CHECK(cudaMemcpyAsync(B.slots, stg, nb * 4, cudaMemcpyHostToDevice, st));
    cur_batch_slots = slots;
  }
  {   // pages taken since the last step (a sequence crossing a 64-token boundary): patch the device block table
    uint32_t n_new = 0;
    for (auto& r : batch) n_new += uint32_t(r->pages.size()) - r->pages_published;
    if (n_new) {
      int32_t* stg = reinterpret_cast<int32_t*>(next_stage());
      uint32_t off = 0;
      for (auto& r : batch) {
        const uint32_t have = r->pages_published, now = uint32_t(r->pages.size());
        if (now == have) continue;
        memcpy(stg + off, r->pages.data() + have, size_t(now - have) * 4);
        LLMLB_CUDA_CHECK(cudaMemcpyAsync(d_block_tables + size_t(r->slot) * pages_per_seq + have, stg + off, size_t(now - have) * 4,
                                         cudaMemcpyHostToDevice, st));
        off += now - have;
        r->pages_published = now;
      }
    }
  }
  InflightStep step;
  step.n_tokens = nb;
  step.reqs = batch;
  step.ev_start = get_event();
  step.ev_end = get_event();
  LLMLB_CUDA_CHECK(cudaEventRecord(step.ev_start, st));
  RC(launch_decode_step(nb));
  step.host_ids = h_out[(out_seq++) % kRing];
  LLMLB_CUDA_CHECK(cudaMemcpyAsync(step.host_ids, B.out_ids, nb * 4, cudaMemcpyDeviceToHost, st));
  LLMLB_CUDA_CHECK(cudaEventRecord(step.ev_end, st));
  {
    std::lock_guard<std::mutex> lk(mu);
    for (auto& r : batch) r->launched++;
    steps_decode++;
    tokens_decode += nb;
    inflight.push_back(std::move(step));
  }
  return LLMLB_OK;
}

void llmlb_engine::release_resources(ReqPtr r) {  // mu held
  if (r->slot >= 0) {
    free_slots.push_back(r->slot);
    r->slot = -1;
  }
  for (int32_t p : r->pages) free_pages.push_back(p);
  r->pages.clear();
  r->pages_published = 0;
  running.erase(std::remove(running.begin(), running.end(), r), running.end());
}

// Evict a running sequence: its pages and slot go back to the pools and it returns to the HEAD of the
// queue with its context extended by what it generated (recomputed at re-admission).  Only called
// with nothing in flight, so every launched token has been harvested.  mu held.
void llmlb_engine::preempt(ReqPtr r) {
  r->prompt.insert(r->prompt.end(), r->gen.begin() + r->gen_in_prompt, r->gen.end());
  r->gen_in_prompt = uint32_t(r->gen.size());
  r->prefilled = 0;
  r->launched = r->harvested;
  r->preempted++;
  release_resources(r);
  waiting.push_front(r);
  preemptions++;
}

void llmlb_engine::finish_request(ReqPtr r, uint32_t reason) {  // mu held
  if (r->finished) return;
  r->finished = true;
  r->finish_reason = reason;
  if (r->events.empty() || r->events.back().finish_reason == LLMLB_FINISH_NONE) {
    if (!r->events.empty() && (reason == LLMLB_FINISH_STOP || reason == LLMLB_FINISH_LENGTH)) {
      r->events.back().finish_reason = reason;
    } else {
      llmlb_token_event ev{};
      ev.token_id = -1;
      ev.index = r->harvested;
      ev.finish_reason = reason;
      ev.prompt_tokens = r->n_prompt0;
      ev.completion_tokens = r->harvested;
      ev.t_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - r->t_submit).count();
      r->events.push_back(ev);
    }
  }
  release_resources(r);
  if (r->client_released) requests.erase(r->id);
  cv_events.notify_all();
}

void llmlb_engine::harvest_one() {
  InflightStep step;
  {
    std::lock_guard<std::mutex> lk(mu);      // readers of `inflight` on API threads hold mu
    step = std::move(inflight.front());
    inflight.pop_front();
  }
  cudaError_t ce = cudaEventSynchronize(step.ev_end);
  float ms = 0.f;
  if (ce == cudaSuccess) cudaEventElapsedTime(&ms, step.ev_start, step.ev_end);
  std::lock_guard<std::mutex> lk(mu);
  if (step.is_prefill) gpu_ms_prefill += ms; else gpu_ms_decode += ms;
  ev_pool.push_back(step.ev_start);
  ev_pool.push_back(step.ev_end);
  auto now = std::chrono::steady_clock::now();
  for (size_t b = 0; b < step.reqs.size(); ++b) {
    const ReqPtr& r = step.reqs[b];
    if (r->finished) continue;  // tokens computed past a stop are dropped
    if (ce != cudaSuccess) { finish_request(r, LLMLB_FINISH_ERROR); continue; }
    const int32_t tok = step.host_ids[b];
    llmlb_token_event ev{};
    ev.token_id = tok;
    ev.index = r->harvested++;
    r->gen.push_back(tok);
    ev.prompt_tokens = r->n_prompt0;
    ev.completion_tokens = r->harvested;
    ev.t_ms = std::chrono::duration<double, std::milli>(now - r->t_submit).count();
    r->events.push_back(ev);
    bool stop_hit = false;
    if (!r->s.ignore_eos)
      for (int32_t sid : r->stop_ids) stop_hit |= (sid == tok);
    if (stop_hit) finish_request(r, LLMLB_FINISH_STOP);
    else if (r->harvested >= r->s.max_tokens) finish_request(r, LLMLB_FINISH_LENGTH);
  }
  cv_events.notify_all();
}

// One scheduling iteration: apply cancellations, pick the next step (prefill chunks first, then
// a decode step over every running sequence), launch it.  `lk` (mu) is held on entry and released
// before the launch.  Deterministic in the scheduler state, which is what lets follower ranks
// replay it (PlanChannel).
bool llmlb_engine::sched_iteration(std::unique_lock<std::mutex>& lk) {
  std::vector<ReqPtr> pf_reqs;
  std::vector<uint32_t> pf_take;
  std::vector<ReqPtr> dec;
  if (!fatal_error.empty()) {   // failed engine (device error, dead follower): everything in flight ends with an error event
    for (auto& r : std::vector<ReqPtr>(running)) finish_request(r, LLMLB_FINISH_ERROR);
    while (!waiting.empty()) { ReqPtr r = waiting.front(); waiting.pop_front(); finish_request(r, LLMLB_FINISH_ERROR); }
    cv_events.notify_all();
    lk.unlock();
    return false;
  }
  // cancellations (client cancel / release, queue timeout, deadline: cancel_reason says which)
  for (auto it = waiting.begin(); it != waiting.end();) {
    if ((*it)->cancel) { ReqPtr r = *it; it = waiting.erase(it); finish_request(r, r->cancel_reason); }
    else ++it;
  }
  for (size_t i = 0; i < running.size();) {
    if (running[i]->cancel && !running[i]->finished) finish_request(running[i], running[i]->cancel_reason);
    else ++i;
  }
  if (!paused) {
    uint32_t budget = cfg.max_step_tokens;
    // continue chunked prefills first
    for (auto& r : running) {
      if (budget == 0) break;
      if (r->prefilled < r->prompt.size()) {
        uint32_t t = std::min<uint32_t>(budget, (uint32_t)r->prompt.size() - r->prefilled);
        pf_reqs.push_back(r); pf_take.push_back(t); budget -= t;
      }
    }
    // admit in FIFO order while a slot, the pages of the CONTEXT (prompt, plus what a preempted
    // sequence had generated) and token budget exist.  Pages for generated tokens are taken one at a
    // time as a sequence crosses a page boundary; when the pool runs dry the most recently admitted
    // sequence is evicted and recomputed later (below).
    while (!waiting.empty() && budget > 0 && !free_slots.empty()) {
      ReqPtr r = waiting.front();
      uint32_t need = ceil_div((uint32_t)r->prompt.size(), kPageTokens);
      // first admission keeps one page per running sequence in reserve, so that admitting does not
      // immediately force an eviction
      const size_t reserve = r->admitted_once ? 0 : running.size();
      if (need + reserve > free_pages.size() && !(running.empty() && need <= free_pages.size())) break;
      waiting.pop_front();
      r->slot = free_slots.back(); free_slots.pop_back();
      for (uint32_t i = 0; i < need; ++i) { r->pages.push_back(free_pages.back()); free_pages.pop_back(); }
      r->admitted_once = true;
      running.push_back(r);
      uint32_t t = std::min<uint32_t>(budget, (uint32_t)r->prompt.size());
      pf_reqs.push_back(r); pf_take.push_back(t); budget -= t;
    }
    if (pf_reqs.empty()) {
      for (auto& r : running)
        if (!r->finished && r->prefilled == r->prompt.size() && r->launched < r->s.max_tokens)
          dec.push_back(r);
      // every sequence of the step needs the page that holds position n_prompt0 + launched - 1
      bool shortage = false;
      for (auto& r : dec) {
        const uint32_t need = ceil_div(r->n_prompt0 + r->launched, kPageTokens);
        while (r->pages.size() < need) {
          if (free_pages.empty()) { shortage = true; break; }
          r->pages.push_back(free_pages.back()); free_pages.pop_back();
        }
        if (shortage) break;
      }
      if (shortage) {
        dec.clear();
        if (inflight.empty()) {
          // nothing in flight: every launched token is known, so a sequence can be evicted.  Victim:
          // the most recently admitted one (the oldest always makes progress).
          ReqPtr victim;
          for (auto it = running.rbegin(); it != running.rend(); ++it) if (!(*it)->finished) { victim = *it; break; }
          if (victim && running.size() > 1) preempt(victim);
          else if (victim) finish_request(victim, LLMLB_FINISH_ERROR);   // a lone sequence the pool cannot hold
          lk.unlock();
          return true;    // state changed: schedule again at once
        }
        // steps in flight: the loop harvests them first, then comes back here
      }
    }
  }
  lk.unlock();
  if (pf_reqs.empty() && dec.empty()) return false;
  std::lock_guard<std::mutex> sl(step_mu);
  int rc = !pf_reqs.empty() ? run_prefill(pf_reqs, pf_take) : run_decode(dec);
  if (rc != LLMLB_OK) {
    std::string msg = g_err;
    cudaStreamSynchronize(st);
    std::lock_guard<std::mutex> lk2(mu);
    fatal_error = msg;
    for (auto& r : std::vector<ReqPtr>(running)) finish_request(r, LLMLB_FINISH_ERROR);
  }
  return true;
}

// Time-based decisions belong to ONE clock: the single rank's, or rank 0's under a plan channel
// (followers replay kPlanExpire).  Lock-step tensor parallelism without a plan channel has no
// timeouts.  mu held.
void llmlb_engine::expire_requests() {
  if (tp > 1 && !(plan_on && plan.leader)) return;
  if (!cfg.queue_timeout_ms && !cfg.request_timeout_ms) return;
  const auto now = std::chrono::steady_clock::now();
  auto mark = [&](const ReqPtr& r, uint32_t reason) {
    r->cancel = true;
    r->cancel_reason = reason;
    uint8_t rec[12];
    memcpy(rec, &r->id, 8); memcpy(rec + 8, &reason, 4);
    plan_log(kPlanExpire, rec, 12);
  };
  for (auto& r : waiting) {
    if (r->cancel) continue;
    const double ms = std::chrono::duration<double, std::milli>(now - r->t_submit).count();
    if (cfg.request_timeout_ms && ms > cfg.request_timeout_ms) mark(r, LLMLB_FINISH_DEADLINE);
    else if (cfg.queue_timeout_ms && !r->admitted_once && ms > cfg.queue_timeout_ms) mark(r, LLMLB_FINISH_QUEUE_TIMEOUT);
  }
  if (cfg.request_timeout_ms)
    for (auto& r : running) {
      if (r->cancel || r->finished) continue;
      if (std::chrono::duration<double, std::milli>(now - r->t_submit).count() > cfg.request_timeout_ms) mark(r, LLMLB_FINISH_DEADLINE);
    }
}

void llmlb_engine::loop() {
  cudaSetDevice(cfg.device);
  for (;;) {
    bool launched = false;
    {
      std::unique_lock<std::mutex> lk(mu);
      cv_sched.wait(lk, [&] {
        return stop || (plan_on && !plan.leader) || !inflight.empty() || (!paused && (!waiting.empty() || !running.empty()));
      });
      if (stop) break;
      if (plan_on && !plan.leader) { lk.unlock(); loop_follower(); return; }
      expire_requests();               // logged as kPlanExpire before the iteration that applies them
      plan_log(kPlanSched);            // followers run the same iteration, concurrently with ours
      launched = sched_iteration(lk);
    }
    while (inflight.size() > lookahead || (!launched && !inflight.empty())) {
      plan_log_locked(kPlanHarvest);
      harvest_one();
      launched = true;  // harvest at most until the window is back to `lookahead`
      if (inflight.size() <= lookahead) break;
    }
  }
  while (!inflight.empty()) { plan_log_locked(kPlanHarvest); harvest_one(); }
  plan_log_locked(kPlanStop);
}

// Follower rank of a tensor-parallel group: replay rank 0's log.  Nobody polls requests here, so
// they are created already released (freed when they finish).
void llmlb_engine::loop_follower() {
  std::vector<uint8_t> buf;
  for (;;) {
    const uint32_t type = plan.read(&buf, plan_abort);
    if (type == 0 || type == kPlanStop) break;
    switch (type) {
      case kPlanSubmit: {
        if (buf.size() < sizeof(uint64_t) + sizeof(llmlb_sampling) + 8) break;
        const uint8_t* p = buf.data();
        auto r = std::make_shared<Request>();
        memcpy(&r->id, p, 8); p += 8;
        memcpy(&r->s, p, sizeof(llmlb_sampling)); p += sizeof(llmlb_sampling);
        uint32_t n_prompt = 0, n_stop = 0;
        memcpy(&n_prompt, p, 4); memcpy(&n_stop, p + 4, 4); p += 8;
        r->prompt.assign(reinterpret_cast<const int32_t*>(p), reinterpret_cast<const int32_t*>(p) + n_prompt);
        r->n_prompt0 = n_prompt;
        p += size_t(n_prompt) * 4;
        r->stop_ids.assign(reinterpret_cast<const int32_t*>(p), reinterpret_cast<const int32_t*>(p) + n_stop);
        r->s.stop_ids = nullptr;
        r->client_released = true;
        r->t_submit = std::chrono::steady_clock::now();
        std::lock_guard<std::mutex> lk(mu);
        requests[r->id] = r;
        waiting.push_back(r);
        break;
      }
      case kPlanCancel:
      case kPlanRelease: {
        uint64_t id = 0;
        if (buf.size() >= 8) memcpy(&id, buf.data(), 8);
        std::lock_guard<std::mutex> lk(mu);
        auto it = requests.find(id);
        if (it != requests.end()) it->second->cancel = true;
        break;
      }
      case kPlanPause: {
        std::lock_guard<std::mutex> lk(mu);
        paused = !buf.empty() && buf[0] != 0;
        break;
      }
      case kPlanExpire: {
        uint64_t id = 0; uint32_t reason = LLMLB_FINISH_CANCELLED;
        if (buf.size() >= 12) { memcpy(&id, buf.data(), 8); memcpy(&reason, buf.data() + 8, 4); }
        std::lock_guard<std::mutex> lk(mu);
        auto it = requests.find(id);
        if (it != requests.end()) { it->second->cancel = true; it->second->cancel_reason = reason; }
        break;
      }
      case kPlanSched: {
        std::unique_lock<std::mutex> lk(mu);
        sched_iteration(lk);
        break;
      }
      case kPlanHarvest:
        if (!inflight.empty()) harvest_one();
        break;
      default:
        break;
    }
  }
  while (!inflight.empty()) harvest_one();
}

// ------------------------------------------------------------------ C ABI -------------------
extern "C" uint32_t llmlb_abi_version(void) { return LLMLB_ABI_VERSION; }
extern "C" const char* llmlb_last_error(void) { return g_err.c_str(); }

extern "C" int llmlb_engine_create(const llmlb_engine_config* cfg, llmlb_engine** out) {
  if (!cfg || !out) { set_error("llmlb_engine_create: null argument"); return LLMLB_E_INVALID_ARG; }
  int n_dev = 0;
  if (cudaGetDeviceCount(&n_dev) != cudaSuccess || n_dev == 0) {
    set_error("llmlb_engine_create: no CUDA device (this library has no CPU path)");
    return LLMLB_E_DEVICE;
  }
  if (cfg->device < 0 || cfg->device >= n_dev) { set_error("llmlb_engine_create: bad device ordinal"); return LLMLB_E_INVALID_ARG; }
  llmlb_engine* e = new llmlb_engine();
  e->cfg = *cfg;
  int rc = e->init();
  if (rc != LLMLB_OK) {
    std::string msg = g_err;
    llmlb_engine_destroy(e);
    set_error(msg);
    return rc;
  }
  *out = e;
  return LLMLB_OK;
}

extern "C" void llmlb_engine_destroy(llmlb_engine* e) {
  if (!e) return;
  {
    std::lock_guard<std::mutex> lk(e->mu);
    e->stop = true;
  }
  e->plan_abort.store(true);
  e->cv_sched.notify_all();
  if (e->worker.joinable()) e->worker.join();
  if (e->plan_on) e->plan.close_channel();
  cudaSetDevice(e->cfg.device);
  if (e->st) cudaStreamSynchronize(e->st);
  for (auto& kv : e->graphs) cudaGraphExecDestroy(kv.second);
  auto F = [](void* p) { if (p) cudaFree(p); };
  F(e->embed); F(e->final_norm); F(e->lm_head);
  for (auto& L : e->layers) { F(L.wqkv); F(L.wo); F(L.wgu); F(L.wdown); F(L.attn_norm); F(L.ffn_norm); }
  F(e->k_pool); F(e->v_pool); F(e->rope); F(e->d_block_tables);
  F(e->x); if (e->tp == 1) F(e->y); F(e->xb); F(e->tp_stage); F(e->ylast); F(e->qkv); F(e->attn); F(e->h); F(e->logits); F(e->logits_l); F(e->x_last); F(e->attn_ws);
  F(e->d_ids); F(e->d_pos); F(e->d_page_of_tok); F(e->d_tiles); F(e->d_last_rows);
  F(e->S.seq_len); F(e->S.last_token); F(e->S.temperature); F(e->S.top_p); F(e->S.top_k); F(e->S.seed); F(e->S.step);
  F(e->B.slots); F(e->B.ids); F(e->B.seq_lens); F(e->B.temperature); F(e->B.top_p); F(e->B.top_k);
  F(e->B.seed); F(e->B.step); F(e->B.out_ids);
  for (int i = 0; i < llmlb_engine::kRing; ++i) {
    if (e->h_stage[i]) cudaFreeHost(e->h_stage[i]);
    if (e->h_out[i]) cudaFreeHost(e->h_out[i]);
  }
  if (e->tp_ready)
    for (uint32_t r = 0; r < e->tp; ++r)
      if (r != e->rank && e->tpc.base[r]) cudaIpcCloseMemHandle(e->tpc.base[r]);
  F(e->xchg); F(e->part_ws); F(e->sk_ws); F(e->sk_cnt);
  for (auto ev : e->ev_pool) cudaEventDestroy(ev);
  if (e->st) cudaStreamDestroy(e->st);
  delete e;
}

extern "C" int llmlb_engine_model_info(const llmlb_engine* e, llmlb_model_info* out) {
  if (!e || !out) { set_error("null argument"); return LLMLB_E_INVALID_ARG; }
  memset(out, 0, sizeof(*out));
  strncpy(out->id, e->cfg.model_id, sizeof(out->id) - 1);
  out->context_length = e->cfg.max_ctx;
  out->vocab = e->M.vocab;
  out->n_layers = e->M.n_layers;
  out->hidden = e->M.hidden;
  out->param_bytes = e->param_bytes;
  return LLMLB_OK;
}

extern "C" int llmlb_engine_health(const llmlb_engine* ce, llmlb_health* out) {
  llmlb_engine* e = const_cast<llmlb_engine*>(ce);
  if (!e || !out) { set_error("null argument"); return LLMLB_E_INVALID_ARG; }
  memset(out, 0, sizeof(*out));
  size_t fr = 0, tot = 0;
  cudaSetDevice(e->cfg.device);
  cudaMemGetInfo(&fr, &tot);
  out->device_count = e->tp;
  out->total_memory_bytes = tot;
  out->used_memory_bytes = tot - fr;
  std::lock_guard<std::mutex> lk(e->mu);
  out->active_requests = (uint32_t)e->running.size();
  out->queued_requests = (uint32_t)e->waiting.size();
  out->free_kv_pages = (uint32_t)e->free_pages.size();
  out->total_kv_pages = e->n_pages;
  out->steps_prefill = e->steps_prefill; out->steps_decode = e->steps_decode;
  out->tokens_prefill = e->tokens_prefill; out->tokens_decode = e->tokens_decode;
  out->gpu_ms_prefill = e->gpu_ms_prefill; out->gpu_ms_decode = e->gpu_ms_decode;
  out->kernel_launches = g_kernel_launches.load();
  out->preemptions = e->preemptions.load();
  return LLMLB_OK;
}

extern "C" int llmlb_request_submit(llmlb_engine* e, const int32_t* prompt_ids, uint32_t n_prompt,
                                    const llmlb_sampling* s, uint64_t* req_id) {
  if (!e || !prompt_ids || !s || !req_id || n_prompt == 0) { set_error("llmlb_request_submit: bad argument"); return LLMLB_E_INVALID_ARG; }
  if (s->max_tokens == 0) { set_error("max_tokens must be > 0"); return LLMLB_E_INVALID_ARG; }
  if (uint64_t(n_prompt) + s->max_tokens > e->cfg.max_ctx) {
    set_error("prompt + max_tokens exceeds the context length");
    return LLMLB_E_INVALID_ARG;
  }
  if (ceil_div(n_prompt + s->max_tokens, kPageTokens) > e->n_pages) { set_error("request can never fit the KV pool"); return LLMLB_E_INVALID_ARG; }
  for (uint32_t i = 0; i < n_prompt; ++i)
    if (prompt_ids[i] < 0 || uint32_t(prompt_ids[i]) >= e->M.vocab) { set_error("token id out of range"); return LLMLB_E_INVALID_ARG; }
  if (s->temperature < 0.f || s->top_p < 0.f) { set_error("negative temperature/top_p"); return LLMLB_E_INVALID_ARG; }
  auto r = std::make_shared<Request>();
  r->prompt.assign(prompt_ids, prompt_ids + n_prompt);
  r->n_prompt0 = n_prompt;
  r->s = *s;
  if (s->stop_ids && s->n_stop_ids) r->stop_ids.assign(s->stop_ids, s->stop_ids + s->n_stop_ids);
  r->s.stop_ids = nullptr;
  r->t_submit = std::chrono::steady_clock::now();
  {
    std::lock_guard<std::mutex> lk(e->mu);
    if (e->plan_on && !e->plan.leader) { set_error("follower rank of a plan channel: requests enter through rank 0"); return LLMLB_E_UNSUPPORTED; }
    if (!e->fatal_error.empty()) { set_error("engine failed: " + e->fatal_error); return LLMLB_E_DEVICE; }
    if (e->waiting.size() >= (e->cfg.queue_max ? e->cfg.queue_max : 4096u)) { set_error("Request queue is full"); return LLMLB_E_QUEUE_FULL; }
    r->id = e->next_id++;
    e->requests[r->id] = r;
    e->waiting.push_back(r);
    *req_id = r->id;
    if (e->plan_on) {   // id, sampling, prompt and stop ids travel to the followers in queue order
      std::vector<uint8_t> rec(8 + sizeof(llmlb_sampling) + 8 + (size_t(n_prompt) + r->stop_ids.size()) * 4);
      uint8_t* p = rec.data();
      memcpy(p, &r->id, 8); p += 8;
      memcpy(p, &r->s, sizeof(llmlb_sampling)); p += sizeof(llmlb_sampling);
      const uint32_t n_stop = uint32_t(r->stop_ids.size());
      memcpy(p, &n_prompt, 4); memcpy(p + 4, &n_stop, 4); p += 8;
      memcpy(p, r->prompt.data(), size_t(n_prompt) * 4); p += size_t(n_prompt) * 4;
      if (n_stop) memcpy(p, r->stop_ids.data(), size_t(n_stop) * 4);
      e->plan_log(kPlanSubmit, rec.data(), uint32_t(rec.size()));
    }
  }
  e->cv_sched.notify_all();
  return LLMLB_OK;
}

extern "C" int llmlb_request_poll(llmlb_engine* e, uint64_t req_id, llmlb_token_event* out,
                                  uint32_t cap, uint32_t* n_out, int timeout_ms) {
  if (!e || !out || !n_out || cap == 0) { set_error("llmlb_request_poll: bad argument"); return LLMLB_E_INVALID_ARG; }
  *n_out = 0;
  std::unique_lock<std::mutex> lk(e->mu);
  auto it = e->requests.find(req_id);
  if (it == e->requests.end()) { set_error("unknown request id"); return LLMLB_E_NOT_FOUND; }
  ReqPtr r = it->second;
  auto ready = [&] { return !r->events.empty() || r->finished; };
  if (!ready() && timeout_ms != 0) {
    if (timeout_ms < 0) e->cv_events.wait(lk, ready);
    else if (!e->cv_events.wait_for(lk, std::chrono::milliseconds(timeout_ms), ready)) return LLMLB_E_TIMEOUT;
  }
  while (*n_out < cap && !r->events.empty()) {
    out[(*n_out)++] = r->events.front();
    r->events.pop_front();
  }
  return LLMLB_OK;
}

extern "C" int llmlb_request_cancel(llmlb_engine* e, uint64_t req_id) {
  if (!e) { set_error("null engine"); return LLMLB_E_INVALID_ARG; }
  {
    std::lock_guard<std::mutex> lk(e->mu);
    auto it = e->requests.find(req_id);
    if (it == e->requests.end()) { set_error("unknown request id"); return LLMLB_E_NOT_FOUND; }
    it->second->cancel = true;
    e->plan_log(kPlanCancel, &req_id, 8);
  }
  e->cv_sched.notify_all();
  return LLMLB_OK;
}

extern "C" int llmlb_request_release(llmlb_engine* e, uint64_t req_id) {
  if (!e) { set_error("null engine"); return LLMLB_E_INVALID_ARG; }
  std::lock_guard<std::mutex> lk(e->mu);
  auto it = e->requests.find(req_id);
  if (it == e->requests.end()) { set_error("unknown request id"); return LLMLB_E_NOT_FOUND; }
  if (it->second->finished) e->requests.erase(it);
  else { it->second->client_released = true; it->second->cancel = true; e->plan_log(kPlanRelease, &req_id, 8); e->cv_sched.notify_all(); }
  return LLMLB_OK;
}

extern "C" int llmlb_engine_pause(llmlb_engine* e, uint32_t paused) {
  if (!e) { set_error("null engine"); return LLMLB_E_INVALID_ARG; }
  {
    std::lock_guard<std::mutex> lk(e->mu);
    if (e->plan_on && !e->plan.leader) { set_error("follower rank of a plan channel: rank 0 pauses the group"); return LLMLB_E_UNSUPPORTED; }
    e->paused = paused != 0;
    const uint8_t v = paused != 0;
    e->plan_log(kPlanPause, &v, 1);
  }
  e->cv_sched.notify_all();
  return LLMLB_OK;
}

// Run every decode-kernel instantiation once eagerly (sets max-dynamic-smem attributes outside of
// graph capture and surfaces launch errors at create time), then clear the state it touched.
int llmlb_engine::warmup() {
  const uint32_t widths[9] = {1, 2, 3, 4, 5, 17, 33, 65, 129};
  const size_t ms = cfg.max_seqs;
  iota_kernel<<<ceil_div(cfg.max_seqs, 128), 128, 0, st>>>(B.slots, cfg.max_seqs);  // slot b for row b
  LLMLB_LAUNCH_CHECK();
  for (uint32_t w : widths) {
    if (w > cfg.max_seqs) break;
    LLMLB_CUDA_CHECK(cudaMemsetAsync(S.seq_len, 0, ms * 4, st));  // every row: empty cache, position 0
    RC(layer_stack_decode(w));
  }
  cur_batch_slots.clear();
  LLMLB_CUDA_CHECK(cudaMemsetAsync(S.seq_len, 0, ms * 4, st));
  LLMLB_CUDA_CHECK(cudaMemsetAsync(S.last_token, 0, ms * 4, st));
  LLMLB_CUDA_CHECK(cudaMemsetAsync(S.step, 0, ms * 8, st));
  LLMLB_CUDA_CHECK(cudaStreamSynchronize(st));
  return LLMLB_OK;
}

// ------------------------------------------------------------------ TP wiring ---------------
extern "C" int llmlb_engine_tp_export(llmlb_engine* e, uint8_t handle[LLMLB_IPC_HANDLE_BYTES]) {
  if (!e || !handle) { set_error("null argument"); return LLMLB_E_INVALID_ARG; }
  if (e->tp == 1 || !e->xchg) { set_error("engine is not tensor-parallel"); return LLMLB_E_UNSUPPORTED; }
  static_assert(sizeof(cudaIpcMemHandle_t) == LLMLB_IPC_HANDLE_BYTES, "ipc handle size");
  cudaSetDevice(e->cfg.device);
  cudaIpcMemHandle_t hnd;
  LLMLB_CUDA_CHECK(cudaIpcGetMemHandle(&hnd, e->xchg));
  memcpy(handle, &hnd, sizeof(hnd));
  return LLMLB_OK;
}

extern "C" int llmlb_engine_tp_import(llmlb_engine* e, const uint8_t* handles, uint32_t n) {
  if (!e || !handles || n != e->tp) { set_error("llmlb_engine_tp_import: need tp_size handles"); return LLMLB_E_INVALID_ARG; }
  if (e->tp == 1) { set_error("engine is not tensor-parallel"); return LLMLB_E_UNSUPPORTED; }
  cudaSetDevice(e->cfg.device);
  std::lock_guard<std::mutex> sl(e->step_mu);
  for (uint32_t r = 0; r < n; ++r) {
    if (r == e->rank) { e->tpc.base[r] = e->xchg; continue; }
    cudaIpcMemHandle_t hnd;
    memcpy(&hnd, handles + size_t(r) * LLMLB_IPC_HANDLE_BYTES, sizeof(hnd));
    void* p = nullptr;
    LLMLB_CUDA_CHECK(cudaIpcOpenMemHandle(&p, hnd, cudaIpcMemLazyEnablePeerAccess));
    e->tpc.base[r] = (uint8_t*)p;
  }
  e->tp_ready = true;
  return e->warmup();
}

// CPU-only self-test of the plan ring (tests/test_plan_ring_cpu.py runs it in two processes): the
// leader writes `n_records` records of pseudo-random size (more bytes than the ring holds, so wrap
// and back-pressure are exercised), the follower reads them back; both return an FNV-1a checksum
// over (type, length, payload).  No GPU involved.
extern "C" int llmlb_debug_plan_ring(const char* shm_name, uint32_t rank, uint32_t n_records, uint64_t seed, uint64_t* checksum) {
  if (!shm_name || !checksum || rank > 1) { set_error("llmlb_debug_plan_ring: bad argument"); return LLMLB_E_INVALID_ARG; }
  PlanChannel ch;
  int rc = ch.open(shm_name, rank, 2);
  if (rc != LLMLB_OK) return rc;
  uint64_t h = 1469598103934665603ull;
  auto mixb = [&](const void* p, size_t n) { const uint8_t* b = static_cast<const uint8_t*>(p); for (size_t i = 0; i < n; ++i) { h ^= b[i]; h *= 1099511628211ull; } };
  std::atomic<bool> never{false};
  std::vector<uint8_t> buf;
  uint64_t state = seed;
  for (uint32_t i = 0; i < n_records; ++i) {
    if (rank == 0) {
      state = mix64(state);
      const uint32_t len = (i % 7 == 0) ? 0u : uint32_t(state % 65537);
      const uint32_t type = 1 + uint32_t((state >> 20) % 6);
      buf.resize(len);
      for (uint32_t k = 0; k < len; ++k) buf[k] = uint8_t(mix64(state + k) >> 13);
      ch.write(type, buf.data(), len);
      mixb(&type, 4); mixb(&len, 4); mixb(buf.data(), len);
    } else {
      const uint32_t type = ch.read(&buf, never);
      const uint32_t len = uint32_t(buf.size());
      mixb(&type, 4); mixb(&len, 4); mixb(buf.data(), len);
    }
  }
  if (rank == 0) {   // do not unlink the ring under a reader that is still draining it
    for (int tries = 0; tries < 6000 && ch.h->tail[1].load(std::memory_order_acquire) != ch.h->head.load(std::memory_order_acquire); ++tries) usleep(1000);
  }
  ch.close_channel();
  *checksum = h;
  return LLMLB_OK;
}

// Rank 0 first (it creates the shared-memory ring), then the followers.  From then on requests are
// submitted on rank 0 only; follower ranks replay its scheduler log (PlanChannel above).
extern "C" int llmlb_engine_tp_plan_channel(llmlb_engine* e, const char* shm_name) {
  if (!e || !shm_name || !*shm_name) { set_error("llmlb_engine_tp_plan_channel: bad argument"); return LLMLB_E_INVALID_ARG; }
  if (e->tp == 1) return LLMLB_OK;   // nothing to coordinate
  if (!e->tp_ready) { set_error("plan channel: import the peer handles first (llmlb_engine_tp_import)"); return LLMLB_E_UNSUPPORTED; }
  std::lock_guard<std::mutex> lk(e->mu);
  if (e->plan_on) { set_error("plan channel already attached"); return LLMLB_E_INVALID_ARG; }
  if (!e->waiting.empty() || !e->running.empty() || !e->inflight.empty()) { set_error("plan channel: attach before submitting requests"); return LLMLB_E_QUEUE_FULL; }
  int rc = e->plan.open(shm_name, e->rank, e->tp);
  if (rc != LLMLB_OK) return rc;
  e->plan_on = true;
  e->cv_sched.notify_all();
  return LLMLB_OK;
}

extern "C" int llmlb_op_allreduce(llmlb_engine* e, float* buf, uint64_t n, void* stream) {
  if (!e || !buf || n % 4) { set_error("llmlb_op_allreduce: bad argument"); return LLMLB_E_INVALID_ARG; }
  if (e->tp == 1) return LLMLB_OK;
  if (!e->tp_ready) { set_error("tp handles not imported"); return LLMLB_E_UNSUPPORTED; }
  if (n * 4 > e->pull_slot_bytes) { set_error("llmlb_op_allreduce: larger than the exchange slot"); return LLMLB_E_INVALID_ARG; }
  // sum = buf_0 + ... : copy buf into the slot, zero buf, pull-add every rank's slot, then a second
  // (empty) barrier so that nobody overwrites the slot while a peer still reads it
  cudaStream_t st = (cudaStream_t)stream;
  float* part = reinterpret_cast<float*>(e->xchg + e->pull_slot_off);
  LLMLB_CUDA_CHECK(cudaMemcpyAsync(part, buf, n * 4, cudaMemcpyDeviceToDevice, st));
  LLMLB_CUDA_CHECK(cudaMemsetAsync(buf, 0, n * 4, st));
  RC(ar_allreduce_add(e->tpc, e->pull_slot_off, buf, n, st));
  return ar_allreduce_add(e->tpc, e->pull_slot_off, buf, 0, st);
}

// ------------------------------------------------------------------ tensors by HF name ------
int llmlb_engine::resolve_tensor(const std::string& name, __nv_bfloat16** base, uint64_t* rows,
                                 uint64_t* cols, uint64_t* ld, uint64_t* full_rows,
                                 uint64_t* full_cols, uint64_t* row0, uint64_t* col0) {
  const uint64_t H = M.hidden, qr = uint64_t(nq_l) * kHeadDim, kr = uint64_t(nkv_l) * kHeadDim;
  *row0 = 0; *col0 = 0;
  if (name == "model.embed_tokens.weight") { *base = embed; *rows = M.vocab; *cols = H; *ld = H; *full_rows = M.vocab; *full_cols = H; return LLMLB_OK; }
  if (name == "model.norm.weight") { *base = final_norm; *rows = 1; *cols = H; *ld = H; *full_rows = 1; *full_cols = H; return LLMLB_OK; }
  if (name == "lm_head.weight") { *base = lm_head; *rows = vocab_l; *cols = H; *ld = H; *full_rows = M.vocab; *full_cols = H; *row0 = uint64_t(rank) * vocab_l; return LLMLB_OK; }
  unsigned l = 0; char rest[96] = {0};
  if (sscanf(name.c_str(), "model.layers.%u.%95s", &l, rest) == 2 && l < M.n_layers) {
    LayerW& L = layers[l];
    std::string r(rest);
    if (r == "self_attn.q_proj.weight") { *base = L.wqkv; *rows = qr; *cols = H; *ld = H; *full_rows = uint64_t(M.n_heads) * kHeadDim; *full_cols = H; *row0 = rank * qr; return LLMLB_OK; }
    if (r == "self_attn.k_proj.weight") { *base = L.wqkv + qr * H; *rows = kr; *cols = H; *ld = H; *full_rows = uint64_t(M.n_kv_heads) * kHeadDim; *full_cols = H; *row0 = rank * kr; return LLMLB_OK; }
    if (r == "self_attn.v_proj.weight") { *base = L.wqkv + (qr + kr) * H; *rows = kr; *cols = H; *ld = H; *full_rows = uint64_t(M.n_kv_heads) * kHeadDim; *full_cols = H; *row0 = rank * kr; return LLMLB_OK; }
    if (r == "self_attn.o_proj.weight") { *base = L.wo; *rows = H; *cols = qr; *ld = qr; *full_rows = H; *full_cols = uint64_t(M.n_heads) * kHeadDim; *col0 = rank * qr; return LLMLB_OK; }
    if (r == "mlp.gate_proj.weight") { *base = L.wgu; *rows = ffn_l; *cols = H; *ld = 2 * H; *full_rows = M.ffn; *full_cols = H; *row0 = uint64_t(rank) * ffn_l; return LLMLB_OK; }
    if (r == "mlp.up_proj.weight") { *base = L.wgu + H; *rows = ffn_l; *cols = H; *ld = 2 * H; *full_rows = M.ffn; *full_cols = H; *row0 = uint64_t(rank) * ffn_l; return LLMLB_OK; }
    if (r == "mlp.down_proj.weight") { *base = L.wdown; *rows = H; *cols = ffn_l; *ld = ffn_l; *full_rows = H; *full_cols = M.ffn; *col0 = uint64_t(rank) * ffn_l; return LLMLB_OK; }
    if (r == "input_layernorm.weight") { *base = L.attn_norm; *rows = 1; *cols = H; *ld = H; *full_rows = 1; *full_cols = H; return LLMLB_OK; }
    if (r == "post_attention_layernorm.weight") { *base = L.ffn_norm; *rows = 1; *cols = H; *ld = H; *full_rows = 1; *full_cols = H; return LLMLB_OK; }
  }
  set_error("unknown tensor name: " + name);
  return LLMLB_E_NOT_FOUND;
}

extern "C" int llmlb_engine_load_tensor(llmlb_engine* e, const char* name, const void* host,
                                        uint64_t rows, uint64_t cols) {
  if (!e || !name || !host) { set_error("null argument"); return LLMLB_E_INVALID_ARG; }
  __nv_bfloat16* base; uint64_t r, c, ld, fr, fc, r0, c0;
  RC(e->resolve_tensor(name, &base, &r, &c, &ld, &fr, &fc, &r0, &c0));
  if (rows * cols != fr * fc || (fr > 1 && (rows != fr || cols != fc))) {
    set_error(std::string("shape mismatch for ") + name);
    return LLMLB_E_INVALID_ARG;
  }
  cudaSetDevice(e->cfg.device);
  std::lock_guard<std::mutex> sl(e->step_mu);
  LLMLB_CUDA_CHECK(cudaStreamSynchronize(e->st));
  const __nv_bfloat16* src = (const __nv_bfloat16*)host + r0 * fc + c0;
  LLMLB_CUDA_CHECK(cudaMemcpy2D(base, ld * 2, src, fc * 2, c * 2, r, cudaMemcpyHostToDevice));
  return LLMLB_OK;
}

extern "C" int llmlb_engine_read_tensor(llmlb_engine* e, const char* name, void* host,
                                        uint64_t cap_bytes, uint64_t* rows, uint64_t* cols) {
  if (!e || !name || !host || !rows || !cols) { set_error("null argument"); return LLMLB_E_INVALID_ARG; }
  __nv_bfloat16* base; uint64_t r, c, ld, fr, fc, r0, c0;
  RC(e->resolve_tensor(name, &base, &r, &c, &ld, &fr, &fc, &r0, &c0));
  if (r * c * 2 > cap_bytes) { set_error("buffer too small"); return LLMLB_E_INVALID_ARG; }
  cudaSetDevice(e->cfg.device);
  std::lock_guard<std::mutex> sl(e->step_mu);
  LLMLB_CUDA_CHECK(cudaStreamSynchronize(e->st));
  LLMLB_CUDA_CHECK(cudaMemcpy2D(host, c * 2, base, ld * 2, c * 2, r, cudaMemcpyDeviceToHost));
  *rows = r; *cols = c;
  return LLMLB_OK;
}

// ------------------------------------------------------------------ parity hooks ------------
static int debug_acquire(llmlb_engine* e) {  // step_mu held
  std::lock_guard<std::mutex> lk(e->mu);
  if (!e->running.empty() || !e->waiting.empty() || !e->inflight.empty()) {
    set_error("debug hooks need an idle engine");
    return LLMLB_E_QUEUE_FULL;
  }
  if (e->debug_slot < 0) {
    if (e->free_slots.empty() || e->free_pages.size() < e->pages_per_seq) { set_error("no free slot/pages"); return LLMLB_E_QUEUE_FULL; }
    e->debug_slot = e->free_slots.back(); e->free_slots.pop_back();
    for (uint32_t i = 0; i < e->pages_per_seq; ++i) { e->debug_pages.push_back(e->free_pages.back()); e->free_pages.pop_back(); }
  }
  return LLMLB_OK;
}

extern "C" int llmlb_debug_reset(llmlb_engine* e) {
  if (!e) { set_error("null engine"); return LLMLB_E_INVALID_ARG; }
  std::lock_guard<std::mutex> sl(e->step_mu);
  std::lock_guard<std::mutex> lk(e->mu);
  if (e->debug_slot >= 0) {
    e->free_slots.push_back(e->debug_slot);
    for (int32_t p : e->debug_pages) e->free_pages.push_back(p);
    e->debug_pages.clear();
    e->debug_slot = -1;
  }
  e->debug_len = 0;
  return LLMLB_OK;
}

extern "C" int llmlb_debug_prefill_logits(llmlb_engine* e, const int32_t* prompt, uint32_t n,
                                          float* logits_last, float* logits_all) {
  if (!e || !prompt || n == 0 || !logits_last) { set_error("bad argument"); return LLMLB_E_INVALID_ARG; }
  if (n > e->cfg.max_step_tokens || n > e->cfg.max_ctx) { set_error("prompt longer than max_step_tokens/max_ctx"); return LLMLB_E_INVALID_ARG; }
  cudaSetDevice(e->cfg.device);
  std::lock_guard<std::mutex> sl(e->step_mu);
  RC(debug_acquire(e));
  cudaStream_t st = e->st;
  const int slot = e->debug_slot;
  std::vector<int32_t> pos(n), page(n), tiles;
  for (uint32_t i = 0; i < n; ++i) { pos[i] = int32_t(i); page[i] = e->debug_pages[i / kPageTokens]; }
  for (uint32_t j = 0; j < n; j += llmlb_engine::kPfTile) { tiles.push_back(int32_t(j)); tiles.push_back(int32_t(std::min<uint32_t>(llmlb_engine::kPfTile, n - j))); tiles.push_back(int32_t(j)); tiles.push_back(slot); }
  LLMLB_CUDA_CHECK(cudaMemcpy(e->d_block_tables + size_t(slot) * e->pages_per_seq, e->debug_pages.data(), e->debug_pages.size() * 4, cudaMemcpyHostToDevice));
  LLMLB_CUDA_CHECK(cudaMemcpy(e->d_ids, prompt, n * 4, cudaMemcpyHostToDevice));
  LLMLB_CUDA_CHECK(cudaMemcpy(e->d_pos, pos.data(), n * 4, cudaMemcpyHostToDevice));
  LLMLB_CUDA_CHECK(cudaMemcpy(e->d_page_of_tok, page.data(), n * 4, cudaMemcpyHostToDevice));
  LLMLB_CUDA_CHECK(cudaMemcpy(e->d_tiles, tiles.data(), tiles.size() * 4, cudaMemcpyHostToDevice));
  slot_init_kernel<<<1, 1, 0, st>>>(e->S, slot, 0.f, 1.f, 0, 0, 0);
  LLMLB_LAUNCH_CHECK();
  RC(llmlb_op_embed(e->embed, e->d_ids, e->x, n, e->M.hidden, e->M.vocab, st));
  llmlb_engine::FwdState fs;
  RC(e->forward_tokens(n, false, 0, (uint32_t)tiles.size() / 4, &fs));
  if (!fs.y_final) RC(e->finish_small_tp(&fs, n));
  const uint32_t chunk = e->cfg.max_seqs;
  const size_t H = e->M.hidden, V = e->M.vocab;
  for (uint32_t c0 = logits_all ? 0 : n - 1; c0 < n; c0 += chunk) {
    uint32_t R = std::min(chunk, n - c0);
    if (fs.y_final) {   // tensor parallel, protocol B: the rows are already normalised (bf16)
      LLMLB_CUDA_CHECK(cudaMemcpyAsync(e->ylast, e->y + size_t(c0) * H, size_t(R) * H * 2, cudaMemcpyDeviceToDevice, st));
      RC(e->logits_from_y(e->ylast, e->m_ylast, R));
    } else {
      LLMLB_CUDA_CHECK(cudaMemcpyAsync(e->x_last, fs.xres + size_t(c0) * H, size_t(R) * H * 4, cudaMemcpyDeviceToDevice, st));
      RC(e->logits_from_x(e->x_last, R));
    }
    LLMLB_CUDA_CHECK(cudaStreamSynchronize(st));
    if (logits_all) LLMLB_CUDA_CHECK(cudaMemcpy(logits_all + size_t(c0) * V, e->logits, size_t(R) * V * 4, cudaMemcpyDeviceToHost));
    if (c0 + R == n) LLMLB_CUDA_CHECK(cudaMemcpy(logits_last, e->logits + size_t(R - 1) * V, V * 4, cudaMemcpyDeviceToHost));
  }
  int32_t len = int32_t(n);
  LLMLB_CUDA_CHECK(cudaMemcpy(e->S.seq_len + slot, &len, 4, cudaMemcpyHostToDevice));
  e->debug_len = n;
  e->cur_batch_slots.clear();
  return LLMLB_OK;
}

extern "C" int llmlb_debug_decode_logits(llmlb_engine* e, int32_t token, float* logits_out) {
  if (!e || !logits_out || token < 0 || uint32_t(token) >= e->M.vocab) { set_error("bad argument"); return LLMLB_E_INVALID_ARG; }
  cudaSetDevice(e->cfg.device);
  std::lock_guard<std::mutex> sl(e->step_mu);
  if (e->debug_slot < 0 || e->debug_len == 0) { set_error("call llmlb_debug_prefill_logits first"); return LLMLB_E_INVALID_ARG; }
  if (e->debug_len + 1 > e->cfg.max_ctx) { set_error("context full"); return LLMLB_E_INVALID_ARG; }
  cudaStream_t st = e->st;
  int32_t slot = e->debug_slot;
  LLMLB_CUDA_CHECK(cudaMemcpy(e->S.last_token + slot, &token, 4, cudaMemcpyHostToDevice));
  LLMLB_CUDA_CHECK(cudaMemcpy(e->B.slots, &slot, 4, cudaMemcpyHostToDevice));
  e->cur_batch_slots.clear();
  decode_prepare_kernel<<<1, 128, 0, st>>>(e->S, e->B, 1);
  LLMLB_LAUNCH_CHECK();
  RC(llmlb_op_embed(e->embed, e->B.ids, e->x, 1, e->M.hidden, e->M.vocab, st));
  llmlb_engine::FwdState fs;
  RC(e->forward_tokens(1, true, 1, 0, &fs));
  RC(e->logits_after_forward(&fs, 1, true));
  LLMLB_CUDA_CHECK(cudaStreamSynchronize(st));
  LLMLB_CUDA_CHECK(cudaMemcpy(logits_out, e->logits, size_t(e->M.vocab) * 4, cudaMemcpyDeviceToHost));
  e->debug_len += 1;
  return LLMLB_OK;
}

// ------------------------------------------------------------------ in-kernel timeline ------
// Debug-only (not in the public header): records per-CTA globaltimer stamps of the decode GEMV and
// attention kernels.  enable(cap) allocates, dump() copies records (6 x u64 each) and resets.
static TraceBuf g_tb{};
extern "C" int llmlb_debug_trace_enable(uint32_t cap) {
  if (g_tb.data) { cudaFree(g_tb.data); cudaFree(g_tb.count); g_tb = TraceBuf{}; }
  if (cap) {
    LLMLB_CUDA_CHECK(cudaMalloc((void**)&g_tb.data, size_t(cap) * 48));
    LLMLB_CUDA_CHECK(cudaMalloc((void**)&g_tb.count, 4));
    LLMLB_CUDA_CHECK(cudaMemset(g_tb.count, 0, 4));
    g_tb.cap = cap;
  }
  ks_set_trace(g_tb);
  attn_set_trace(g_tb);
  tc_set_trace(g_tb);
  tp_set_trace(g_tb);
  tc2_set_trace(g_tb);
  return LLMLB_OK;
}
extern "C" int llmlb_debug_trace_dump(unsigned long long* out, uint32_t cap_records, uint32_t* n) {
  if (!g_tb.data) { *n = 0; return LLMLB_OK; }
  LLMLB_CUDA_CHECK(cudaDeviceSynchronize());
  uint32_t cnt = 0;
  LLMLB_CUDA_CHECK(cudaMemcpy(&cnt, g_tb.count, 4, cudaMemcpyDeviceToHost));
  if (cnt > g_tb.cap) cnt = g_tb.cap;
  if (cnt > cap_records) cnt = cap_records;
  LLMLB_CUDA_CHECK(cudaMemcpy(out, g_tb.data, size_t(cnt) * 48, cudaMemcpyDeviceToHost));
  LLMLB_CUDA_CHECK(cudaMemset(g_tb.count, 0, 4));
  *n = cnt;
  return LLMLB_OK;
}
