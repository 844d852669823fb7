/*
 * llmlb_b200.h — C ABI of the B200-native in-process inference backend for llmlb.
 *
 * This is the drop-in boundary (SURVEY.md §8b).  In the reference, model work is
 * reached through one HTTP call: `reqwest POST {base_url}/v1/...` at
 *   llmlb/src/api/openai.rs:995-1005   (chat/completions builder + send)
 *   llmlb/src/api/proxy.rs:372-401     (forward_to_endpoint, used by responses.rs:257)
 * and the endpoint is probed through
 *   llmlb/src/health/endpoint_checker.rs:515-577  (GET /api/health, GET /v1/models)
 *   llmlb/src/metadata/xllm.rs:48-61              (GET /api/models/{model}/info)
 * The functions below are what an FFI crate in the gateway binds instead of that
 * HTTP client: plain pointers and sizes, no C++/torch types, caller-owned buffers.
 *
 * Error convention: 0 = OK, <0 = LLMLB_E_*; text via llmlb_last_error() (thread local).
 * Mapping to the gateway's LbError → HTTP status (llmlb/src/api/error.rs:31-110):
 *   E_INVALID_ARG→400  E_MODEL_NOT_FOUND→404  E_QUEUE_FULL→503/429  E_TIMEOUT→504
 *   E_DEVICE/E_INTERNAL→502
 *
 * Threading: every export is thread-safe; submit / poll(timeout_ms=0) / cancel never block
 * on the GPU (callers are tokio workers, llmlb/src/main.rs:64,131).
 */
#ifndef LLMLB_B200_H
#define LLMLB_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LLMLB_ABI_VERSION 1

enum {
  LLMLB_OK = 0,
  LLMLB_E_INVALID_ARG = -1,
  LLMLB_E_MODEL_NOT_FOUND = -2,
  LLMLB_E_QUEUE_FULL = -3,
  LLMLB_E_TIMEOUT = -4,
  LLMLB_E_DEVICE = -5,
  LLMLB_E_INTERNAL = -6,
  LLMLB_E_NOT_FOUND = -7,   /* unknown request id / tensor name */
  LLMLB_E_UNSUPPORTED = -8
};

/* ---------------------------------------------------------------- engine ---- */

typedef struct llmlb_engine llmlb_engine; /* opaque; one per GPU rank */

/* Llama-family decoder geometry (Llama-3-8B: 4096/32/32/8/128/14336/128256, theta 5e5, eps 1e-5). */
typedef struct llmlb_model_config {
  uint32_t hidden;       /* model width */
  uint32_t n_layers;
  uint32_t n_heads;      /* query heads */
  uint32_t n_kv_heads;   /* GQA key/value heads */
  uint32_t head_dim;     /* must be 128 */
  uint32_t ffn;          /* SwiGLU inner width */
  uint32_t vocab;
  float rope_theta;
  float rms_eps;
} llmlb_model_config;

typedef struct llmlb_engine_config {
  uint32_t abi_version;      /* LLMLB_ABI_VERSION */
  llmlb_model_config model;
  char model_id[128];        /* id reported to /v1/models (sync/parser.rs:78-110) */
  int32_t device;            /* CUDA ordinal of this rank */
  uint32_t tp_rank;          /* tensor-parallel rank of this process */
  uint32_t tp_size;          /* 1, 2, 4 or 8 (must divide n_kv_heads) */
  uint32_t max_seqs;         /* concurrent sequences (continuous batch width) */
  uint32_t max_ctx;          /* tokens per sequence (prompt + generated) */
  uint32_t kv_block_tokens;  /* tokens per KV page; must be 64 */
  uint32_t kv_pages;         /* pages in the pool; 0 = size from max_seqs*max_ctx */
  uint32_t max_step_tokens;  /* prefill tokens packed into one step (0 = 2048) */
  uint64_t synthetic_seed;   /* weights are generated on-device from this seed (see
                                llmlb_engine_load_tensor to overwrite with real ones) */
  uint32_t use_cuda_graphs;  /* capture decode steps per batch width */
  uint32_t gemm_impl;        /* must be 0 (tcgen05/TMEM/TMA tiles); anything else: LLMLB_E_INVALID_ARG */
  uint32_t lookahead;        /* decode steps in flight before the host reads tokens (0 = 2) */
  /* Back-pressure, mirroring the gateway's own queue (llmlb/src/config.rs:80-99, QueueConfig) and its
   * per-request inference timeout (llmlb/src/types/endpoint.rs:389).  0 = no limit. */
  uint32_t queue_max;          /* waiting requests beyond this: submit returns LLMLB_E_QUEUE_FULL (gateway: 429) */
  uint32_t queue_timeout_ms;   /* a request still waiting for admission after this finishes QUEUE_TIMEOUT (504) */
  uint32_t request_timeout_ms; /* a request not finished this long after submit finishes DEADLINE (504 timeout) */
  uint32_t attn_impl;          /* must be 0 (prefill attention on tcgen05 + TMEM + TMA); anything else: LLMLB_E_INVALID_ARG */
  uint32_t tp_proto;           /* must be 0 (tensor-parallel decode exchange of {value, epoch} pairs); anything else:
                                  LLMLB_E_INVALID_ARG */
  uint32_t reserved[3];
} llmlb_engine_config;

int llmlb_engine_create(const llmlb_engine_config* cfg, llmlb_engine** out);
/* Stops the scheduler, drops whatever is still queued or running and frees the device.  The ONE call that is not safe
 * against the others: no call on `e` may be in progress (a thread blocked in llmlb_request_poll included) or start once
 * this one has begun.  A gateway drains first (inference_gate.rs: reject new work, wait for in-flight bodies, then abort
 * the rest with llmlb_request_cancel) and destroys the engine last. */
void llmlb_engine_destroy(llmlb_engine* e);

/* Tensor-parallel wiring (one process per GPU).  Each rank exports a CUDA IPC handle of its
 * exchange buffer; the host gathers all handles (any out-of-band channel, e.g.
 * torch.distributed.all_gather) and hands the table back.  After import the engine's
 * projections finish with a peer-memory all-reduce over NVLink.  */
#define LLMLB_IPC_HANDLE_BYTES 64
int llmlb_engine_tp_export(llmlb_engine* e, uint8_t handle[LLMLB_IPC_HANDLE_BYTES]);
int llmlb_engine_tp_import(llmlb_engine* e, const uint8_t* handles /* tp_size*64 */, uint32_t n);
/* Serving with tp_size > 1: rank 0 owns the request queue; it logs every scheduler-state change
 * (submit, cancel, release, pause, scheduling iteration, harvest) to a POSIX shared-memory ring
 * `shm_name` and the follower ranks replay the log, so all ranks launch identical steps.  Call
 * after llmlb_engine_tp_import and before any submit, on rank 0 FIRST (it creates the ring), then
 * on the followers.  Afterwards submit/poll/cancel/pause only on rank 0 (followers return
 * LLMLB_E_UNSUPPORTED).  No-op for tp_size == 1. */
int llmlb_engine_tp_plan_channel(llmlb_engine* e, const char* shm_name);

/* Replace a synthetic tensor with real weights (host pointer, row-major bf16, the FULL
 * un-sharded tensor: the engine takes this rank's slice).  Names follow the HF Llama
 * checkpoint: "model.embed_tokens.weight", "model.layers.N.self_attn.q_proj.weight", ... */
int llmlb_engine_load_tensor(llmlb_engine* e, const char* name, const void* host_bf16,
                             uint64_t rows, uint64_t cols);
/* Copy this rank's slice of a tensor back to the host as bf16 (debug / CPU-baseline feed).
 * name as above; returns rows/cols of the slice. cap_bytes guards the buffer. */
int llmlb_engine_read_tensor(llmlb_engine* e, const char* name, void* host_bf16,
                             uint64_t cap_bytes, uint64_t* rows, uint64_t* cols);

typedef struct llmlb_model_info {  /* feeds GET /v1/models and /api/models/{m}/info */
  char id[128];
  uint32_t context_length;
  uint32_t vocab;
  uint32_t n_layers;
  uint32_t hidden;
  uint64_t param_bytes;            /* bf16 bytes of matmul weights held by this rank */
} llmlb_model_info;
int llmlb_engine_model_info(const llmlb_engine* e, llmlb_model_info* out);

typedef struct llmlb_health {      /* feeds GET /api/health (endpoint_checker.rs:515-557) */
  uint32_t device_count;
  uint64_t total_memory_bytes;
  uint64_t used_memory_bytes;
  uint32_t active_requests;
  uint32_t queued_requests;
  uint32_t free_kv_pages;
  uint32_t total_kv_pages;
  uint64_t steps_prefill;
  uint64_t steps_decode;
  uint64_t tokens_prefill;
  uint64_t tokens_decode;
  double gpu_ms_prefill;           /* CUDA-event time spent in prefill steps */
  double gpu_ms_decode;            /* CUDA-event time spent in decode steps */
  uint64_t kernel_launches;        /* launches of this library's kernels so far */
  uint64_t preemptions;            /* sequences evicted (pages reclaimed, recomputed later) so far */
} llmlb_health;
int llmlb_engine_health(const llmlb_engine* e, llmlb_health* out);

/* --------------------------------------------------------------- requests --- */

typedef struct llmlb_sampling {
  uint32_t max_tokens;             /* generated-token budget (max_tokens / max_output_tokens) */
  float temperature;               /* 0 = greedy arg-max */
  uint32_t top_k;                  /* 0 = off */
  float top_p;                     /* >=1 or 0 = off */
  uint64_t seed;                   /* per-request RNG stream */
  const int32_t* stop_ids;         /* optional stop / EOS token ids */
  uint32_t n_stop_ids;
  uint32_t ignore_eos;             /* benchmark mode: generate exactly max_tokens */
} llmlb_sampling;

enum { LLMLB_FINISH_NONE = 0, LLMLB_FINISH_STOP = 1, LLMLB_FINISH_LENGTH = 2,
       LLMLB_FINISH_CANCELLED = 3, LLMLB_FINISH_ERROR = 4,
       LLMLB_FINISH_QUEUE_TIMEOUT = 5,   /* never admitted within queue_timeout_ms ("Queue wait timeout", openai.rs:862-882) */
       LLMLB_FINISH_DEADLINE = 6 };      /* request_timeout_ms passed (classify_upstream_request_error: 504 "timeout") */

typedef struct llmlb_token_event {
  int32_t token_id;
  uint32_t index;                  /* 0-based index among generated tokens */
  uint32_t finish_reason;          /* LLMLB_FINISH_*; non-zero on the last event */
  uint32_t prompt_tokens;          /* usage, valid on every event */
  uint32_t completion_tokens;
  double t_ms;                     /* host ms since submit when the token became visible */
} llmlb_token_event;

/* Non-blocking enqueue; prompt_ids are copied.  */
int llmlb_request_submit(llmlb_engine* e, const int32_t* prompt_ids, uint32_t n_prompt,
                         const llmlb_sampling* s, uint64_t* req_id);
/* Drain up to cap events. timeout_ms: 0 = return at once, <0 = wait until at least one. */
int llmlb_request_poll(llmlb_engine* e, uint64_t req_id, llmlb_token_event* out, uint32_t cap,
                       uint32_t* n_out, int timeout_ms);
/* Client disconnect / drain abort (inference_gate.rs:73-76). */
int llmlb_request_cancel(llmlb_engine* e, uint64_t req_id);
/* Forget a finished request (frees its event queue). */
int llmlb_request_release(llmlb_engine* e, uint64_t req_id);
/* Hold (1) / resume (0) the scheduler: queued requests are not admitted while paused.  Used to
 * line up identical queues on all tensor-parallel ranks before the first step. */
int llmlb_engine_pause(llmlb_engine* e, uint32_t paused);

/* Debug/parity hooks: run the prompt as ONE prefill and return fp32 logits of every position
 * (n_prompt x vocab, this rank's vocab slice gathered on rank 0 only when tp_size==1), and
 * teacher-forced single-token decode steps for per-step logit parity against the oracle. */
int llmlb_debug_prefill_logits(llmlb_engine* e, const int32_t* prompt_ids, uint32_t n_prompt,
                               float* logits_last /* vocab */, float* logits_all /* or NULL */);
int llmlb_debug_decode_logits(llmlb_engine* e, int32_t token_id, float* logits /* vocab */);
int llmlb_debug_reset(llmlb_engine* e);

const char* llmlb_last_error(void);
uint32_t llmlb_abi_version(void);

/* ------------------------------------------------ kernel-level entry points --
 * Device-pointer API used by the parity tests and the roofline micro-benchmarks
 * (one per SURVEY.md §8(a2) row).  `stream` is a cudaStream_t cast to void*.
 * All matrices row-major; W is [n_out, k] bf16 (HF layout).                     */

/* a2.1  x[t,:] = E[ids[t],:]  (bf16 table -> fp32 residual stream) */
int llmlb_op_embed(const void* table_bf16, const int32_t* ids, float* x_f32, uint32_t n_tokens,
                   uint32_t hidden, uint32_t vocab, void* stream);
/* a2.2  y = x * rsqrt(mean(x^2)+eps) * g   (fp32 in, bf16 out) */
int llmlb_op_rmsnorm(const float* x_f32, const void* gain_bf16, void* y_bf16, uint32_t n_tokens,
                     uint32_t hidden, float eps, void* stream);

/* Epilogues shared by the decode GEMV and the tensor-core GEMM. */
enum { LLMLB_EPI_STORE_BF16 = 0,   /* out_bf16[t,n]  = acc                         */
       LLMLB_EPI_RESID_F32 = 1,    /* out_f32[t,n]  += acc   (residual add)        */
       LLMLB_EPI_SILU_MUL = 2,     /* out_bf16[t,n/2] = silu(acc[2i])*acc[2i+1]    */
       LLMLB_EPI_STORE_F32 = 3 };  /* out_f32[t,n]   = acc   (logits)              */

/* a2.3/8/9/10/11 decode path: HBM-bound GEMV for 1..4 tokens.  If gain!=NULL the input is the
 * fp32 residual stream and RMSNorm is fused into the prologue; else x is bf16. */
int llmlb_op_gemv(const void* w_bf16, const void* x, const void* gain_bf16, float eps, void* out,
                  uint32_t n_tokens, uint32_t n_out, uint32_t k, uint32_t epilogue,
                  uint32_t out_stride, void* stream);
/* prefill / batched path: out[t,n] = sum_k x[t,k]*W[n,k] on tensor cores (tcgen05 + TMEM + TMA tiles).
 * impl must be 0: the round-1 mma.sync (1) and stream-K (2) variants left the library (tools/experiments/) and return
 * LLMLB_E_UNSUPPORTED.  x is bf16 [n_tokens,k]; k a multiple of 8; SILU_MUL needs an even n_out (interleaved gate/up rows). */
int llmlb_op_gemm(const void* w_bf16, const void* x_bf16, void* out, uint32_t n_tokens,
                  uint32_t n_out, uint32_t k, uint32_t epilogue, uint32_t out_stride,
                  uint32_t impl, void* stream);

/* RoPE table: fp32 (cos, sin) pairs [max_pos][64] for head_dim 128, HF rotate-half pairing. */
int llmlb_op_rope_table(float* table, uint32_t max_pos, float theta, void* stream);
/* KV pages: K and V pools are [page][kv_head][64 tokens][128] bf16.
 * a2.4+a2.5 prefill: rotate q,k in place inside qkv [t, (nq+2nkv)*128] and append k,v to pages.
 * page_of_token[t] = page holding positions[t] (negative = do not append). */
int llmlb_op_rope_append(void* qkv_bf16, const int32_t* positions, const int32_t* page_of_token,
                         const float* rope_table, void* k_pages, void* v_pages, uint32_t n_tokens,
                         uint32_t n_heads, uint32_t n_kv_heads, void* stream);
/* a2.6 causal GQA prefill attention over paged K/V on the 5th-generation tensor cores (tcgen05.mma, S and
 * PV in TMEM, Q/K/V staged by TMA; V is consumed MN-major straight from its [token][d] pages).
 * tiles: int32[n_tiles][4] = {first q row in qkv, q rows in tile (<=128), position of first row, row into
 * block_tables}; k_pages / v_pages are ONE layer's pool [n_pages][n_kv][64][128]; n_tokens = rows of qkv. */
int llmlb_op_prefill_attention_tc(const void* qkv_bf16, uint32_t n_tokens, const void* k_pages,
                                  const void* v_pages, uint32_t n_pages, const int32_t* block_tables,
                                  uint32_t bt_stride, const int32_t* tiles, uint32_t n_tiles,
                                  void* out_bf16, uint32_t n_heads, uint32_t n_kv_heads, void* stream);
/* a2.4+a2.5+a2.7 decode: per sequence rotate the new q,k, append k,v, attend over the pages.
 * seq_lens[b] = tokens INCLUDING the new one; bt_rows[b] = block-table row of sequence b (NULL =
 * identity).  workspace: llmlb_op_decode_attention_ws(ws_seqs, n_heads, n_splits) bytes, zeroed
 * once by the caller (the kernel leaves its tickets zeroed). */
size_t llmlb_op_decode_attention_ws(uint32_t ws_seqs, uint32_t n_heads, uint32_t max_splits);
int llmlb_op_decode_attention(const void* qkv_bf16, void* k_pages, void* v_pages,
                              const int32_t* block_tables, uint32_t bt_stride,
                              const int32_t* bt_rows, const int32_t* seq_lens, uint32_t n_seqs,
                              void* out_bf16, uint32_t n_heads, uint32_t n_kv_heads,
                              const float* rope_table, uint32_t n_splits, uint32_t ws_seqs,
                              void* workspace, void* stream);
/* a2.12 sampling: arg-max when temperature==0 else temperature/top-k/top-p with a counter RNG.
 * params: per-row {temperature, top_p} floats, {top_k} ints, {seed, step} u64. */
int llmlb_op_sample(const float* logits, uint32_t n_rows, uint32_t vocab, const float* temperature,
                    const float* top_p, const int32_t* top_k, const uint64_t* seed,
                    const uint64_t* step, int32_t* out_ids, void* stream);
/* a2.13 all-reduce(sum) of fp32 [n] across tp ranks through peer-mapped buffers. */
int llmlb_op_allreduce(llmlb_engine* e, float* buf_f32, uint64_t n, void* stream);

/* synthetic weights: fills a [rows, cols] bf16 slice whose global origin is (row0, col0) in a
 * tensor with `ld` columns; value depends only on (seed, tensor_id, global index). */
int llmlb_op_synth_bf16(void* out_bf16, uint64_t rows, uint64_t cols, uint64_t row0,
                        uint64_t col0, uint64_t ld, uint64_t seed, uint32_t tensor_id, float std,
                        void* stream);

#ifdef __cplusplus
}
#endif
#endif /* LLMLB_B200_H */
