"""ctypes binding of include/llmlb_b200.h (the same stub a cgo / Rust-FFI caller would write).

There is no CPU fallback: loading fails loudly when the shared library has not been built, and
engine creation fails when no CUDA device is visible.
"""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libllmlb_b200.so")

OK = 0
E_INVALID_ARG, E_MODEL_NOT_FOUND, E_QUEUE_FULL, E_TIMEOUT = -1, -2, -3, -4
E_DEVICE, E_INTERNAL, E_NOT_FOUND, E_UNSUPPORTED = -5, -6, -7, -8
EPI_STORE_BF16, EPI_RESID_F32, EPI_SILU_MUL, EPI_STORE_F32 = 0, 1, 2, 3
FINISH_NONE, FINISH_STOP, FINISH_LENGTH, FINISH_CANCELLED, FINISH_ERROR, FINISH_QUEUE_TIMEOUT, FINISH_DEADLINE = 0, 1, 2, 3, 4, 5, 6
ABI_VERSION = 1


class ModelConfig(C.Structure):
    _fields_ = [("hidden", C.c_uint32), ("n_layers", C.c_uint32), ("n_heads", C.c_uint32),
                ("n_kv_heads", C.c_uint32), ("head_dim", C.c_uint32), ("ffn", C.c_uint32),
                ("vocab", C.c_uint32), ("rope_theta", C.c_float), ("rms_eps", C.c_float)]


class EngineConfig(C.Structure):
    _fields_ = [("abi_version", C.c_uint32), ("model", ModelConfig), ("model_id", C.c_char * 128),
                ("device", C.c_int32), ("tp_rank", C.c_uint32), ("tp_size", C.c_uint32),
                ("max_seqs", C.c_uint32), ("max_ctx", C.c_uint32), ("kv_block_tokens", C.c_uint32),
                ("kv_pages", C.c_uint32), ("max_step_tokens", C.c_uint32),
                ("synthetic_seed", C.c_uint64), ("use_cuda_graphs", C.c_uint32),
                ("gemm_impl", C.c_uint32), ("lookahead", C.c_uint32), ("queue_max", C.c_uint32),
                ("queue_timeout_ms", C.c_uint32), ("request_timeout_ms", C.c_uint32), ("attn_impl", C.c_uint32),
                ("tp_proto", C.c_uint32), ("reserved", C.c_uint32 * 3)]


class ModelInfo(C.Structure):
    _fields_ = [("id", C.c_char * 128), ("context_length", C.c_uint32), ("vocab", C.c_uint32),
                ("n_layers", C.c_uint32), ("hidden", C.c_uint32), ("param_bytes", C.c_uint64)]


class Health(C.Structure):
    _fields_ = [("device_count", C.c_uint32), ("total_memory_bytes", C.c_uint64),
                ("used_memory_bytes", C.c_uint64), ("active_requests", C.c_uint32),
                ("queued_requests", C.c_uint32), ("free_kv_pages", C.c_uint32),
                ("total_kv_pages", C.c_uint32), ("steps_prefill", C.c_uint64),
                ("steps_decode", C.c_uint64), ("tokens_prefill", C.c_uint64),
                ("tokens_decode", C.c_uint64), ("gpu_ms_prefill", C.c_double),
                ("gpu_ms_decode", C.c_double), ("kernel_launches", C.c_uint64), ("preemptions", C.c_uint64)]


class Sampling(C.Structure):
    _fields_ = [("max_tokens", C.c_uint32), ("temperature", C.c_float), ("top_k", C.c_uint32),
                ("top_p", C.c_float), ("seed", C.c_uint64), ("stop_ids", C.POINTER(C.c_int32)),
                ("n_stop_ids", C.c_uint32), ("ignore_eos", C.c_uint32)]


class TokenEvent(C.Structure):
    _fields_ = [("token_id", C.c_int32), ("index", C.c_uint32), ("finish_reason", C.c_uint32),
                ("prompt_tokens", C.c_uint32), ("completion_tokens", C.c_uint32),
                ("t_ms", C.c_double)]


u32, u64, i32, f32, vp, cp = C.c_uint32, C.c_uint64, C.c_int32, C.c_float, C.c_void_p, C.c_char_p
_P = C.POINTER

# name -> (restype, argtypes); mirrors every prototype in include/llmlb_b200.h
PROTOTYPES = {
    "llmlb_engine_create": (C.c_int, [_P(EngineConfig), _P(vp)]),
    "llmlb_engine_destroy": (None, [vp]),
    "llmlb_engine_tp_export": (C.c_int, [vp, _P(C.c_uint8)]),
    "llmlb_engine_tp_import": (C.c_int, [vp, _P(C.c_uint8), u32]),
    "llmlb_engine_tp_plan_channel": (C.c_int, [vp, cp]),
    "llmlb_engine_load_tensor": (C.c_int, [vp, cp, vp, u64, u64]),
    "llmlb_engine_read_tensor": (C.c_int, [vp, cp, vp, u64, _P(u64), _P(u64)]),
    "llmlb_engine_model_info": (C.c_int, [vp, _P(ModelInfo)]),
    "llmlb_engine_health": (C.c_int, [vp, _P(Health)]),
    "llmlb_engine_pause": (C.c_int, [vp, u32]),
    "llmlb_request_submit": (C.c_int, [vp, _P(i32), u32, _P(Sampling), _P(u64)]),
    "llmlb_request_poll": (C.c_int, [vp, u64, _P(TokenEvent), u32, _P(u32), C.c_int]),
    "llmlb_request_cancel": (C.c_int, [vp, u64]),
    "llmlb_request_release": (C.c_int, [vp, u64]),
    "llmlb_debug_prefill_logits": (C.c_int, [vp, _P(i32), u32, _P(f32), _P(f32)]),
    "llmlb_debug_decode_logits": (C.c_int, [vp, i32, _P(f32)]),
    "llmlb_debug_reset": (C.c_int, [vp]),
    "llmlb_last_error": (cp, []),
    "llmlb_abi_version": (u32, []),
    "llmlb_op_embed": (C.c_int, [vp, vp, vp, u32, u32, u32, vp]),
    "llmlb_op_rmsnorm": (C.c_int, [vp, vp, vp, u32, u32, f32, vp]),
    "llmlb_op_gemv": (C.c_int, [vp, vp, vp, f32, vp, u32, u32, u32, u32, u32, vp]),
    "llmlb_op_gemm": (C.c_int, [vp, vp, vp, u32, u32, u32, u32, u32, u32, vp]),
    "llmlb_op_rope_table": (C.c_int, [vp, u32, f32, vp]),
    "llmlb_op_rope_append": (C.c_int, [vp, vp, vp, vp, vp, vp, u32, u32, u32, vp]),
    "llmlb_op_prefill_attention_tc": (C.c_int, [vp, u32, vp, vp, u32, vp, u32, vp, u32, vp, u32, u32, vp]),
    "llmlb_op_decode_attention_ws": (C.c_size_t, [u32, u32, u32]),
    "llmlb_op_decode_attention": (C.c_int, [vp, vp, vp, vp, u32, vp, vp, u32, vp, u32, u32, vp,
                                            u32, u32, vp, vp]),
    "llmlb_op_sample": (C.c_int, [vp, u32, u32, vp, vp, vp, vp, vp, vp, vp]),
    "llmlb_op_allreduce": (C.c_int, [vp, vp, u64, vp]),
    "llmlb_op_synth_bf16": (C.c_int, [vp, u64, u64, u64, u64, u64, u64, u32, f32, vp]),
}

_lib = None


class LlmlbError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("llmlb_b200 error %d: %s" % (code, msg))
        self.code = code


def lib():
    """Loads libllmlb_b200.so (built by llmlb_b200/build.py). Raises if it is missing."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise FileNotFoundError(
                LIB_PATH + " is missing: run `python -m llmlb_b200.build` (nvcc, sm_100a). "
                "There is no CPU implementation of this path.")
        L = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
        for name, (res, args) in PROTOTYPES.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def last_error():
    return (lib().llmlb_last_error() or b"").decode("utf-8", "replace")


def check(rc):
    if rc != OK:
        raise LlmlbError(rc, last_error())
    return rc


LLAMA3_8B = dict(hidden=4096, n_layers=32, n_heads=32, n_kv_heads=8, head_dim=128, ffn=14336,
                 vocab=128256, rope_theta=500000.0, rms_eps=1e-5)
LLAMA3_70B = dict(hidden=8192, n_layers=80, n_heads=64, n_kv_heads=8, head_dim=128, ffn=28672,
                  vocab=128256, rope_theta=500000.0, rms_eps=1e-5)
# small geometry used by the parity tests (same code paths, oracle finishes in seconds)
LLAMA_TINY = dict(hidden=512, n_layers=2, n_heads=8, n_kv_heads=2, head_dim=128, ffn=1024,
                  vocab=2048, rope_theta=500000.0, rms_eps=1e-5)


# mid geometry whose projections fit the persistent decode chain kernel (K multiple of 2048, 7
# chunks per warp on the down projection like Llama-3-8B) while the oracle still runs in seconds
LLAMA_MID = dict(hidden=2048, n_layers=2, n_heads=16, n_kv_heads=4, head_dim=128, ffn=14336,
                 vocab=4096, rope_theta=500000.0, rms_eps=1e-5)


class Engine:
    """Thin owner of an llmlb_engine*; methods map 1:1 onto the C ABI."""

    def __init__(self, model, model_id="llama-3-8b-synthetic", device=0, tp_rank=0, tp_size=1,
                 max_seqs=8, max_ctx=1024, kv_pages=0, max_step_tokens=0, seed=0,
                 use_cuda_graphs=True, lookahead=0, queue_max=0, queue_timeout_ms=0, request_timeout_ms=0, tp_proto=0):
        cfg = EngineConfig()
        cfg.abi_version = ABI_VERSION
        for k, v in model.items():
            setattr(cfg.model, k, v)
        cfg.model_id = model_id.encode()
        cfg.device, cfg.tp_rank, cfg.tp_size = device, tp_rank, tp_size
        cfg.max_seqs, cfg.max_ctx, cfg.kv_block_tokens = max_seqs, max_ctx, 64
        cfg.kv_pages, cfg.max_step_tokens = kv_pages, max_step_tokens
        cfg.synthetic_seed = seed
        cfg.use_cuda_graphs = 1 if use_cuda_graphs else 0
        cfg.lookahead = lookahead
        cfg.queue_max, cfg.queue_timeout_ms, cfg.request_timeout_ms = queue_max, queue_timeout_ms, request_timeout_ms
        cfg.tp_proto = tp_proto   # must be 0: the library refuses any other value at create
        self.model = dict(model)
        self.cfg = cfg
        self._h = vp()
        check(lib().llmlb_engine_create(C.byref(cfg), C.byref(self._h)))

    def close(self):
        if self._h:
            lib().llmlb_engine_destroy(self._h)
            self._h = vp()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    # ---- requests ----
    def submit(self, prompt_ids, max_tokens, temperature=0.0, top_k=0, top_p=1.0, seed=0,
               stop_ids=(), ignore_eos=False):
        n = len(prompt_ids)
        arr = (i32 * n)(*prompt_ids)
        s = Sampling()
        s.max_tokens, s.temperature, s.top_k, s.top_p, s.seed = max_tokens, temperature, top_k, top_p, seed
        stops = (i32 * max(1, len(stop_ids)))(*stop_ids)
        s.stop_ids = C.cast(stops, _P(i32)) if stop_ids else None
        s.n_stop_ids = len(stop_ids)
        s.ignore_eos = 1 if ignore_eos else 0
        rid = u64()
        check(lib().llmlb_request_submit(self._h, arr, n, C.byref(s), C.byref(rid)))
        return rid.value

    def poll(self, rid, cap=256, timeout_ms=0):
        buf = (TokenEvent * cap)()
        n = u32()
        rc = lib().llmlb_request_poll(self._h, rid, buf, cap, C.byref(n), timeout_ms)
        if rc == E_TIMEOUT:
            return []
        check(rc)
        return [dict(token_id=e.token_id, index=e.index, finish_reason=e.finish_reason,
                     prompt_tokens=e.prompt_tokens, completion_tokens=e.completion_tokens,
                     t_ms=e.t_ms) for e in buf[:n.value]]

    def generate(self, prompt_ids, max_tokens, **kw):
        """submit + drain; returns (token ids, events)."""
        rid = self.submit(prompt_ids, max_tokens, **kw)
        toks, evs = [], []
        while True:
            got = self.poll(rid, timeout_ms=-1)
            evs.extend(got)
            for e in got:
                if e["token_id"] >= 0:
                    toks.append(e["token_id"])
            if got and got[-1]["finish_reason"] != FINISH_NONE:
                break
        self.release(rid)
        return toks, evs

    def cancel(self, rid):
        check(lib().llmlb_request_cancel(self._h, rid))

    def release(self, rid):
        check(lib().llmlb_request_release(self._h, rid))

    def pause(self, paused=True):
        check(lib().llmlb_engine_pause(self._h, 1 if paused else 0))

    def health(self):
        h = Health()
        check(lib().llmlb_engine_health(self._h, C.byref(h)))
        return {k: getattr(h, k) for k, _ in Health._fields_}

    def model_info(self):
        m = ModelInfo()
        check(lib().llmlb_engine_model_info(self._h, C.byref(m)))
        d = {k: getattr(m, k) for k, _ in ModelInfo._fields_}
        d["id"] = d["id"].decode()
        return d

    # ---- tensors (numpy uint16 views of bf16) ----
    def read_tensor(self, name, max_elems):
        import numpy as np
        buf = np.empty(max_elems, dtype=np.uint16)
        r, c = u64(), u64()
        check(lib().llmlb_engine_read_tensor(self._h, name.encode(), buf.ctypes.data, buf.nbytes,
                                             C.byref(r), C.byref(c)))
        return buf[: r.value * c.value].reshape(r.value, c.value)

    def load_tensor(self, name, arr_u16):
        import numpy as np
        a = np.ascontiguousarray(arr_u16, dtype=np.uint16)
        rows, cols = (a.shape if a.ndim == 2 else (1, a.shape[0]))
        check(lib().llmlb_engine_load_tensor(self._h, name.encode(), a.ctypes.data, rows, cols))

    # ---- parity hooks ----
    def debug_prefill_logits(self, prompt_ids, all_positions=False):
        import numpy as np
        n, v = len(prompt_ids), self.model["vocab"]
        arr = (i32 * n)(*prompt_ids)
        last = np.empty(v, dtype=np.float32)
        full = np.empty((n, v), dtype=np.float32) if all_positions else None
        check(lib().llmlb_debug_prefill_logits(
            self._h, arr, n, last.ctypes.data_as(_P(f32)),
            full.ctypes.data_as(_P(f32)) if all_positions else None))
        return (last, full) if all_positions else last

    def debug_decode_logits(self, token):
        import numpy as np
        out = np.empty(self.model["vocab"], dtype=np.float32)
        check(lib().llmlb_debug_decode_logits(self._h, int(token), out.ctypes.data_as(_P(f32))))
        return out

    def debug_reset(self):
        check(lib().llmlb_debug_reset(self._h))

    # ---- tensor parallel ----
    def tp_export(self):
        buf = (C.c_uint8 * 64)()
        check(lib().llmlb_engine_tp_export(self._h, buf))
        return bytes(buf)

    def tp_import(self, handles):
        blob = b"".join(handles)
        arr = (C.c_uint8 * len(blob)).from_buffer_copy(blob)
        check(lib().llmlb_engine_tp_import(self._h, arr, len(handles)))

    def tp_plan_channel(self, name):
        """Rank 0 first (creates the shared-memory log), then the followers; afterwards only rank 0
        submits and the other ranks replay its scheduler."""
        check(lib().llmlb_engine_tp_plan_channel(self._h, name.encode()))
