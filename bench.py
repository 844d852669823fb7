#!/usr/bin/env python
"""bench.py — decode tok/s + prefill tok/s for Llama-3-8B bf16, 512-in/128-out (BASELINE.json).

`python bench.py --gpus N --steps K --warmup W` prints ONE JSON line on rank 0.  One "step" = one
whole request through the engine: a 512-token prompt is prefilled and 128 tokens are decoded
greedily (EOS disabled) — BASELINE.json configs[1].  K steps are timed, after W untimed ones.

`--dump-outputs DIR` writes, after the timed steps, what the last timed step returned to its caller:
one [batch, 128] float64 array per token-event field, DIR/<field>.npy (token_id, index,
finish_reason, prompt_tokens, completion_tokens; the wall-clock t_ms is left out).  Prompts and
weights are seeded, so two builds run with the same arguments can be compared array for array.

  value        decode tok/s from CUDA-event time of the decode steps (inputs resident in HBM)
  prefill      prefill tok/s from CUDA-event time of the prefill steps (+ tensor roofline)
  e2e          the WHOLE request as a client sees it through the C ABI with HOST buffers
               (llmlb_request_submit(host prompt ids) ... last llmlb_request_poll event): prompt H2D,
               prefill and all token D2H inside; tok/s = generated tokens / that time — the
               reference's own TPS formula (llmlb/src/api/benchmarks.rs:467-474)
  roofline     HBM roofline of the decode step (GEMV-dominated) and of the dominant GEMV kernel
  parity       BEFORE anything is timed: N=1 — the engine's greedy tokens teacher-forced through the
               CPU oracle at full 8B geometry; N>1 — the sharded engine's 128 tokens teacher-forced
               through a tp=1 engine of the same weights on rank 0's GPU.  Rule: every token must be
               within `tol` of the checker's arg-max logit (near-ties may resolve differently).
  streams      BASELINE.json configs[2] (N=1: 64 concurrent streams) / configs[3] (N=8: 128 streams):
               decode tok/s, step roofline, TTFT p50/p95, whole-job tok/s seen by the client
  reference_shape   the reference benchmark's workload (20 requests, concurrency 4, temperature 0.2;
               llmlb/src/api/benchmarks.rs:25-34) through submit/poll, per-request TPS mean/p50/p95
  cpu_baseline the oracle (CPU restatement) timed on the host cores on a bounded sample

N > 1 (torchrun, one rank per GPU): the model is sharded tensor-parallel over the N ranks (our own
push kernels over NVLink peer memory, see llmlb_b200/csrc/tp_common.cuh; torch.distributed/NCCL
carries the 64-byte IPC handles, the barriers and the max-over-ranks of the timings) and the SAME
workload is timed ("scaling": "strong").

`--impl reference` times the reference path's CPU stand-in: the oracle port of the model on the
host cores (the reference repository proxies to an external CPU llama.cpp/Ollama server that is
not in the tree and cannot be installed here — SURVEY.md §8c/8d).
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True     # the benchmark writes nothing into the tree it runs from (which may be read-only)

PROMPT, GEN = 512, 128
PARITY_TOL_CPU = 0.30    # margin to the fp32 CPU oracle's arg-max logit (logit std ~1.3 at 8B; bf16 activations): the near-tie bound of
                         # tests/test_parity_8b_gpu.py (measured there: max|dlogit| 0.20; measured here: margins 0.05-0.22)
PARITY_TOL_TP = 0.10     # margin to the tp=1 engine's arg-max logit (same kernels, other summation order)


def algorithmic_bytes_per_decode_step(m, batch, ctx, tp=1):
    """SURVEY.md §8d: all matmul weights + lm_head once per step, plus the KV of every sequence."""
    H, L, F, V = m["hidden"], m["n_layers"], m["ffn"], m["vocab"]
    nq, nkv, hd = m["n_heads"], m["n_kv_heads"], m["head_dim"]
    per_layer = H * (nq + 2 * nkv) * hd + nq * hd * H + 3 * H * F
    w = (per_layer * L + V * H) * 2
    kv = 2 * L * nkv * hd * 2 * ctx * batch
    return (w + kv) / tp


def prefill_flops(m, n):
    H, L, F, V = m["hidden"], m["n_layers"], m["ffn"], m["vocab"]
    nq, nkv, hd = m["n_heads"], m["n_kv_heads"], m["head_dim"]
    per_layer = H * (nq + 2 * nkv) * hd + nq * hd * H + 3 * H * F
    attn = L * 4 * n * n * nq * hd / 2
    return 2.0 * per_layer * L * n + 2.0 * V * H + attn


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("hbm_gbs", 6650.0), d.get("bf16_tflops", 1590.0), d.get("bf16_tflops_sustained", 1400.0), "measured"
    return 6650.0, 1590.0, 1400.0, "fallback"


def pct(xs, q):
    xs = sorted(xs)
    if not xs:
        return None
    return xs[min(len(xs) - 1, int(round(q * (len(xs) - 1))))]


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region (recipe: B200_PROFILING.md)."""

    def __init__(self, index=0):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm = sorted(int(float(r[0])) for r in self.rows if r and r[0].replace(".", "").isdigit())
        mx = [int(float(r[1])) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 3 + i and r[3 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(self.rows)}


def make_prompt(i, vocab, n=PROMPT):
    import numpy as np
    return np.random.RandomState(1000 + i).randint(0, vocab, n).astype("int32").tolist()


DUMP_FIELDS = ("token_id", "index", "finish_reason", "prompt_tokens", "completion_tokens")


def dump_outputs(out_dir, requests):
    """requests: per request, the token events the engine returned -> out_dir/<field>.npy, float64 [requests, events]."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for f in DUMP_FIELDS:
        np.save(os.path.join(out_dir, f + ".npy"), np.array([[e[f] for e in evs] for evs in requests], dtype=np.float64))


# ------------------------------------------------------------------------------ CPU arms ----
def cpu_reference_run(model, steps, warmup, sample_prompt=32, sample_gen=4, forced=None, weights="bf16", sd_bits=None):
    """Oracle port on the host cores: synthetic bf16 weights (C generator), C/OpenMP matmuls.
    Bounded sample of the 512/128 workload: `sample_prompt` prompt tokens + `sample_gen` decoded
    tokens per step, full 8B geometry (nothing skipped).
    forced = (prompt ids, generated ids) of the GPU engine: the first step feeds THOSE tokens instead
    of the oracle's own arg-max (same work, same timing) and records, per token, how far the engine's
    choice is from the oracle's arg-max logit -> the parity record of the N=1 line."""
    import numpy as np
    import torch
    from oracle import synth_native
    from oracle.llama_ref import LlamaRef
    os.environ.setdefault("OMP_WAIT_POLICY", "passive")
    cores = synth_native.effective_cpus()
    torch.set_num_threads(cores)
    synth_native.set_threads(cores)
    t0 = time.time()
    # weights="q4_0": every matmul weight as ggml Q4_0 blocks (4.5 bits/weight) — the weight width of the reference path's own
    # CPU configuration (BASELINE.json configs[0]: llama.cpp, Llama-3-8B q4); same model, same sample, same formula
    if sd_bits is None:
        sd_bits = synth_native.synth_state_dict_bits(model, seed=0)     # pass it in to share the 16 GB between the two legs
    sd = synth_native.q4_from_bits(sd_bits) if weights == "q4_0" else sd_bits
    ref = LlamaRef(model, sd)
    t_load = time.time() - t0
    # probe one lm_head-sized GEMV and shrink the sample if this host is slow, so the run stays
    # inside its time box (~30 s of CPU work per step) whatever the core quota is
    if weights == "q4_0":
        pw = sd["lm_head.weight"]
        px = np.zeros((1, pw.k), dtype=np.float32)
        synth_native.linear_q4_0(pw.blocks, pw.k, px)
        tp0 = time.time(); synth_native.linear_q4_0(pw.blocks, pw.k, px); probe = time.time() - tp0
        est_token_s = probe * (algorithmic_bytes_per_decode_step(model, 0, 0) / (pw.blocks.shape[0] * pw.k * 2.0))
    else:
        probe_w = sd["lm_head.weight"].bits
        px = np.zeros((1, probe_w.shape[1]), dtype=np.float32)
        synth_native.linear_bf16(probe_w, px)
        tp0 = time.time(); synth_native.linear_bf16(probe_w, px); probe = time.time() - tp0
        est_token_s = probe * (algorithmic_bytes_per_decode_step(model, 0, 0) / (probe_w.size * 2.0))
    if forced is None and est_token_s * (sample_prompt / 4.0 + sample_gen) > 30.0:
        sample_gen = max(1, min(sample_gen, int(10.0 / max(est_token_s, 1e-3))))
        sample_prompt = max(4, min(sample_prompt, int(4 * 15.0 / max(est_token_s, 1e-3))))
    dec_tok = dec_s = pre_tok = pre_s = 0.0
    parity = None
    for it in range(warmup + steps):
        use_forced = forced is not None and it == 0
        prompt = forced[0] if use_forced else make_prompt(it, model["vocab"], sample_prompt)
        n_gen = len(forced[1]) - 1 if use_forced else sample_gen
        ref.reset()
        a = time.time()
        lg = ref.forward(prompt)[-1]
        b = time.time()
        margins, agree = [], 0
        tok = forced[1][0] if use_forced else int(torch.argmax(lg))
        if use_forced:
            margins.append(float(lg.max() - lg[tok])); agree += int(int(torch.argmax(lg)) == tok)
        for j in range(n_gen):
            lg = ref.forward([tok])[-1]
            tok = forced[1][j + 1] if use_forced else int(torch.argmax(lg))
            if use_forced:
                margins.append(float(lg.max() - lg[tok])); agree += int(int(torch.argmax(lg)) == tok)
        c = time.time()
        if use_forced:
            parity = {"checker": "CPU oracle (oracle/llama_ref.py + llama_cpu.c), full 8B geometry, fp32 activations",
                      "prompt_tokens": len(prompt), "tokens_checked": len(margins), "top1_agree": agree,
                      "max_margin": max(margins), "tol": PARITY_TOL_CPU, "logit_std": float(lg.std()),
                      "ok": bool(max(margins) <= PARITY_TOL_CPU)}
        if it >= warmup:
            pre_tok += len(prompt); pre_s += b - a
            dec_tok += n_gen; dec_s += c - b
    return {"decode_tok_s": dec_tok / dec_s, "prefill_tok_s": pre_tok / pre_s, "cores": cores,
            "weights_s": t_load, "ms_per_step": 1e3 * (pre_s + dec_s) / max(1, steps), "parity": parity,
            "sample": "%d prompt + %d decoded tokens per step, full Llama-3-8B geometry, %s (oracle/llama_cpu.c), %d threads"
                      % (sample_prompt, sample_gen, "ggml Q4_0 weights (4.5 bits/weight) x Q8_0 activations, integer block dot products (AVX2), C/OpenMP" if weights == "q4_0"
                         else "bf16 weights, C/OpenMP fp32-accumulate linears", cores)}


def run_reference(args):
    from llmlb_b200.ffi import LLAMA3_8B, LLAMA_TINY
    model = LLAMA_TINY if args.model == "tiny" else LLAMA3_8B
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    r = cpu_reference_run(model, args.steps, args.warmup, args.cpu_prompt, args.cpu_gen)
    line = {"impl": "reference", "metric": "decode_tok_s", "value": r["decode_tok_s"], "unit": "tok/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": workload_config(args, model, 1),
            "prefill": {"value": r["prefill_tok_s"], "unit": "tok/s"},
            "cpu_baseline": {"value": r["decode_tok_s"], "unit": "tok/s", "cores": r["cores"], "kind": "port",
                             "sample": r["sample"]},
            "e2e": {"value": r["decode_tok_s"], "unit": "tok/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


def workload_config(args, model, tp):
    return {"workload": "Llama-3-8B bf16, batch=1, %d-in/%d-out greedy decode (BASELINE.json configs[1])" % (PROMPT, GEN)
            if args.model == "8b" else "tiny-geometry debug run (NOT the benchmark config)",
            "model_geometry": model, "prompt_tokens": PROMPT, "generated_tokens": GEN, "batch": args.batch,
            "parallelism": "tp%d" % tp, "weights": "synthetic seed 0, N(0,0.02^2) via integer hash",
            "l2": "inputs larger than L2: 15 GB of weights are streamed per decode step (126 MB L2)"}


# ------------------------------------------------------------------------------ GPU arm -----
def gemv_microbench(model, hbm_peak):
    """Dominant decode kernel (gate/up GEMV, fused RMSNorm + SiLU*mul): CUDA events on the launch
    stream, rotating over > L2 worth of distinct weight copies."""
    import torch
    from llmlb_b200 import ffi
    L = ffi.lib()
    H, F = model["hidden"], model["ffn"]
    n_out = 2 * F
    copies = max(2, int(400e6 // (n_out * H * 2)) + 1)
    w = [torch.empty(n_out, H, dtype=torch.bfloat16, device="cuda").normal_(0, 0.02) for _ in range(copies)]
    x = torch.randn(1, H, device="cuda")
    g = torch.ones(H, dtype=torch.bfloat16, device="cuda")
    out = torch.empty(1, F, dtype=torch.bfloat16, device="cuda")
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    vp = lambda t: C.c_void_p(t.data_ptr())

    def run(i):
        ffi.check(L.llmlb_op_gemv(vp(w[i % copies]), vp(x), vp(g), 1e-5, vp(out), 1, n_out, H, ffi.EPI_SILU_MUL, F, st))
    for i in range(6):
        run(i)
    torch.cuda.synchronize()
    iters = 40
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for i in range(iters):
        run(i)
    b.record()
    torch.cuda.synchronize()
    us = a.elapsed_time(b) * 1e3 / iters
    bytes_ = n_out * H * 2
    traffic = 244.44e6 if (n_out, H) == (28672, 4096) else None
    return {"kernel": "gemv_ks_kernel<1,SILU_MUL,NORM,1> %dx%d (gate/up, fused RMSNorm + SiLU*up)" % (n_out, H),
            "bytes_per_launch": bytes_, "us_per_launch": us, "achieved": bytes_ / us / 1e3, "unit": "GB/s",
            "frac": bytes_ / us / 1e3 / hbm_peak, "traffic": traffic,
            "traffic_source": "not measured in this run: dram__bytes_read.sum + dram__bytes_write.sum of one launch in the committed ncu --set full capture profiles/r1_final_gemv_ks_ncu_full.txt (241.20 + 3.24 MB)"}


def run_ours(args):
    import numpy as np
    import torch
    from llmlb_b200 import build, ffi
    build.build()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    tp = world
    dist = None
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    model = ffi.LLAMA_TINY if args.model == "tiny" else ffi.LLAMA3_8B
    hbm_peak, tf_burst, tf_sust, peak_src = measured_peaks()
    n_streams = args.streams if args.streams >= 0 else (128 if world >= 8 else 64)
    max_seqs = max(4, args.batch, n_streams)
    eng = ffi.Engine(model, model_id="llama-3-8b-synthetic", device=local, tp_rank=rank, tp_size=tp,
                     max_seqs=max_seqs, max_ctx=1024, seed=0, use_cuda_graphs=not args.no_graphs, tp_proto=args.tp_proto)
    if world > 1:
        handles = [None] * world
        dist.all_gather_object(handles, eng.tp_export())
        eng.tp_import(handles)
        dist.barrier()

    def barrier():
        if world > 1:
            dist.barrier()

    def run_requests(prompts, n_new, **kw):
        """Submit all prompts at once (identical queues on every rank when tp > 1), drain them.
        Returns (per-request token events, per-request host wall ms from submit to last event)."""
        if world > 1:
            eng.pause(True)
        t_sub = time.perf_counter()
        rids = [eng.submit(p, n_new, ignore_eos=True, **kw) for p in prompts]
        if world > 1:
            dist.barrier()
            eng.pause(False)
        evs = {r: [] for r in rids}
        pending = set(rids)
        while pending:
            for r in list(pending):
                got = eng.poll(r, cap=256, timeout_ms=-1 if len(pending) == 1 else 2)
                evs[r].extend(got)
                if got and got[-1]["finish_reason"]:
                    pending.discard(r)
        wall_ms = (time.perf_counter() - t_sub) * 1e3
        for r in rids:
            eng.release(r)
        return [[e for e in evs[r] if e["token_id"] >= 0] for r in rids], wall_ms

    # ---------------- parity, before anything is timed ----------------
    parity = None
    forced_for_cpu = None
    if not args.no_parity:
        if world == 1:
            # the engine's own greedy tokens for the CPU leg's prompt; the oracle is run later (it is the
            # cpu_baseline leg) with these tokens teacher-forced
            pp = make_prompt(0, model["vocab"], args.cpu_prompt)
            toks, _ = run_requests([pp], args.cpu_gen + 1)
            forced_for_cpu = (pp, [t["token_id"] for t in toks[0]])
        else:
            pp = make_prompt(0, model["vocab"])
            toks, _ = run_requests([pp], GEN)
            got = [t["token_id"] for t in toks[0]]
            allt = [None] * world
            dist.all_gather_object(allt, got)
            if rank == 0:
                with ffi.Engine(model, device=local, max_seqs=4, max_ctx=1024, seed=0) as one:
                    lg = one.debug_prefill_logits(pp)
                    margins, agree = [], 0
                    for i, t in enumerate(got):
                        margins.append(float(lg.max() - lg[t])); agree += int(int(np.argmax(lg)) == t)
                        if i + 1 < len(got):
                            lg = one.debug_decode_logits(t)
                parity = {"checker": "tp=1 engine of the same weights on rank 0's GPU, teacher-forced with the tp=%d tokens" % world,
                          "prompt_tokens": PROMPT, "tokens_checked": len(margins), "top1_agree": agree,
                          "max_margin": max(margins), "tol": PARITY_TOL_TP,
                          "ranks_identical": all(a == got for a in allt),
                          "ok": bool(max(margins) <= PARITY_TOL_TP and all(a == got for a in allt) and len(got) == GEN)}
            barrier()
    if args.parity_only:
        if rank == 0:
            print(json.dumps({"parity_only": True, "n_gpus": world, "max_seqs": max_seqs, "parity": parity}))
            sys.stdout.flush()
        eng.close()
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return

    # ---------------- main leg: batch-1 requests ----------------
    for i in range(args.warmup):
        run_requests([make_prompt((10_000 + i) * args.batch + j, model["vocab"]) for j in range(args.batch)], GEN)
    torch.cuda.synchronize()
    barrier()
    h0 = eng.health()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    t0 = time.perf_counter()
    first_to_last_ms, n_dec_tokens, req_tps, req_ms = 0.0, 0, [], []
    toks = []
    for i in range(args.steps):
        toks, _ = run_requests([make_prompt(i * args.batch + j, model["vocab"]) for j in range(args.batch)], GEN)
        lo, hi = [], []
        for tk in toks:
            assert len(tk) == GEN, "request produced %d tokens" % len(tk)
            lo.append(tk[0]["t_ms"]); hi.append(tk[-1]["t_ms"])
            n_dec_tokens += len(tk) - 1
            req_tps.append(len(tk) / (tk[-1]["t_ms"] / 1e3))
            req_ms.append(tk[-1]["t_ms"])
        first_to_last_ms += max(hi) - min(lo)
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, toks)
    h1 = eng.health()
    d = lambda k: h1[k] - h0[k]
    vals = torch.tensor([d("gpu_ms_decode"), d("gpu_ms_prefill"), wall * 1e3, first_to_last_ms, sum(req_ms)],
                        dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(vals, op=dist.ReduceOp.MAX)
    gpu_ms_dec, gpu_ms_pre, wall_ms, ftl_ms, req_ms_sum = [float(v) for v in vals]
    dec_tokens, pre_tokens, dec_steps = d("tokens_decode"), d("tokens_prefill"), d("steps_decode")
    main_launches = d("kernel_launches")
    decode_tok_s = dec_tokens / (gpu_ms_dec / 1e3)
    prefill_tok_s = pre_tokens / (gpu_ms_pre / 1e3)

    # ---------------- streams leg: BASELINE configs[2] / [3] ----------------
    streams = None
    if n_streams > 1:
        def stream_prompts(i):
            return [make_prompt(500_000 + i * n_streams + j, model["vocab"]) for j in range(n_streams)]
        run_requests(stream_prompts(0), GEN)          # warm-up (captures the decode graph of this width)
        torch.cuda.synchronize()
        barrier()
        s0 = eng.health()
        ttft, walls, tot = [], [], 0
        for i in range(args.stream_steps):
            toks, wall_i = run_requests(stream_prompts(1 + i), GEN)
            for tk in toks:
                assert len(tk) == GEN
                ttft.append(tk[0]["t_ms"]); tot += len(tk)
            walls.append(wall_i)
        torch.cuda.synchronize()
        s1 = eng.health()
        ds = lambda k: s1[k] - s0[k]
        sv = torch.tensor([ds("gpu_ms_decode"), ds("gpu_ms_prefill"), sum(walls)], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(sv, op=dist.ReduceOp.MAX)
        s_dec_ms, s_pre_ms, s_wall_ms = [float(v) for v in sv]
        step_s = s_dec_ms / 1e3 / max(1, ds("steps_decode"))
        bytes_step = algorithmic_bytes_per_decode_step(model, n_streams, PROMPT + GEN / 2, tp)
        streams = {"workload": "BASELINE.json configs[%d]: %d concurrent streams submitted at t=0, %d-in/%d-out, continuous batching through submit/poll, tp%d"
                               % (3 if world >= 8 else 2, n_streams, PROMPT, GEN, tp),
                   "n_streams": n_streams, "steps": args.stream_steps,
                   "decode_tok_s": ds("tokens_decode") / (s_dec_ms / 1e3), "decode_ms_per_step": step_s * 1e3,
                   "prefill_tok_s": ds("tokens_prefill") / (s_pre_ms / 1e3),
                   "roofline": {"bound": "hbm", "achieved": bytes_step / step_s / 1e9, "peak": hbm_peak, "unit": "GB/s",
                                "frac": bytes_step / step_s / 1e9 / hbm_peak, "peak_source": peak_src,
                                "what": "%.2f GB algorithmic per decode step per GPU (weights + %d x %d-token KV)" % (bytes_step / 1e9, n_streams, int(PROMPT + GEN / 2))},
                   "ttft_ms_p50": pct(ttft, 0.5), "ttft_ms_p95": pct(ttft, 0.95),
                   "e2e_tok_s": tot / (s_wall_ms / 1e3),
                   "gpu_launches": int(ds("kernel_launches"))}

    # ---------------- the reference benchmark's own workload shape (single engine, N = 1) ----------------
    ref_shape = None
    if world == 1 and not args.no_ref_shape:
        n_req, conc = 20, 4
        rs0 = eng.health()
        t_start = time.perf_counter()
        inflight, done_tps, next_i = {}, [], 0
        while next_i < n_req or inflight:
            while next_i < n_req and len(inflight) < conc:
                rid = eng.submit(make_prompt(700_000 + next_i, model["vocab"]), GEN, temperature=0.2, seed=next_i, ignore_eos=True)
                inflight[rid] = []
                next_i += 1
            for rid in list(inflight):
                got = eng.poll(rid, cap=256, timeout_ms=2)
                inflight[rid].extend(got)
                if got and got[-1]["finish_reason"]:
                    tk = [e for e in inflight.pop(rid) if e["token_id"] >= 0]
                    eng.release(rid)
                    done_tps.append(len(tk) / (tk[-1]["t_ms"] / 1e3))   # output_tokens / (send -> last byte)
        wall_rs = time.perf_counter() - t_start
        rs1 = eng.health()
        ref_shape = {"workload": "20 requests, concurrency 4, temperature 0.2, %d-in/%d-out (llmlb/src/api/benchmarks.rs:25-34); TPS = output_tokens / (submit -> last event), :467-474" % (PROMPT, GEN),
                     "tps_mean": sum(done_tps) / len(done_tps), "tps_p50": pct(done_tps, 0.5), "tps_p95": pct(done_tps, 0.95),
                     "aggregate_tok_s": n_req * GEN / wall_rs, "gpu_launches": int(rs1["kernel_launches"] - rs0["kernel_launches"])}

    if rank == 0:
        ctx = PROMPT + GEN / 2
        bytes_step = algorithmic_bytes_per_decode_step(model, args.batch, ctx, tp)
        step_s = gpu_ms_dec / 1e3 / max(1, dec_steps)
        achieved = bytes_step / step_s / 1e9
        kern = gemv_microbench(model, hbm_peak) if (world == 1 and not args.no_micro) else None
        fl = prefill_flops(model, PROMPT) * (pre_tokens / PROMPT) / tp
        pre_tf = fl / (gpu_ms_pre / 1e3) / 1e12
        whole_req_tps = (args.steps * args.batch * GEN) / (req_ms_sum / 1e3)   # = mean per-request TPS at batch 1
        line = {
            "metric": "decode_tok_s", "value": decode_tok_s, "unit": "tok/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": wall_ms / args.steps,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "bf16",
            "data": "synthetic", "config": workload_config(args, model, tp),
            "prefill": {"value": prefill_tok_s, "unit": "tok/s",
                        "roofline": {"bound": "tensor", "achieved": pre_tf, "peak": tf_burst, "unit": "TFLOP/s",
                                     "frac": pre_tf / tf_burst, "peak_source": peak_src + " (burst cuBLAS bf16)"}},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak,
                         "traffic": (32 * (50.39e6 + 33.60e6 + 244.44e6 + 120.83e6) + 1050.7e6) if (args.model == "8b" and tp == 1 and args.batch == 1) else None,
                         "traffic_source": "not measured in this run: sum over the step's projections of dram__bytes_read+write from the committed ncu --set full captures under profiles/ (lm_head: algorithmic)",
                         "peak_source": peak_src,
                         "what": "whole decode step (%.2f GB algorithmic per step per GPU / %.3f ms CUDA-event step time)" % (bytes_step / 1e9, step_s * 1e3),
                         "kernel": kern},
            "e2e": {"value": whole_req_tps, "unit": "tok/s", "h2d_bytes_per_step": PROMPT * 4 * args.batch,
                    "d2h_bytes_per_step": GEN * 4 * args.batch,
                    "what": "whole request through llmlb_request_submit/poll with host buffers: generated tokens / (submit -> last token event); prompt H2D, prefill and token D2H inside",
                    "decode_only_tok_s": n_dec_tokens / (ftl_ms / 1e3)},
            "gpu_launches": int(main_launches), "clocks": clocks, "parity": parity,
            "streams": streams, "reference_shape": ref_shape,
        }
        if args.cpu_baseline and world == 1:
            eng.close()
            from oracle import synth_native as _sn
            _sn.set_threads(_sn.effective_cpus())
            sd_bits = _sn.synth_state_dict_bits(model, seed=0)
            r = cpu_reference_run(model, 1, 0, args.cpu_prompt, args.cpu_gen, forced=forced_for_cpu, sd_bits=sd_bits)
            line["cpu_baseline"] = {"value": r["decode_tok_s"], "unit": "tok/s", "cores": r["cores"], "kind": "port",
                                    "sample": r["sample"], "prefill_tok_s": r["prefill_tok_s"]}
            if r["parity"]:
                line["parity"] = r["parity"]
            if not args.no_cpu_q4:
                # context, not the reference arm: the same port at the weight width BASELINE.json configs[0] quotes the reference
                # path on (llama.cpp, Llama-3-8B q4): ggml Q4_0 weights, activations quantised to Q8_0, integer block dot products
                # (llama.cpp's CPU scheme restated in oracle/llama_cpu.c, quantisers pinned bit for bit to the gguf package).
                # The bf16 figure above stays the like-for-like baseline of the bf16 engine.
                # In a child process with a time box: whatever happens there (an instruction the host lacks, memory, a hang), the
                # line of this run is printed.
                try:
                    del r, sd_bits
                    cp = subprocess.run([sys.executable, os.path.abspath(__file__), "--cpu-q4-child", "--model", args.model,
                                         "--cpu-prompt", str(args.cpu_prompt), "--cpu-gen", str(args.cpu_gen)],
                                        capture_output=True, text=True, timeout=240)
                    rows = [l for l in cp.stdout.splitlines() if l.startswith("{")]
                    line["cpu_baseline"]["q4_0"] = json.loads(rows[-1]) if rows else {"unavailable": "child exited %d: %s" % (cp.returncode, cp.stderr.strip()[-200:])}
                except Exception as ex:
                    line["cpu_baseline"]["q4_0"] = {"unavailable": "%s: %s" % (type(ex).__name__, ex)}
        line["parity_ok"] = None if line["parity"] is None else line["parity"]["ok"]
        print(json.dumps(line))
        sys.stdout.flush()
    eng.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the token events of the last timed step as DIR/<field>.npy")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--model", default="8b", choices=["8b", "tiny"])
    ap.add_argument("--batch", type=int, default=1, help="concurrent streams per step of the main leg (1 = BASELINE configs[1])")
    ap.add_argument("--streams", type=int, default=-1, help="streams leg width (-1: 64, or 128 at 8 GPUs; 0: skip)")
    ap.add_argument("--stream-steps", type=int, default=2)
    ap.add_argument("--no-graphs", action="store_true")
    ap.add_argument("--tp-proto", type=int, default=0, help="tensor-parallel decode exchange: 0 = value+epoch pairs, 1 = flags")
    ap.add_argument("--no-micro", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--parity-only", action="store_true", help="diagnostic: print the tp parity record and stop")
    ap.add_argument("--no-ref-shape", action="store_true")
    ap.add_argument("--no-cpu-baseline", dest="cpu_baseline", action="store_false")
    ap.add_argument("--no-cpu-q4", action="store_true", help="skip the Q4_0-weights context figure of the CPU baseline (about 20 s)")
    ap.add_argument("--cpu-prompt", type=int, default=32)
    ap.add_argument("--cpu-gen", type=int, default=8)
    ap.add_argument("--cpu-q4-child", action="store_true", help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.cpu_q4_child:     # the Q4_0 x Q8_0 leg of the CPU baseline, run by run_ours in its own process
        from llmlb_b200.ffi import LLAMA3_8B, LLAMA_TINY
        rq = cpu_reference_run(LLAMA_TINY if args.model == "tiny" else LLAMA3_8B, 1, 0, args.cpu_prompt, args.cpu_gen, weights="q4_0")
        print(json.dumps({"value": rq["decode_tok_s"], "unit": "tok/s", "prefill_tok_s": rq["prefill_tok_s"], "cores": rq["cores"],
                          "kind": "port", "sample": rq["sample"]}))
        return
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs needs --impl ours")
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
