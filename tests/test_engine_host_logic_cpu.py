"""The engine's HOST side — request queue, iteration-level scheduler, page allocator, preemption, timeouts, event
delivery, the locking of the C ABI — on a machine without a GPU: the UNMODIFIED product library runs over
tests/support/fake_cudart.cpp, a test double of libcudart in which memory is host memory and launches do nothing.
No arithmetic happens (every token id is 0), so nothing here says anything about kernels or parity; what is checked is
counts, ordering, resource accounting and thread safety, at a step rate no GPU reaches.  The same scenarios run under
ThreadSanitizer / AddressSanitizer builds of the library in the long pass recorded in DESIGN.md.

Mechanics: the outer test starts pytest on this file in a child process with LD_PRELOAD = the fake runtime (it must not
be loaded into a process that imports torch); the scenario tests skip themselves unless they run in that child."""
import os
import subprocess
import sys
import threading
import time

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
FAKE_DIR = os.path.join(HERE, "support", "_build", "fake_cudart")
FAKE = os.path.join(FAKE_DIR, "libcudart.so.12")
INNER = os.environ.get("LLMLB_FAKE_CUDART") == "1"
inner = pytest.mark.skipif(not INNER, reason="runs in the child process that preloads the fake CUDA runtime")


def build_fake():
    os.makedirs(FAKE_DIR, exist_ok=True)
    src = os.path.join(HERE, "support", "fake_cudart.cpp")
    if not os.path.exists(FAKE) or os.path.getmtime(FAKE) < os.path.getmtime(src):
        subprocess.check_call(["g++", "-O1", "-g", "-std=c++17", "-shared", "-fPIC", "-I/usr/local/cuda/include", src, "-Wl,-soname,libcudart.so.12",
                               "-Wl,--version-script=" + os.path.join(HERE, "support", "fake_cudart.map"), "-o", FAKE])
    return FAKE


def test_engine_host_logic_over_the_fake_cuda_runtime(built_lib):
    if INNER:
        pytest.skip("already inside")
    env = dict(os.environ, LD_PRELOAD=build_fake(), LLMLB_FAKE_CUDART="1")
    # two child sessions: steps that take no time at all, and (for the scenarios that need requests to BE running while the
    # test acts on them) decode steps of 2 ms.  -s: a sanitizer report must reach the log, not pytest's capture file
    for extra_env, select in (({}, "scenario and not slowstep"), ({"FAKE_CUDART_STEP_US": "2000"}, "slowstep")):
        r = subprocess.run([sys.executable, "-m", "pytest", os.path.abspath(__file__), "-x", "-q", "-s", "-p", "no:cacheprovider", "-k", select],
                           capture_output=True, text=True, timeout=900, env=dict(env, **extra_env), cwd=ROOT)
        assert r.returncode == 0, r.stdout[-6000:] + r.stderr[-3000:]
        assert " passed" in r.stdout and "skipped" not in r.stdout.splitlines()[-1], r.stdout[-500:]


# ---------------------------------------------------------------------------------------------------------------------
TINY = dict(hidden=512, n_layers=2, n_heads=8, n_kv_heads=2, head_dim=128, ffn=1024, vocab=2048, rope_theta=500000.0, rms_eps=1e-5)
NONE, STOP, LENGTH, CANCELLED, ERROR, QUEUE_TIMEOUT, DEADLINE = range(7)


def _ffi():
    from llmlb_b200 import ffi
    alt = os.environ.get("LLMLB_HOST_LOGIC_LIB")      # a sanitizer build of the same sources (long pass, DESIGN.md)
    if alt:
        ffi.LIB_PATH = alt
    return ffi


def drain(eng, rid, timeout_s=30):
    evs, t0 = [], time.time()
    while time.time() - t0 < timeout_s:
        got = eng.poll(rid, timeout_ms=50)
        evs += got
        if got and got[-1]["finish_reason"]:
            return evs
    raise AssertionError("request %d did not finish: %s" % (rid, evs[-3:]))


def settle(eng, timeout_s=10):
    """wait until the scheduler has nothing left, then return health"""
    t0 = time.time()
    while time.time() - t0 < timeout_s:
        h = eng.health()
        if h["active_requests"] == 0 and h["queued_requests"] == 0:
            return h
        time.sleep(0.01)
    raise AssertionError("engine did not go idle: %s" % eng.health())


@inner
def test_scenario_events_are_complete_ordered_and_accounted():
    ffi = _ffi()
    with ffi.Engine(TINY, max_seqs=8, max_ctx=1024) as eng:
        h0 = eng.health()
        rids = [eng.submit(list(range(1, 1 + n)), m, ignore_eos=True) for n, m in ((5, 1), (64, 7), (65, 40), (300, 128), (1, 3))]
        for rid, (n, m) in zip(rids, ((5, 1), (64, 7), (65, 40), (300, 128), (1, 3))):
            evs = drain(eng, rid)
            toks = [e for e in evs if e["token_id"] >= 0]
            assert [e["index"] for e in toks] == list(range(m)) and len(toks) == m
            assert all(e["prompt_tokens"] == n for e in evs) and [e["completion_tokens"] for e in toks] == list(range(1, m + 1))
            assert [e["finish_reason"] for e in evs[:-1]] == [NONE] * (len(evs) - 1) and evs[-1]["finish_reason"] == LENGTH
            assert all(a["t_ms"] <= b["t_ms"] for a, b in zip(evs, evs[1:]))
            eng.release(rid)
        h = settle(eng)
        assert h["free_kv_pages"] == h["total_kv_pages"] == h0["total_kv_pages"]          # every page came back
        assert h["tokens_prefill"] - h0["tokens_prefill"] == 5 + 64 + 65 + 300 + 1
        # a prefill step samples the first token; every later token is one decode step of its sequence
        assert h["tokens_decode"] - h0["tokens_decode"] == sum(m - 1 for m in (1, 7, 40, 128, 3))
        with pytest.raises(ffi.LlmlbError):
            eng.poll(rids[0])                                                              # released ids are gone


@inner
def test_scenario_stop_ids_cancel_release_and_argument_checks():
    ffi = _ffi()
    with ffi.Engine(TINY, max_seqs=4, max_ctx=512) as eng:
        # every sampled id is 0 here: a stop id of 0 ends the request at its first token, ignore_eos overrides it
        evs = drain(eng, eng.submit([3, 4, 5], 50, stop_ids=[0]))
        assert [e["finish_reason"] for e in evs] == [STOP] and evs[0]["completion_tokens"] == 1
        evs = drain(eng, eng.submit([3, 4, 5], 6, stop_ids=[0], ignore_eos=True))
        assert len(evs) == 6 and evs[-1]["finish_reason"] == LENGTH
        evs = drain(eng, eng.submit([3, 4, 5], 6, stop_ids=[7, 9]))
        assert len(evs) == 6 and evs[-1]["finish_reason"] == LENGTH
        # cancel: while paused nothing is scheduled, so the request is still waiting when the cancel lands
        eng.pause(True)
        rid = eng.submit([1] * 40, 100, ignore_eos=True)
        assert eng.poll(rid, timeout_ms=20) == []
        eng.cancel(rid)
        eng.pause(False)
        evs = drain(eng, rid)
        assert evs[-1]["finish_reason"] == CANCELLED and evs[-1]["token_id"] == -1 and evs[-1]["completion_tokens"] == 0
        # release of a request in flight cancels it and frees everything it held
        rid = eng.submit([1] * 200, 300, ignore_eos=True)
        eng.release(rid)
        h = settle(eng)
        assert h["free_kv_pages"] == h["total_kv_pages"]
        for bad in (lambda: eng.submit([], 4), lambda: eng.submit([1, 2], 0), lambda: eng.submit([TINY["vocab"]], 4), lambda: eng.submit([-1], 4),
                    lambda: eng.submit([1] * 500, 100), lambda: eng.submit([1], 4, temperature=-1.0), lambda: eng.cancel(10 ** 9), lambda: eng.release(10 ** 9)):
            with pytest.raises(ffi.LlmlbError):
                bad()
        assert settle(eng)["free_kv_pages"] == h["total_kv_pages"]


@inner
def test_scenario_oversubscribed_pages_preempt_and_everything_still_completes():
    """kv_pages far below what the running set needs: sequences take pages as they grow, the youngest is evicted when the
    pool runs dry and recomputed later; every request still delivers exactly max_tokens events, in order, once."""
    ffi = _ffi()
    with ffi.Engine(TINY, max_seqs=8, max_ctx=1024, kv_pages=14) as eng:          # 14 pages x 64 tokens for 8 x (100 + 300) tokens
        rids = [eng.submit([1 + i] * 100, 300, ignore_eos=True) for i in range(8)]
        for rid in rids:
            evs = drain(eng, rid, 60)
            toks = [e for e in evs if e["token_id"] >= 0]
            assert [e["index"] for e in toks] == list(range(300)) and evs[-1]["finish_reason"] == LENGTH
            assert all(e["prompt_tokens"] == 100 for e in evs)                  # usage reports the client's prompt, not the recompute context
            eng.release(rid)
        h = settle(eng)
        assert h["preemptions"] > 0 and h["free_kv_pages"] == h["total_kv_pages"] == 14
        assert h["tokens_prefill"] > 800                                        # recomputed contexts were prefilled again
        # a request the pool can never hold is refused at submit, not starved
        with pytest.raises(ffi.LlmlbError):
            eng.submit([1] * 600, 400)


@inner
def test_scenario_queue_limit_queue_timeout_and_deadline():
    ffi = _ffi()
    with ffi.Engine(TINY, max_seqs=1, max_ctx=512, queue_max=2, queue_timeout_ms=150, request_timeout_ms=60000) as eng:
        eng.pause(True)                                                         # nothing is admitted: the queue only grows
        a, b = eng.submit([1, 2, 3], 5), eng.submit([1, 2, 3], 5)
        with pytest.raises(ffi.LlmlbError) as ei:
            eng.submit([1, 2, 3], 5)
        assert ei.value.code == ffi.E_QUEUE_FULL
        time.sleep(0.4)                                                         # both waited longer than queue_timeout_ms
        eng.pause(False)
        for rid in (a, b):
            evs = drain(eng, rid)
            assert [e["finish_reason"] for e in evs] == [QUEUE_TIMEOUT] and evs[0]["completion_tokens"] == 0
        assert settle(eng)["queued_requests"] == 0
    with ffi.Engine(TINY, max_seqs=2, max_ctx=512, request_timeout_ms=120) as eng:
        eng.pause(True)
        rid = eng.submit([1, 2, 3], 5, ignore_eos=True)
        time.sleep(0.3)
        eng.pause(False)
        assert drain(eng, rid)[-1]["finish_reason"] == DEADLINE
        evs = drain(eng, eng.submit([1, 2, 3], 5, ignore_eos=True))            # a fresh request is unaffected
        assert len(evs) == 5 and evs[-1]["finish_reason"] == LENGTH


@inner
def test_scenario_many_threads_submit_poll_cancel_release_concurrently():
    """The ABI promises thread safety (tokio workers call it): 12 threads mix every entry point against one engine whose
    steps take microseconds, so interleavings that a GPU's millisecond steps hide are hit thousands of times."""
    import random
    ffi = _ffi()
    with ffi.Engine(TINY, max_seqs=8, max_ctx=512, kv_pages=24, queue_max=4096) as eng:
        errors, done = [], [0]
        lock = threading.Lock()

        def worker(seed):
            rs = random.Random(seed)
            try:
                for _ in range(60):
                    n, m = rs.randint(1, 120), rs.randint(1, 60)
                    rid = eng.submit([rs.randrange(TINY["vocab"]) for _ in range(n)], m, ignore_eos=True, temperature=rs.choice([0.0, 0.7]), seed=seed)
                    action = rs.random()
                    if action < 0.15:
                        eng.release(rid)                                        # fire and forget
                        continue
                    if action < 0.35:
                        time.sleep(rs.random() * 0.002)
                        eng.cancel(rid)
                    evs = drain(eng, rid, 60)
                    toks = [e for e in evs if e["token_id"] >= 0]
                    assert [e["index"] for e in toks] == list(range(len(toks)))
                    fr = evs[-1]["finish_reason"]
                    assert fr in (LENGTH, CANCELLED) and (fr != LENGTH or len(toks) == m) and len(toks) <= m
                    eng.health()
                    eng.release(rid)
                    with lock:
                        done[0] += 1
            except Exception as e:                                              # noqa: BLE001
                errors.append(repr(e))

        th = [threading.Thread(target=worker, args=(i,)) for i in range(12)]
        [t.start() for t in th]
        [t.join() for t in th]
        assert not errors, errors[:3]
        h = settle(eng, 30)
        assert done[0] > 400 and h["free_kv_pages"] == h["total_kv_pages"] == 24 and h["active_requests"] == 0


@inner
def test_scenario_destroy_with_requests_in_flight_and_many_engines():
    ffi = _ffi()
    for i in range(20):
        eng = ffi.Engine(TINY, max_seqs=4, max_ctx=512)
        rids = [eng.submit([1, 2, 3, 4], 200, ignore_eos=True) for _ in range(6)]
        if i % 2:
            eng.poll(rids[0], timeout_ms=5)
        eng.close()                                                             # waiting + running + in-flight steps: must not hang or crash


# ---- tensor-parallel serving through the plan channel: two PROCESSES, rank 0 owns the queue, rank 1 replays its log ----
def _tp_rank(rank, world, handles, barrier, name, out_q):
    try:
        # give a decode step a duration: with zero-time steps the scheduler thread re-takes the engine mutex so fast that a
        # cancel() can wait behind hundreds of steps (std::mutex is not fair; on a GPU the scheduler sleeps in the event wait)
        os.environ["FAKE_CUDART_STEP_US"] = "200"
        ffi = _ffi()
        eng = ffi.Engine(TINY, model_id="tp-plan", device=0, tp_rank=rank, tp_size=world, max_seqs=8, max_ctx=1024, seed=0)
        h = eng.tp_export()
        handles[rank * 64:(rank + 1) * 64] = list(h)
        barrier.wait(60)
        blob = bytes(handles[:])
        eng.tp_import([blob[r * 64:(r + 1) * 64] for r in range(world)])       # maps the peer's exchange region (shared memory under the fake runtime)
        barrier.wait(60)
        if rank == 0:
            eng.tp_plan_channel(name)
        barrier.wait(60)
        if rank != 0:
            eng.tp_plan_channel(name)
        barrier.wait(60)
        res = {}
        if rank == 0:
            prompts = [[(7 * i + j) % TINY["vocab"] for j in range(n)] for i, n in enumerate((64, 200, 17, 333, 90, 41))]
            gens = [24, 40, 12, 30, 900, 20]
            solo = drain(eng, eng.submit(prompts[0], gens[0], ignore_eos=True))
            rids = []
            for i, (p, g) in enumerate(zip(prompts, gens)):
                rids.append(eng.submit(p, g, ignore_eos=True))
                if i == 4:
                    eng.cancel(rids[4])                                         # steps take microseconds here: cancel before it can run dry
                time.sleep(0.001 * (i % 3))
            outs = [drain(eng, r, 60) for r in rids]
            for r in rids:
                eng.release(r)
            res = {"solo": len(solo), "lens": [sum(e["token_id"] >= 0 for e in o) for o in outs], "reasons": [o[-1]["finish_reason"] for o in outs]}
            settle(eng, 30)
        else:
            try:
                eng.submit([1, 2, 3], 4)
                res["follower_accepted_submit"] = True
            except ffi.LlmlbError:
                pass
        barrier.wait(120)                                                       # the follower keeps replaying until rank 0 is done
        if rank != 0:                                                           # ... and has drained the log: poll its counters until they stop moving
            last, t0 = None, time.time()
            while time.time() - t0 < 20:
                cur = eng.health()["kernel_launches"]
                if cur == last:
                    break
                last = cur
                time.sleep(0.2)
        hz = eng.health()
        res["counters"] = {k: hz[k] for k in ("steps_prefill", "steps_decode", "tokens_decode", "tokens_prefill", "kernel_launches", "preemptions")}
        res["pages"] = (hz["free_kv_pages"], hz["total_kv_pages"])
        out_q.put((rank, res))
        barrier.wait(60)
        eng.close()
    except Exception as e:                                                      # noqa: BLE001
        out_q.put((rank, {"error": repr(e)}))
        try:
            barrier.abort()
        except Exception:                                                       # noqa: BLE001
            pass


@inner
def test_scenario_two_rank_plan_channel_follower_replays_the_leader():
    """What `tools/tp_plan_check.py` does on GPUs, on the host side only: the follower's scheduler, fed by the leader's
    shared-memory log, takes the same steps — identical step / token / launch counters, all pages back on both ranks —
    through staggered arrivals, chunked prefill and a mid-flight cancellation; a follower refuses submits."""
    import multiprocessing as mp
    ctx = mp.get_context("spawn")
    world = 2
    handles = ctx.Array("B", 64 * world)
    barrier = ctx.Barrier(world)
    q = ctx.Queue()
    name = "llmlb_plan_cpu_%d" % os.getpid()
    ps = [ctx.Process(target=_tp_rank, args=(r, world, handles, barrier, name, q)) for r in range(world)]
    [p.start() for p in ps]
    got = dict(q.get(timeout=180) for _ in range(world))
    [p.join(60) for p in ps]
    assert all("error" not in v for v in got.values()), got
    lead, foll = got[0], got[1]
    assert lead["solo"] == 24 and lead["reasons"][4] == CANCELLED and lead["lens"][4] < 900
    assert all(lead["lens"][i] == g and lead["reasons"][i] == LENGTH for i, g in ((0, 24), (1, 40), (2, 12), (3, 30), (5, 20)))
    assert "follower_accepted_submit" not in foll
    assert lead["counters"] == foll["counters"], (lead["counters"], foll["counters"])
    assert lead["pages"][0] == lead["pages"][1] and foll["pages"][0] == foll["pages"][1]
    assert all(p.exitcode == 0 for p in ps)


@inner
def test_scenario_scheduler_invariants_over_random_workloads():
    """Property test of the scheduler (hypothesis): random engine shapes (sequences, page pool, prefill chunk, run-ahead) and
    random request mixes, some cancelled.  Invariants: exactly max_tokens events per surviving request with contiguous
    indices; usage reports the client's prompt; every page and slot comes back; prefill work >= the prompts (equal without
    preemption) in >= ceil(tokens / chunk) steps; without preemption one decode launch per token after the first."""
    from hypothesis import HealthCheck, given, settings, strategies as st
    ffi = _ffi()
    N = [0]

    @settings(max_examples=150, deadline=None, suppress_health_check=list(HealthCheck), derandomize=True)
    @given(st.integers(1, 8), st.integers(6, 40), st.sampled_from([64, 128, 500, 2048]), st.sampled_from([0, 1, 3]),
           st.lists(st.tuples(st.integers(1, 300), st.integers(1, 80), st.booleans()), min_size=1, max_size=14))
    def run(max_seqs, kv_pages, chunk, lookahead, reqs):
        N[0] += 1
        reqs = [(n, m, c) for n, m, c in reqs if (n + m + 63) // 64 <= kv_pages]            # submit refuses what can never fit
        if not reqs:
            return
        with ffi.Engine(TINY, max_seqs=max_seqs, max_ctx=512, kv_pages=kv_pages, max_step_tokens=chunk, lookahead=lookahead) as eng:
            eng.pause(True)                                                                  # one well-defined arrival order
            rids = [eng.submit([(i + j) % TINY["vocab"] for j in range(n)], m, ignore_eos=True) for i, (n, m, c) in enumerate(reqs)]
            for rid, (n, m, c) in zip(rids, reqs):
                if c:
                    eng.cancel(rid)
            eng.pause(False)
            for rid, (n, m, c) in zip(rids, reqs):
                evs = drain(eng, rid, 60)
                toks = [e for e in evs if e["token_id"] >= 0]
                assert all(e["prompt_tokens"] == n for e in evs)
                if c:
                    assert evs[-1]["finish_reason"] == CANCELLED and not toks                 # cancelled before it was ever scheduled
                else:
                    assert [e["index"] for e in toks] == list(range(m)) and evs[-1]["finish_reason"] == LENGTH
                eng.release(rid)
            h = settle(eng)
            live = [(n, m) for n, m, c in reqs if not c]
            assert h["free_kv_pages"] == h["total_kv_pages"] == kv_pages and h["active_requests"] == 0
            assert h["tokens_prefill"] >= sum(n for n, _ in live)
            assert h["steps_prefill"] >= -(-sum(n for n, _ in live) // chunk) or not live
            if h["preemptions"] == 0:
                assert h["tokens_prefill"] == sum(n for n, _ in live)
                assert h["tokens_decode"] == sum(m - 1 for _, m in live)

    run()
    assert N[0] >= 100, N                                                                   # the property really ran


@inner
def test_scenario_config5_workload_shape_through_the_scheduler():
    """BASELINE.json configs[4] as the scheduler sees it (tools/bench_70b_mixed.py measured it on 8 GPUs): Llama-3-70B widths,
    48 requests with prompts U[512, 8064] + 128 generated tokens, 8192-token contexts, 2048-token prefill chunks, 32 running
    sequences, the page pool over-subscribed to 20 % of the job (the GPU run used 35 %; with this seed's lengths that does
    not evict yet).  Every request completes with exactly 128 tokens, prompts are
    chunked, sequences are preempted and recomputed, all pages return.  (Two layers: depth does not change scheduling.)"""
    import random
    ffi = _ffi()
    model = dict(ffi.LLAMA3_70B, n_layers=2)
    rs = random.Random(7)
    lens = [rs.randint(512, 8064) for _ in range(48)]
    kv_pages = int(0.20 * sum((n + 128 + 63) // 64 for n in lens))
    with ffi.Engine(model, max_seqs=32, max_ctx=8192, kv_pages=kv_pages, max_step_tokens=2048) as eng:
        eng.pause(True)
        rids = [eng.submit([(i * 31 + j) % model["vocab"] for j in range(n)], 128, ignore_eos=True) for i, n in enumerate(lens)]
        eng.pause(False)
        for rid, n in zip(rids, lens):
            evs = drain(eng, rid, 120)
            toks = [e for e in evs if e["token_id"] >= 0]
            assert [e["index"] for e in toks] == list(range(128)) and evs[-1]["finish_reason"] == LENGTH and evs[-1]["prompt_tokens"] == n
            eng.release(rid)
        h = settle(eng, 30)
        assert h["free_kv_pages"] == h["total_kv_pages"] == kv_pages
        assert h["preemptions"] > 0 and h["tokens_prefill"] > sum(lens)                      # recomputation happened
        assert h["steps_prefill"] >= -(-sum(lens) // 2048)


@inner
def test_scenario_load_and_read_tensor_shard_slices():
    """llmlb_engine_load_tensor takes the FULL Hugging Face tensor on every rank and keeps that rank's Megatron slice
    (q/k/v/gate/up/lm_head by output rows, o/down by input columns, norms and the embedding replicated);
    llmlb_engine_read_tensor returns the slice.  Under the fake runtime "device" memory is real memory, so the product's own
    address arithmetic (fused qkv, interleaved gate/up rows) is checked against plain numpy slicing for tp = 1, 2 and 4."""
    import numpy as np
    ffi = _ffi()
    M = dict(TINY, n_kv_heads=4, n_heads=16)
    H, F, V, hd = M["hidden"], M["ffn"], M["vocab"], M["head_dim"]
    full = {"model.embed_tokens.weight": (V, H), "model.norm.weight": (1, H), "lm_head.weight": (V, H)}
    for l in range(M["n_layers"]):
        p = "model.layers.%d." % l
        full.update({p + "self_attn.q_proj.weight": (M["n_heads"] * hd, H), p + "self_attn.k_proj.weight": (M["n_kv_heads"] * hd, H),
                     p + "self_attn.v_proj.weight": (M["n_kv_heads"] * hd, H), p + "self_attn.o_proj.weight": (H, M["n_heads"] * hd),
                     p + "mlp.gate_proj.weight": (F, H), p + "mlp.up_proj.weight": (F, H), p + "mlp.down_proj.weight": (H, F),
                     p + "input_layernorm.weight": (1, H), p + "post_attention_layernorm.weight": (1, H)})
    rs = np.random.RandomState(0)
    data = {k: rs.randint(0, 65536, size=s).astype(np.uint16) for k, s in full.items()}
    by_rows = ("q_proj", "k_proj", "v_proj", "gate_proj", "up_proj", "lm_head")
    by_cols = ("o_proj", "down_proj")
    for tp in (1, 2, 4):
        engs = [ffi.Engine(M, tp_rank=r, tp_size=tp, max_seqs=2, max_ctx=256) for r in range(tp)]
        try:
            for r, e in enumerate(engs):
                for name, a in data.items():
                    e.load_tensor(name, a if a.shape[0] > 1 else a.reshape(-1))
                for name, a in data.items():           # read everything back only after everything was loaded: slices must not overlap
                    got = e.read_tensor(name, a.size)
                    if any(k in name for k in by_rows):
                        n = a.shape[0] // tp
                        want = a[r * n:(r + 1) * n]
                    elif any(k in name for k in by_cols):
                        n = a.shape[1] // tp
                        want = a[:, r * n:(r + 1) * n]
                    else:
                        want = a
                    assert got.shape == want.shape and np.array_equal(got, want), (tp, r, name)
            e = engs[0]
            with pytest.raises(ffi.LlmlbError):
                e.load_tensor("model.layers.0.mlp.up_proj.weight", data["model.layers.0.mlp.down_proj.weight"])      # transposed shape
            with pytest.raises(ffi.LlmlbError):
                e.load_tensor("model.layers.9.mlp.up_proj.weight", data["model.layers.0.mlp.up_proj.weight"])        # no such layer
            with pytest.raises(ffi.LlmlbError):
                e.read_tensor("model.rotary.inv_freq", 16)
            with pytest.raises(ffi.LlmlbError):
                e.read_tensor("lm_head.weight", 8)                                                                   # buffer too small
        finally:
            for e in engs:
                e.close()


@inner
def test_scenario_allocation_footprint_of_the_baseline_configurations_fits_a_b200():
    """What the engine allocates (every cudaMalloc, counted by the fake runtime) for the BASELINE.json configurations, against
    180 GB per GPU and against the sizes DESIGN.md section 3 states: bf16 matmul weights per rank, 2 x layers x kv_heads/tp x
    64 x 128 x 2 B per KV page, and a remainder (embedding table, activations, workspaces, exchange region) under 3 GB."""
    ffi = _ffi()
    GB = 1e9
    for tag, model, kw, weights_gb in (
            ("configs[1] 8B batch 1", ffi.LLAMA3_8B, dict(max_seqs=8, max_ctx=1024), 15.01),
            ("configs[2] 8B 64 streams", ffi.LLAMA3_8B, dict(max_seqs=64, max_ctx=1024), 15.01),
            ("8B 128 x 8192 on one GPU", ffi.LLAMA3_8B, dict(max_seqs=128, max_ctx=8192), 15.01),
            ("configs[3] 8B tp8 128 streams", ffi.LLAMA3_8B, dict(max_seqs=128, max_ctx=1024, tp_size=8, tp_rank=3), 15.01 / 8),
            ("configs[4] 70B tp8 8192 ctx", ffi.LLAMA3_70B, dict(max_seqs=32, max_ctx=8192, tp_size=8, tp_rank=7), 139.0 / 8)):
        with ffi.Engine(model, **kw) as e:
            h, mi = e.health(), e.model_info()
            tp = kw.get("tp_size", 1)
            assert h["total_kv_pages"] == kw["max_seqs"] * kw["max_ctx"] // 64, tag
            kv = h["total_kv_pages"] * model["n_layers"] * 2 * (model["n_kv_heads"] // tp) * 64 * 128 * 2
            assert abs(mi["param_bytes"] / GB - weights_gb) < 0.02 * weights_gb + 0.01, (tag, mi["param_bytes"])
            rest = h["used_memory_bytes"] - mi["param_bytes"] - kv
            assert 0 < rest < 3 * GB, (tag, rest)
            assert h["used_memory_bytes"] < 180 * GB, (tag, h["used_memory_bytes"])


@inner
def test_scenario_random_api_call_sequences_never_break_the_engine():
    """A stateful random walk over the whole C ABI of one engine — submit (valid and invalid), poll, cancel, release (also
    twice, also of ids that never existed), pause toggles, health, model info, tensor load / read, the debug hooks while
    requests are in flight (they must refuse, not interfere) — 6000 operations.  Every call returns OK or a documented
    error code; at the end everything drains and every page is back.  (Runs under ASan/TSan in the sanitizer pass.)"""
    import random
    import numpy as np
    ffi = _ffi()
    rs = random.Random(3)
    ok_errors = {ffi.E_INVALID_ARG, ffi.E_QUEUE_FULL, ffi.E_TIMEOUT, getattr(ffi, "E_NOT_FOUND", -4), getattr(ffi, "E_UNSUPPORTED", -6)}
    with ffi.Engine(TINY, max_seqs=4, max_ctx=512, kv_pages=20, queue_max=16) as eng:
        live, dead = [], []
        paused = False
        n_ok = n_err = 0
        for step in range(6000):
            op = rs.randrange(12)
            try:
                if op <= 2:
                    n = rs.choice([0, 1, 5, 64, 65, 200, 511, 600])
                    m = rs.choice([0, 1, 3, 40, 300])
                    ids = [rs.randrange(-1 if rs.random() < 0.02 else 0, TINY["vocab"] + (1 if rs.random() < 0.02 else 0)) for _ in range(n)]
                    live.append(eng.submit(ids, m, ignore_eos=rs.random() < 0.5, temperature=rs.choice([0.0, 0.5, -1.0]), stop_ids=rs.choice([(), (0,), (5, 6)])))
                elif op <= 5 and live:
                    rid = rs.choice(live)
                    evs = eng.poll(rid, cap=rs.choice([1, 4, 256]), timeout_ms=rs.choice([0, 0, 1]))
                    assert all(a["index"] <= b["index"] for a, b in zip(evs, evs[1:]))
                elif op == 6 and live:
                    eng.cancel(rs.choice(live))
                elif op == 7 and (live or dead):
                    rid = rs.choice(live + dead)
                    eng.release(rid)
                    if rid in live:
                        live.remove(rid); dead.append(rid)
                elif op == 8:
                    paused = not paused
                    eng.pause(paused)
                elif op == 9:
                    h = eng.health()
                    assert h["free_kv_pages"] <= h["total_kv_pages"] == 20
                    eng.model_info()
                elif op == 10:
                    name = rs.choice(["model.norm.weight", "model.layers.1.mlp.up_proj.weight", "model.layers.7.mlp.up_proj.weight", "nope"])
                    if rs.random() < 0.5:
                        eng.read_tensor(name, rs.choice([16, 1 << 20]))
                    else:
                        eng.load_tensor(name, np.zeros(rs.choice([(1, 512), (1024, 512), (3, 3)]), dtype=np.uint16))
                elif op == 11:
                    if rs.random() < 0.5:
                        eng.debug_prefill_logits([1, 2, 3])
                    else:
                        eng.debug_reset()
                n_ok += 1
            except ffi.LlmlbError as e:
                assert e.code in ok_errors, (step, op, e)
                n_err += 1
        eng.pause(False)
        try:
            eng.debug_reset()
        except ffi.LlmlbError:
            pass
        for rid in live:
            eng.release(rid)
        h = settle(eng, 60)
        assert h["free_kv_pages"] == h["total_kv_pages"] == 20 and n_ok > 2000 and n_err > 300, (n_ok, n_err, h)


@inner
def test_scenario_slowstep_release_of_a_running_request_does_not_touch_its_neighbour():
    """Regression (found by AddressSanitizer over the fake runtime, fixed in engine.cu): finish_request took the request by
    reference to an element of `running` and erased that element — the reference then named the NEXT running request: the
    released request was never dropped from the id table (a leak per fire-and-forget release), the neighbour could be dropped
    instead while still running (its client would then get "unknown request id", and the last owner died inside erase:
    heap-use-after-free).  Needs requests that are running while the test acts, hence 2 ms decode steps."""
    assert os.environ.get("FAKE_CUDART_STEP_US") == "2000"
    ffi = _ffi()
    with ffi.Engine(TINY, max_seqs=4, max_ctx=512) as eng:
        a = eng.submit([1, 2, 3], 300, ignore_eos=True)
        b = eng.submit([4, 5, 6], 120, ignore_eos=True)
        c = eng.submit([7, 8, 9], 120, ignore_eos=True)
        for rid in (a, b, c):                                     # all three are running (each has produced a token)
            t0 = time.time()
            while not eng.poll(rid, cap=1, timeout_ms=100):
                assert time.time() - t0 < 10
        eng.release(a)                                            # in flight: cancelled by the scheduler, then dropped
        eng.release(b)                                            # its neighbour in `running`, also fire-and-forget
        time.sleep(0.1)
        for rid in (a, b):
            with pytest.raises(ffi.LlmlbError) as ei:             # both are gone from the id table (a second release finds nothing)
                eng.release(rid)
            assert ei.value.code == ffi.E_NOT_FOUND
        evs = drain(eng, c, 30)                                   # the third one is untouched: every token, still pollable
        assert evs[-1]["finish_reason"] == LENGTH and evs[-1]["completion_tokens"] == 120
        eng.release(c)
        h = settle(eng)
        assert h["free_kv_pages"] == h["total_kv_pages"]


@inner
def test_scenario_concurrent_random_walks_share_requests_across_threads():
    """Six threads run the random walk of the previous scenario against ONE engine and ONE shared list of request ids, so
    a thread polls what another cancels, releases what a third one is draining, and toggles pause under everybody: the
    interleavings the id-table bug above needed, thousands of times.  Every call returns OK or a documented error; in the
    end the engine drains and every page is back."""
    import random
    ffi = _ffi()
    ok_errors = {ffi.E_INVALID_ARG, ffi.E_QUEUE_FULL, ffi.E_TIMEOUT, ffi.E_NOT_FOUND, ffi.E_UNSUPPORTED}
    with ffi.Engine(TINY, max_seqs=6, max_ctx=512, kv_pages=30, queue_max=64) as eng:
        ids, lock, errors = [], threading.Lock(), []

        def walk(seed):
            rs = random.Random(seed)
            try:
                for _ in range(1500):
                    op = rs.randrange(10)
                    with lock:
                        rid = rs.choice(ids) if ids else None
                    try:
                        if op <= 2:
                            n, m = rs.choice([1, 5, 64, 65, 200]), rs.choice([1, 3, 40, 200])
                            new = eng.submit([rs.randrange(TINY["vocab"]) for _ in range(n)], m, ignore_eos=rs.random() < 0.7, stop_ids=rs.choice([(), (0,)]))
                            with lock:
                                ids.append(new)
                        elif op <= 5 and rid is not None:
                            evs = eng.poll(rid, cap=rs.choice([1, 8, 256]), timeout_ms=rs.choice([0, 0, 1]))
                            assert all(a["index"] <= b["index"] for a, b in zip(evs, evs[1:]))
                        elif op == 6 and rid is not None:
                            eng.cancel(rid)
                        elif op == 7 and rid is not None:
                            eng.release(rid)
                            with lock:
                                if rid in ids and rs.random() < 0.8:
                                    ids.remove(rid)                      # sometimes the id stays listed: double releases, polls of dead ids
                        elif op == 8:
                            eng.pause(rs.random() < 0.3)
                        else:
                            h = eng.health()
                            assert h["free_kv_pages"] <= h["total_kv_pages"] == 30
                    except ffi.LlmlbError as e:
                        assert e.code in ok_errors, e
            except Exception as e:                                       # noqa: BLE001
                errors.append(repr(e))

        th = [threading.Thread(target=walk, args=(s,)) for s in range(6)]
        [t.start() for t in th]
        [t.join() for t in th]
        assert not errors, errors[:3]
        eng.pause(False)
        for rid in list(ids):
            try:
                eng.release(rid)
            except ffi.LlmlbError:
                pass
        h = settle(eng, 60)
        assert h["free_kv_pages"] == h["total_kv_pages"] == 30


def _tp_rank_random(rank, world, handles, barrier, name, out_q):
    try:
        import random
        os.environ["FAKE_CUDART_STEP_US"] = "100"
        ffi = _ffi()
        eng = ffi.Engine(TINY, model_id="tp-plan", device=0, tp_rank=rank, tp_size=world, max_seqs=4, max_ctx=512, kv_pages=10, queue_max=32,
                         queue_timeout_ms=10, request_timeout_ms=40, seed=0)
        handles[rank * 64:(rank + 1) * 64] = list(eng.tp_export())
        barrier.wait(60)
        blob = bytes(handles[:])
        eng.tp_import([blob[r * 64:(r + 1) * 64] for r in range(world)])
        barrier.wait(60)
        if rank == 0:
            eng.tp_plan_channel(name)
        barrier.wait(60)
        if rank != 0:
            eng.tp_plan_channel(name)
        barrier.wait(60)
        res = {"finish": {}}
        if rank == 0:
            rs = random.Random(11)
            live = []
            for _ in range(700):
                op = rs.randrange(10)
                try:
                    if op <= 3:
                        live.append(eng.submit([rs.randrange(TINY["vocab"]) for _ in range(rs.choice([1, 30, 64, 65, 150]))], rs.choice([1, 5, 40, 300]),
                                               ignore_eos=True, temperature=rs.choice([0.0, 0.8]), seed=rs.randrange(100)))
                    elif op <= 5 and live:
                        for e in eng.poll(rs.choice(live), timeout_ms=rs.choice([0, 1])):
                            if e["finish_reason"]:
                                res["finish"][e["finish_reason"]] = res["finish"].get(e["finish_reason"], 0) + 1
                    elif op == 6 and live:
                        eng.cancel(rs.choice(live))
                    elif op == 7 and live:
                        eng.release(live.pop(rs.randrange(len(live))))
                    elif op == 8:
                        eng.pause(rs.random() < 0.25)
                    else:
                        time.sleep(rs.choice([0, 0.001, 0.02]))              # lets queue timeouts and deadlines expire on the leader's clock
                except ffi.LlmlbError as e:
                    assert e.code in (ffi.E_QUEUE_FULL, ffi.E_INVALID_ARG, ffi.E_NOT_FOUND), e
            eng.pause(False)
            for r in live:
                eng.release(r)
            settle(eng, 60)
        barrier.wait(180)
        if rank != 0:
            last, t0 = None, time.time()
            while time.time() - t0 < 30:
                cur = eng.health()["kernel_launches"]
                if cur == last:
                    break
                last = cur
                time.sleep(0.3)
        hz = eng.health()
        res["counters"] = {k: hz[k] for k in ("steps_prefill", "steps_decode", "tokens_decode", "tokens_prefill", "kernel_launches", "preemptions")}
        res["pages"] = (hz["free_kv_pages"], hz["total_kv_pages"])
        out_q.put((rank, res))
        barrier.wait(60)
        eng.close()
    except Exception as e:                                                      # noqa: BLE001
        import traceback
        out_q.put((rank, {"error": repr(e) + traceback.format_exc()[-800:]}))
        try:
            barrier.abort()
        except Exception:                                                       # noqa: BLE001
            pass


@inner
def test_scenario_two_rank_plan_channel_replays_every_kind_of_event():
    """The leader runs a 700-operation random walk — submits (greedy and sampled), polls, cancels, releases in flight, pause
    toggles, sleeps that let queue timeouts (10 ms) and deadlines (40 ms) expire on ITS clock, a 10-page pool that forces
    preemption — and the follower, which sees nothing but the shared-memory log, must end with the same step, token, launch
    and preemption counters and every page free: each logged event type (submit, cancel, release, pause, expire, schedule,
    harvest) is replayed in order."""
    import multiprocessing as mp
    ctx = mp.get_context("spawn")
    world = 2
    handles, barrier, q = ctx.Array("B", 64 * world), ctx.Barrier(world), ctx.Queue()
    name = "llmlb_plan_rnd_%d" % os.getpid()
    ps = [ctx.Process(target=_tp_rank_random, args=(r, world, handles, barrier, name, q)) for r in range(world)]
    [p.start() for p in ps]
    got = dict(q.get(timeout=300) for _ in range(world))
    [p.join(60) for p in ps]
    assert all("error" not in v for v in got.values()), got
    lead, foll = got[0], got[1]
    assert lead["counters"] == foll["counters"], (lead["counters"], foll["counters"])
    assert lead["pages"][0] == lead["pages"][1] == 10 and foll["pages"] == lead["pages"]
    assert lead["counters"]["steps_decode"] > 100
    # which of cancel / queue timeout / deadline / preemption occur depends on the leader's clock; at least expiry did
    assert set(lead["finish"]) & {5, 6}, lead["finish"]
    assert all(p.exitcode == 0 for p in ps)


@inner
def test_scenario_tensor_parallel_depth_limit_is_refused_not_wrapped():
    """The decode exchange numbers its collectives (two per layer) in the low 8 bits of a 32-bit epoch: 127 layers fit
    (Llama-3.1-405B has 126), a deeper tensor-parallel stack would alias epochs of consecutive steps — create refuses it;
    a single-GPU engine has no such limit."""
    ffi = _ffi()
    ffi.Engine(dict(ffi.LLAMA3_70B, n_layers=126), tp_size=8, tp_rank=0, max_seqs=2, max_ctx=256).close()
    with pytest.raises(ffi.LlmlbError) as ei:
        ffi.Engine(dict(ffi.LLAMA3_70B, n_layers=128), tp_size=8, tp_rank=0, max_seqs=2, max_ctx=256)
    assert "127 layers" in str(ei.value)
    ffi.Engine(dict(TINY, n_layers=200), max_seqs=2, max_ctx=256).close()


@inner
@pytest.mark.parametrize("field,value", [("attn_impl", 1), ("tp_proto", 1), ("tp_proto", 2)])
def test_scenario_implementation_switches_other_than_zero_are_refused_at_create(field, value):
    """gemm_impl, attn_impl and tp_proto keep their places in the config struct, but the library holds one implementation
    of each: any value other than 0 is refused at create, not ignored.  The same config with 0 creates an engine."""
    import ctypes as C
    ffi = _ffi()
    cfg = ffi.EngineConfig()
    cfg.abi_version = ffi.ABI_VERSION
    for k, v in TINY.items():
        setattr(cfg.model, k, v)
    cfg.max_seqs, cfg.max_ctx, cfg.kv_block_tokens = 2, 256, 64
    setattr(cfg, field, value)
    h = C.c_void_p()
    assert ffi.lib().llmlb_engine_create(C.byref(cfg), C.byref(h)) == ffi.E_INVALID_ARG and not h
    assert field in ffi.last_error()
    setattr(cfg, field, 0)
    assert ffi.lib().llmlb_engine_create(C.byref(cfg), C.byref(h)) == ffi.OK and h
    ffi.lib().llmlb_engine_destroy(h)
