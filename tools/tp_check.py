"""Tensor-parallel parity check (run under torchrun, one rank per GPU):

    python -m torch.distributed.run --nproc-per-node 2 --master-addr 127.0.0.1 tools/tp_check.py [--geom odd]

Every rank builds a small geometry sharded tp=world and wires the peer-memory exchange through the
C ABI.  Rank 0 compares with the CPU oracle (oracle/llama_ref.py) AND with a tp=1 engine of the same
model on its own GPU:
  * prefill logits of a 150-token prompt          -> protocol B (reduce-scatter / all-gather by address),
                                                     row chunks that do not divide evenly
  * prefill logits of a 3-token prompt            -> protocol A through the non-decode path (fold kernel)
  * two teacher-forced decode steps               -> protocol A fused into the GEMV prologue / epilogue
  * 3 staggered requests + 7 concurrent requests  -> CUDA-graph decode at widths 1..3 (A) and 7 (B),
                                                     packed prefill, all ranks must emit identical tokens
`--geom odd` uses an FFN width whose down projection the fused GEMV does not take at 3-4 rows, so
the unfused push / fold kernels run too.  tests/test_tp_gpu.py launches this for 2, 4 and 8 GPUs."""
import argparse
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from llmlb_b200 import ffi  # noqa: E402

TOL = 0.03        # max |dlogit| vs the fp32 oracle (tests/test_engine_gpu.py LOGIT_TOL)
NEAR = 0.06       # teacher-forced tokens must be within this of the oracle's arg-max logit


def geometry(world, kind):
    if kind == "8b4":                         # full Llama-3-8B widths, 4 layers: the shard shapes of the benchmark
        cfg = dict(ffi.LLAMA3_8B)
        cfg["n_layers"] = 4
        return cfg
    cfg = dict(ffi.LLAMA_TINY)
    cfg["n_kv_heads"] = max(2, world)         # kv heads must divide by tp
    cfg["n_heads"] = 4 * cfg["n_kv_heads"]
    cfg["hidden"] = 128 * cfg["n_heads"] // 2 if world <= 2 else 1024
    if kind == "odd":
        cfg["ffn"] = 5120 * world             # per-rank K = 5120 = 20 chunks of 256: the fused GEMV takes <= 2 rows
    return cfg


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--geom", default="tiny", choices=["tiny", "odd", "8b4"])
    args = ap.parse_args()
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    cfg = geometry(world, args.geom)
    eng = ffi.Engine(cfg, device=local, tp_rank=rank, tp_size=world, max_seqs=8, max_ctx=1024, seed=0)
    handles = [None] * world
    dist.all_gather_object(handles, eng.tp_export())
    eng.tp_import(handles)
    dist.barrier()
    big = args.geom == "8b4"
    prompt = np.random.RandomState(3).randint(0, cfg["vocab"], 512 if big else 150).tolist()
    lg = eng.debug_prefill_logits(prompt)
    step = [eng.debug_decode_logits(7), eng.debug_decode_logits(99)]
    eng.debug_reset()
    lg3 = eng.debug_prefill_logits(prompt[:3])
    step3 = eng.debug_decode_logits(11)
    eng.debug_reset()
    dist.barrier()

    def run_batch(prompts, n_new):   # identical queues on every rank, then go
        eng.pause(True)
        rids = [eng.submit(p, n_new, ignore_eos=True) for p in prompts]
        dist.barrier()
        eng.pause(False)
        outs = []
        for r in rids:
            out = []
            while True:
                ev = eng.poll(r, timeout_ms=-1)
                out += [e["token_id"] for e in ev if e["token_id"] >= 0]
                if ev and ev[-1]["finish_reason"]:
                    break
            eng.release(r)
            outs.append(out)
        return outs

    p3 = [prompt[: 40 + 30 * i] for i in range(3)]
    toks3 = run_batch(p3, 24)
    p7 = [np.random.RandomState(50 + i).randint(0, cfg["vocab"], 9 + 11 * i).tolist() for i in range(7)]
    toks7 = run_batch(p7, 10)
    gathered = [None] * world
    dist.all_gather_object(gathered, (lg[:64].tolist(), toks3, toks7))
    eng.close()
    ok = True
    if rank == 0 and big:
        # 8B widths: the tp = 1 engine (itself pinned to the oracle by tests/test_parity_8b_gpu.py) is the checker
        with ffi.Engine(cfg, device=local, max_seqs=8, max_ctx=1024, seed=0) as one:
            l1 = one.debug_prefill_logits(prompt)
            s1 = [one.debug_decode_logits(7), one.debug_decode_logits(99)]
            one.debug_reset()
            l3 = one.debug_prefill_logits(prompt[:3])
            s3 = one.debug_decode_logits(11)
            one.debug_reset()
            ref3 = [one.generate(p, 24, ignore_eos=True)[0] for p in p3]
            # batched steps (3-wide protocol A, 7-wide protocol B): every token the sharded engine picked must be a
            # near-arg-max of the tp=1 engine's logits when teacher-forced along the sharded engine's own tokens
            worst = 0.0
            for pr, ts in list(zip(p3, toks3)) + list(zip(p7, toks7)):
                cur = one.debug_prefill_logits(pr)
                for j, tok in enumerate(ts):
                    worst = max(worst, float(cur.max() - cur[tok]))
                    if j + 1 < len(ts):
                        cur = one.debug_decode_logits(tok)
                one.debug_reset()
        d = [float(np.abs(lg - l1).max()), float(np.abs(step[0] - s1[0]).max()), float(np.abs(step[1] - s1[1]).max()),
             float(np.abs(lg3 - l3).max()), float(np.abs(step3 - s3).max())]
        same = all(g == gathered[0] for g in gathered)
        eq3 = sum(int(a == b) for a, b in zip(toks3, ref3))
        lens_ok = all(len(t) == 24 for t in toks3) and all(len(t) == 10 for t in toks7)
        print("tp=%d geom=8b4 max|dlogit| vs tp=1 engine: prefill512 %.4g decode %.4g %.4g prefill3 %.4g decode %.4g (logit std %.3f); "
              "ranks identical: %s; staggered requests token-identical to tp=1: %d/3; worst margin of a batched-step token to the tp=1 arg-max %.4f; lengths ok: %s"
              % (world, d[0], d[1], d[2], d[3], d[4], float(l1.std()), same, eq3, worst, lens_ok))
        # measured on B200: 0.062 (tp=2), 0.072 (tp=8) on prefill512 at a logit std of 1.28 (bf16 partials on the wire, N-way order)
        ok = max(d) < 0.10 and same and lens_ok and worst < 0.2
    elif rank == 0:
        from oracle.llama_ref import LlamaRef
        from oracle.synth import synth_state_dict
        sd = synth_state_dict(cfg, 0)
        ref = LlamaRef(cfg, sd)
        rl = ref.forward(prompt).numpy()[-1]
        e0 = float(np.abs(lg - rl).max())
        e1 = float(np.abs(step[0] - ref.forward([7]).numpy()[-1]).max())
        e2 = float(np.abs(step[1] - ref.forward([99]).numpy()[-1]).max())
        ref.reset()
        e3 = float(np.abs(lg3 - ref.forward(prompt[:3]).numpy()[-1]).max())
        e4 = float(np.abs(step3 - ref.forward([11]).numpy()[-1]).max())
        same = all(g == gathered[0] for g in gathered)
        # teacher-forced: every engine token must be a (near-)arg-max of the oracle's logits
        agree, total, near = 0, 0, True
        detail = []
        # the near-arg-max margin follows the rounding noise of the widest dot product: the "odd" geometry's FFN grows with
        # the world size (5120 per rank), and bf16 activation rounding accumulates ~ sqrt(K)
        near_tol = NEAR * max(1.0, (cfg["ffn"] / 10240.0) ** 0.5)
        for ps, ts in ((p3, toks3), (p7, toks7)):
            for pr, t in zip(ps, ts):
                r2 = LlamaRef(cfg, sd)
                cur = r2.forward(pr).numpy()[-1]
                a = 0
                for tok in t:
                    near &= bool(cur[tok] >= cur.max() - near_tol)
                    a += int(tok == int(np.argmax(cur)))
                    total += 1
                    cur = r2.forward([tok]).numpy()[-1]
                agree += a
                detail.append("%d/%d" % (a, len(t)))
        lens_ok = all(len(t) == 24 for t in toks3) and all(len(t) == 10 for t in toks7)
        # the same model on ONE GPU: tensor parallelism only changes the summation order
        with ffi.Engine(cfg, device=local, max_seqs=8, max_ctx=512, seed=0) as one:
            l1 = one.debug_prefill_logits(prompt)
            s1 = [one.debug_decode_logits(7), one.debug_decode_logits(99)]
        d0 = float(np.abs(lg - l1).max())
        d1 = max(float(np.abs(a - b).max()) for a, b in zip(step, s1))
        print("tp=%d geom=%s max|dlogit| vs oracle: prefill150 %.4g decode %.4g %.4g prefill3 %.4g decode %.4g; vs tp=1 engine: prefill %.4g decode %.4g; "
              "ranks identical: %s; top-1 agreement %d/%d (per request %s), all near-argmax: %s, lengths ok: %s"
              % (world, args.geom, e0, e1, e2, e3, e4, d0, d1, same, agree, total, " ".join(detail), near, lens_ok))
        ok = max(e0, e1, e2, e3, e4) < TOL and max(d0, d1) < TOL and same and near and lens_ok and agree >= int(0.9 * total)
    flag = torch.tensor([1 if ok else 0], device="cuda")
    dist.broadcast(flag, 0)
    dist.destroy_process_group()
    sys.exit(0 if flag.item() else 1)


if __name__ == "__main__":
    main()
