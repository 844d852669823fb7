"""Tensor-parallel determinism / parity probe (torchrun, one rank per GPU).  One 512-token prompt, 128 greedy
tokens, generated --runs times through submit/poll on the sharded engine:
  * how many distinct token sequences came out (a race shows up as run-to-run differences),
  * run 0 teacher-forced through the sharded engine's OWN eager parity hooks (debug_prefill_logits /
    debug_decode_logits): margin of every generated token to that path's arg-max — separates
    "submit path vs eager path of the same engine" from "tp vs tp=1",
  * run 0 teacher-forced through a tp=1 engine on rank 0's GPU (what bench.py's parity record does).

    python -m torch.distributed.run --nproc-per-node 2 --master-addr 127.0.0.1 tools/tp_race_probe.py --max-seqs 64"""
import argparse
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from llmlb_b200 import ffi  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--max-seqs", type=int, default=64)
    ap.add_argument("--lookahead", type=int, default=0)
    ap.add_argument("--no-graphs", action="store_true")
    ap.add_argument("--runs", type=int, default=4)
    ap.add_argument("--gen", type=int, default=128)
    ap.add_argument("--kv-pages", type=int, default=0)
    ap.add_argument("--tag", default="")
    args = ap.parse_args()
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    model = ffi.LLAMA3_8B
    eng = ffi.Engine(model, device=local, tp_rank=rank, tp_size=world, max_seqs=args.max_seqs, max_ctx=1024, seed=0,
                     kv_pages=args.kv_pages, use_cuda_graphs=not args.no_graphs, lookahead=args.lookahead)
    handles = [None] * world
    dist.all_gather_object(handles, eng.tp_export())
    eng.tp_import(handles)
    dist.barrier()
    prompt = np.random.RandomState(1000).randint(0, model["vocab"], 512).astype("int32").tolist()

    def gen():
        eng.pause(True)
        rid = eng.submit(prompt, args.gen, ignore_eos=True)
        dist.barrier()
        eng.pause(False)
        out = []
        while True:
            ev = eng.poll(rid, timeout_ms=-1)
            out += [e["token_id"] for e in ev if e["token_id"] >= 0]
            if ev and ev[-1]["finish_reason"]:
                break
        eng.release(rid)
        return out

    seqs = [gen() for _ in range(args.runs)]
    # the engine's own eager path, teacher-forced with run 0 (every rank takes part: the collectives need all of them)
    lg = eng.debug_prefill_logits(prompt)
    own_m, own_agree = [], 0
    for i, t in enumerate(seqs[0]):
        own_m.append(float(lg.max() - lg[t])); own_agree += int(int(np.argmax(lg)) == t)
        if i + 1 < len(seqs[0]):
            lg = eng.debug_decode_logits(t)
    eng.debug_reset()
    allr = [None] * world
    dist.all_gather_object(allr, seqs)
    if rank == 0:
        first_div = [next((i for i, (a, b) in enumerate(zip(s, seqs[0])) if a != b), None) for s in seqs]
        with ffi.Engine(model, device=local, max_seqs=4, max_ctx=1024, seed=0) as one:
            lg = one.debug_prefill_logits(prompt)
            m1, agree1 = [], 0
            for i, t in enumerate(seqs[0]):
                m1.append(float(lg.max() - lg[t])); agree1 += int(int(np.argmax(lg)) == t)
                if i + 1 < len(seqs[0]):
                    lg = one.debug_decode_logits(t)
        worst = int(np.argmax(m1))
        print("%s tp=%d max_seqs=%d graphs=%s lookahead=%d: %d distinct sequences in %d runs (first divergence %s), ranks identical %s | "
              "vs own eager path: top-1 %d/%d, max margin %.4f at step %d | vs tp=1 engine: top-1 %d/%d, max margin %.4f at step %d, margins > 0.1 at steps %s"
              % (args.tag, world, args.max_seqs, not args.no_graphs, args.lookahead or 2, len(set(map(tuple, seqs))), len(seqs), first_div,
                 all(a == seqs for a in allr), own_agree, len(own_m), max(own_m), int(np.argmax(own_m)), agree1, len(m1), max(m1), worst,
                 [i for i, v in enumerate(m1) if v > 0.1]))
        sys.stdout.flush()
    eng.close()
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
