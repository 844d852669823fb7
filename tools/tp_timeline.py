"""In-kernel %globaltimer timeline of one prefill step and one decode step at tensor-parallel width N
(or N = 1): where the time between and inside the kernels goes — launch gaps, dependency waits,
flag waits of the push collectives.  Rank 0's GPU is traced.

    python -m torch.distributed.run --nproc-per-node 2 --master-addr 127.0.0.1 tools/tp_timeline.py [--streams 1]
    python tools/tp_timeline.py          # single GPU

Records (llmlb_debug_trace_*): thread 0 of every CTA appends (tag, cta|smid, t0..t3 in ns)."""
import argparse
import ctypes as C
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from llmlb_b200 import ffi  # noqa: E402

EPI = {0: "bf16", 1: "resid", 2: "silu", 3: "f32", 4: "partial", 5: "pushRS", 6: "pushRS-LL"}


def name(tag):
    kind = tag >> 60
    n_out, k = (tag >> 32) & 0xFFFFFF, tag & 0xFFFFFFFF
    if tag == 1:
        return "decode_attention"
    if kind == 0:
        tpm = (tag >> 58) & 3
        return "gemv%s %dx%d" % ({0: "", 1: "+consume", 2: "+push"}[tpm], n_out, k)
    if kind == 3:
        return "tp_reduce_norm T=%d" % k
    if kind == 4:
        return "gemm_tc2[%s] %dx%d" % (EPI.get((tag >> 56) & 15, "?"), n_out, k)
    if kind == 6:
        return "gemm_tc[%s] %dx%d" % (EPI.get((tag >> 56) & 15, "?"), n_out, k)
    if kind == 5:
        return "(consume detail) %dx%d" % (n_out, k)
    return "tag%x" % tag


def launches_of(r):
    """cluster the per-CTA records of every tag into launches (CTAs of one grid start within ~2 us)"""
    out = []
    for tag in np.unique(r[:, 0]):
        t = int(tag)
        if (t >> 60) in (2, 5):
            continue
        rows = r[r[:, 0] == tag]
        rows = rows[np.argsort(rows[:, 2])]
        start = 0
        for i in range(1, len(rows) + 1):
            if i == len(rows) or int(rows[i, 2]) - int(rows[i - 1, 2]) > 3000:
                blk = rows[start:i].astype(np.int64)
                t3 = blk[:, 5] if (t >> 60) not in (4, 6) else blk[:, 4]
                out.append({"tag": t, "n": len(blk), "t0": int(blk[:, 2].min()), "dep": int(blk[:, 3].max()),
                            "mid": int(blk[:, 4].max()), "end": int(t3.max()), "end_first": int(t3.min())})
                start = i
    out.sort(key=lambda l: l["t0"])
    return out


def report(title, ls, detail_rows=None, max_lines=16):
    if not ls:
        return
    base = ls[0]["t0"]
    print("\n== %s: %d launches, %.1f us from first start to last end" % (title, len(ls), (max(l["end"] for l in ls) - base) / 1e3))
    print("%-34s %5s %9s %9s %9s %9s %9s" % ("kernel", "ctas", "start", "dep_ok", "phase2", "end", "gap_prev"))
    prev = None
    for l in ls[:max_lines]:
        gap = (l["t0"] - prev) / 1e3 if prev is not None else 0.0
        print("%-34s %5d %9.2f %9.2f %9.2f %9.2f %9.2f" % (name(l["tag"]), l["n"], (l["t0"] - base) / 1e3, (l["dep"] - base) / 1e3,
                                                          (l["mid"] - base) / 1e3, (l["end"] - base) / 1e3, gap))
        prev = l["end"]
    tot = {}
    prev = None
    for l in ls:
        d = tot.setdefault(name(l["tag"]), {"n": 0, "span": 0.0, "after_dep": 0.0, "exposed": 0.0})
        d["n"] += 1
        d["span"] += (l["end"] - l["t0"]) / 1e3
        d["after_dep"] += (l["end"] - l["dep"]) / 1e3
        d["exposed"] += (l["end"] - max(l["t0"], prev if prev is not None else l["t0"])) / 1e3   # time not hidden under the previous kernel
        prev = l["end"] if prev is None else max(prev, l["end"])
    print("%-34s %4s %10s %12s %12s" % ("totals by kernel", "n", "span_us", "after_dep_us", "exposed_us"))
    for k, d in sorted(tot.items(), key=lambda kv: -kv[1]["exposed"]):
        print("%-34s %4d %10.1f %12.1f %12.1f" % (k, d["n"], d["span"], d["after_dep"], d["exposed"]))
    if detail_rows is not None and len(detail_rows):
        a = detail_rows.astype(np.int64)
        w = (a[:, 3] - a[:, 2]) / 1e3   # dependency satisfied -> every peer's pairs arrived and folded
        f = (a[:, 4] - a[:, 3]) / 1e3   # fold done -> norm done
        print("GEMV consumers (protocol A): wait for + fold of the pushed pairs after the local dependency: mean %.2f us, p95 %.2f, max %.2f; norm: mean %.2f us"
              % (w.mean(), np.percentile(w, 95), w.max(), f.mean()))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--streams", type=int, default=1)
    ap.add_argument("--gen", type=int, default=6)
    args = ap.parse_args()
    rank, world, local = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("LOCAL_RANK", 0))
    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    L = ffi.lib()
    L.llmlb_debug_trace_enable.argtypes = [C.c_uint32]
    L.llmlb_debug_trace_dump.argtypes = [C.c_void_p, C.c_uint32, C.POINTER(C.c_uint32)]
    model = ffi.LLAMA3_8B
    eng = ffi.Engine(model, device=local, tp_rank=rank, tp_size=world, max_seqs=max(4, args.streams), max_ctx=1024, seed=0)
    if world > 1:
        handles = [None] * world
        dist.all_gather_object(handles, eng.tp_export())
        eng.tp_import(handles)
        dist.barrier()

    def run(n_new):
        if world > 1:
            eng.pause(True)
        rids = [eng.submit(np.random.RandomState(i).randint(0, model["vocab"], 512).tolist(), n_new, ignore_eos=True) for i in range(args.streams)]
        if world > 1:
            dist.barrier()
            eng.pause(False)
        for r in rids:
            while True:
                ev = eng.poll(r, timeout_ms=-1)
                if ev and ev[-1]["finish_reason"]:
                    break
            eng.release(r)
    run(8)   # warm: graphs captured
    cap = 1500000
    if world > 1:
        dist.barrier()
    L.llmlb_debug_trace_enable(cap if rank == 0 else 0)
    run(args.gen)
    if rank == 0:
        buf = np.zeros((cap, 6), dtype=np.uint64)
        n = C.c_uint32()
        L.llmlb_debug_trace_dump(buf.ctypes.data, cap, C.byref(n))
        L.llmlb_debug_trace_enable(0)
        r = buf[: n.value]
        if os.environ.get("TRACE_OUT"):
            np.save(os.environ["TRACE_OUT"], r)
        ls = launches_of(r)
        vl = model["vocab"] // world
        heads = [i for i, l in enumerate(ls) if (l["tag"] >> 60) in (0, 4, 6) and ((l["tag"] >> 32) & 0xFFFFFF) == vl]
        # one lm_head grid whose CTAs start more than 3 us apart (PDL early starters) shows up as adjacent pieces: keep the last
        heads = [h for j, h in enumerate(heads) if j + 1 == len(heads) or heads[j + 1] - h > 4]
        print("tp=%d streams=%d: %d trace records, %d launches, %d lm_head launches" % (world, args.streams, len(r), len(ls), len(heads)))
        det = r[(r[:, 0] >> np.uint64(60)) == np.uint64(5)]
        if heads:
            report("prefill step (512 tokens x %d)" % args.streams, ls[: heads[0] + 1], max_lines=14)
            if len(heads) >= 3:
                lo, hi = heads[-2] + 1, heads[-1] + 1
                win = ls[lo:hi]
                d = det[(det[:, 2] >= np.uint64(win[0]["t0"])) & (det[:, 2] <= np.uint64(win[-1]["end"]))] if len(det) else None
                report("decode step", win, d, max_lines=14)
    eng.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
