"""Random arguments into every kernel-level entry point (llmlb_op_*) on the fake CUDA runtime: pointers are valid device
allocations or NULL, integers come from {0, 1, small, odd, the model's, huge}.  Nothing executes; what is tested is the HOST
side of each entry point: every call returns (OK or a negative error code) — no crash, no division by zero, no launch the
fake runtime refuses for its shape (block > 1024 threads, shared memory without opt-in, broken cluster).
usage: op_fuzz.py <calls> <seed>"""
import ctypes as C
import os
import random
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from llmlb_b200 import ffi  # noqa: E402

L = ffi.lib()
cu = C.CDLL("libcudart.so.12")
cu.cudaMalloc.argtypes = [C.POINTER(C.c_void_p), C.c_size_t]


def dmalloc(n):
    p = C.c_void_p()
    assert cu.cudaMalloc(C.byref(p), n) == 0
    return p


BIG = [dmalloc(1 << 32) for _ in range(6)]             # address space only
rs = random.Random(int(sys.argv[2]))
INTS = [0, 1, 2, 3, 4, 5, 7, 8, 16, 31, 32, 63, 64, 65, 127, 128, 129, 255, 256, 512, 1000, 1024, 2048, 4096, 6144, 14336, 128256, 1 << 20, (1 << 31) - 1, (1 << 32) - 1]


def ptr():
    return rs.choice(BIG) if rs.random() < 0.93 else None


def u():
    return rs.choice(INTS)


def f():
    return rs.choice([0.0, 1e-5, 1.0, -1.0, 5e5, float("inf"), float("nan")])


calls = crashes = 0
hist = {}
for _ in range(int(sys.argv[1])):
    op = rs.randrange(11)
    if op == 0:
        rc = L.llmlb_op_embed(ptr(), ptr(), ptr(), u(), u(), u(), None)
    elif op == 1:
        rc = L.llmlb_op_rmsnorm(ptr(), ptr(), ptr(), u(), u(), f(), None)
    elif op == 2:
        rc = L.llmlb_op_gemv(ptr(), ptr(), ptr(), f(), ptr(), u(), u(), u(), rs.randrange(6), u(), None)
    elif op == 3:
        rc = L.llmlb_op_gemm(ptr(), ptr(), ptr(), u(), u(), u(), rs.randrange(6), u(), rs.randrange(3), None)
    elif op == 4:
        rc = L.llmlb_op_rope_table(ptr(), u(), f(), None)
    elif op == 5:
        rc = L.llmlb_op_rope_append(ptr(), ptr(), ptr(), ptr(), ptr(), ptr(), u(), u(), u(), None)
    elif op == 6:
        rc = L.llmlb_op_prefill_attention_tc(ptr(), u(), ptr(), ptr(), u(), ptr(), u(), ptr(), u(), ptr(), u(), u(), None)
    elif op == 7:
        L.llmlb_op_decode_attention_ws(u(), u(), u())
        rc = L.llmlb_op_decode_attention(ptr(), ptr(), ptr(), ptr(), u(), ptr(), ptr(), u(), ptr(), u(), u(), ptr(), u(), u(), ptr(), None)
    elif op == 8:
        rc = L.llmlb_op_sample(ptr(), u(), u(), ptr(), ptr(), ptr(), ptr(), ptr(), ptr(), None)
    elif op == 9:
        rc = L.llmlb_op_synth_bf16(ptr(), u(), u(), u(), u(), u(), u(), rs.randrange(40), f(), None)
    else:
        rc = L.llmlb_op_allreduce(None, ptr(), u(), None)
    calls += 1
    hist[rc] = hist.get(rc, 0) + 1
    assert rc <= 0, (op, rc)
print("calls", calls, "return codes", sorted(hist.items()))
