"""Tensor-parallel parity on real GPUs (SURVEY.md §8e, row a2.13): launches tools/tp_check.py under
torchrun for every world size the box offers (2, 4, 8).  Each run compares the sharded engine with the
CPU oracle AND with a tp=1 engine of the same model, for both exchange protocols (decode push of
{value, epoch} pairs; reduce-scatter + all-gather), the fused and the unfused producer / consumer
kernels, CUDA-graph decode and packed prefill.  Skipped on 1-GPU boxes
(the driver's scaling run carries its own `parity` record from bench.py there)."""
import os
import socket
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _n_gpus():
    try:
        import torch
        return torch.cuda.device_count() if torch.cuda.is_available() else 0
    except Exception:
        return 0


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


@pytest.mark.gpu
@pytest.mark.parametrize("geom", ["tiny", "odd", "8b4"])
@pytest.mark.parametrize("world", [2, 4, 8])
def test_tensor_parallel_matches_oracle_and_single_gpu(built_lib, world, geom):
    if _n_gpus() < world:
        pytest.skip("needs %d GPUs" % world)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world),
           "--master-addr", "127.0.0.1", "--master-port", str(_free_port()),
           os.path.join(ROOT, "tools", "tp_check.py"), "--geom", geom]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-3000:] + "\n" + r.stderr[-3000:]
    assert "ranks identical: True" in r.stdout
