"""-m gpu: bench.py --dump-outputs writes what its last timed step returned — the token events of the request of step
K-1 — and those are the tokens the engine gives any caller for that seeded prompt."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from llmlb_b200 import ffi

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FIELDS = ["completion_tokens", "finish_reason", "index", "prompt_tokens", "token_id"]
PROMPT, GEN = 512, 128


def test_dump_outputs_are_the_last_timed_step(built_lib, tmp_path):
    steps = 2
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--model", "tiny", "--steps", str(steps), "--warmup", "1",
                          "--streams", "0", "--no-parity", "--no-ref-shape", "--no-micro", "--no-cpu-baseline",
                          "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-3000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1 and json.loads(lines[0])["steps"] == steps
    assert sorted(os.listdir(tmp_path)) == [f + ".npy" for f in FIELDS]
    got = {f: np.load(tmp_path / (f + ".npy")) for f in FIELDS}
    for a in got.values():
        assert a.dtype == np.float64 and a.shape == (1, GEN)
    prompt = np.random.RandomState(1000 + steps - 1).randint(0, ffi.LLAMA_TINY["vocab"], PROMPT).tolist()   # bench.make_prompt
    with ffi.Engine(ffi.LLAMA_TINY, max_seqs=4, max_ctx=1024, seed=0) as eng:
        toks, _ = eng.generate(prompt, GEN, ignore_eos=True)
    assert got["token_id"][0].astype(np.int64).tolist() == toks
    assert got["index"][0].tolist() == list(range(GEN))
    assert got["completion_tokens"][0].tolist() == list(range(1, GEN + 1))
    assert set(got["prompt_tokens"][0].tolist()) == {PROMPT}
    assert got["finish_reason"][0, -1] == ffi.FINISH_LENGTH and not got["finish_reason"][0, :-1].any()
