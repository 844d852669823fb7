"""The engine's launch plan, read without a GPU: tests/support/launch_plan_sweep.py runs the product library over the fake
CUDA runtime and logs every kernel launch for EVERY prefill width 1..2048 and decode batch width 1..128 of Llama-3-8B
(tp 1, 2, 4, 8) and Llama-3-70B (tp 8) shapes.  Checked on each launch:

  * co-residency: kernels whose CTAs wait for each other inside the grid (the in-kernel K-split of gemm_tc / gemm_tc2 parks
    partial tiles and spins on a per-tile counter) must fit the GPU in one wave — at most 148 CTAs at one CTA per SM; gemv_ks
    is held to the same bound.  A wider grid would hang the device; GPU tests only ever try a few widths.
  * hardware limits: <= 1024 threads per CTA, <= 227 KiB dynamic shared memory, cluster size <= 16 and grid divisible by it.
  * every launch with more than 48 KiB of dynamic shared memory was preceded by the opt-in for THAT kernel function (each
    template instantiation needs its own cudaFuncSetAttribute; a missing one only fails at the widths that pick it) — the
    fake runtime refuses the launch otherwise, like the driver.
  * every TMA descriptor the engine builds for these geometries passes the argument rules of cuTensorMapEncodeTiled (checked
    inside the fake runtime's stand-in: alignment, dims, strides, box dims, swizzle span); a refused descriptor fails engine
    creation here exactly as it would on the device.
"""
import collections
import os
import re
import subprocess
import sys

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import test_engine_host_logic_cpu as HL  # noqa: E402

SM_COUNT, MAX_SMEM = 148, 227 * 1024
MANGLED = {}


_PLANS = {}


def plan(tmp_path, model, tp):
    if (model, tp) not in _PLANS:
        _PLANS[(model, tp)] = _plan(tmp_path, model, tp)
    return _PLANS[(model, tp)]


def _plan(tmp_path, model, tp):
    log = str(tmp_path / ("launch_%s_tp%d.log" % (model, tp)))
    env = dict(os.environ, LD_PRELOAD=HL.build_fake(), FAKE_CUDART_LAUNCH_LOG=log)
    r = subprocess.run([sys.executable, os.path.join(HERE, "support", "launch_plan_sweep.py"), model, str(tp)], env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    ctx, out = "init", collections.defaultdict(list)                 # engine creation: weight generation, tables, warm-up
    for line in open(log):
        if line.startswith("###"):
            ctx = line[4:].strip()
            continue
        p = line.split()
        name = re.sub(r"^_ZN5llmlb\d+|^_Z\d+", "", p[0])
        MANGLED[name] = p[0]
        out[ctx].append((name, tuple(map(int, p[1:4])), tuple(map(int, p[4:7])), int(p[7]), tuple(map(int, p[8:11])), int(p[11])))
    return out


@pytest.mark.parametrize("model,tp", [("8b", 1), ("8b", 2), ("8b", 4), ("8b", 8), ("70b", 8)])
def test_every_width_of_the_launch_plan_respects_co_residency_and_hardware_limits(built_lib, tmp_path, model, tp):
    steps = plan(tmp_path, model, tp)
    assert len([k for k in steps if k.startswith("prefill")]) == 2048 and len([k for k in steps if k.startswith("decode")]) == 128
    assert len([k for k in steps if k.startswith("long")]) == 4                              # 3800-token contexts, batch 1 / 3 / 5 / 32
    assert len(steps["ctx131072"]) > 64 * 10                                                 # one 130 000-token prompt in 64 chunks + decode
    n = 0
    seen_ksplit_kernels = set()
    for ctx, launches in steps.items():
        assert launches, ctx
        for name, grid, block, smem, cluster, pdl in launches:
            n += 1
            ctas, threads, csize = grid[0] * grid[1] * grid[2], block[0] * block[1] * block[2], cluster[0] * cluster[1] * cluster[2]
            assert threads <= 1024 and smem <= MAX_SMEM, (ctx, name, block, smem)
            assert csize <= 16 and all(g % c == 0 for g, c in zip(grid, cluster)), (ctx, name, grid, cluster)
            if name.startswith(("gemm_tc_kernel", "gemm_tc2_kernel", "gemv_ks_kernel")):
                seen_ksplit_kernels.add(name.split("I")[0])
                assert ctas <= SM_COUNT, "%s: %s launches %d CTAs that wait for each other: more than one wave of %d SMs" % (ctx, name, ctas, SM_COUNT)
                if name.startswith("gemm_tc2_kernel"):
                    assert cluster == (2, 1, 1) and ctas % 2 == 0, (ctx, name, cluster)        # cta_group::2 pairs
    assert {"gemm_tc_kernel", "gemm_tc2_kernel", "gemv_ks_kernel"} <= seen_ksplit_kernels and n > 50000


@pytest.mark.skipif(__import__("shutil").which("cuobjdump") is None, reason="cuobjdump not on PATH")
def test_every_kernel_launched_as_a_programmatic_dependent_waits_for_its_predecessor(built_lib, tmp_path):
    """Launch plan x SASS: a kernel that the engine launches with the programmatic-stream-serialization attribute may start
    while its predecessor is still running, so it MUST execute griddepcontrol.wait (SASS: ACQBULK) before touching what the
    predecessor writes.  Every kernel name that appears with the attribute anywhere in the plans (all widths, tp 1 and 8) has
    to contain that instruction; the companion test tests/test_sass_pdl_cpu.py bounds what may be loaded ahead of it."""
    import glob
    pdl_kernels, plain_kernels = set(), set()
    for model, tp in (("8b", 1), ("8b", 8)):
        for launches in plan(tmp_path, model, tp).values():
            for name, grid, block, smem, cluster, pdl in launches:
                (pdl_kernels if pdl else plain_kernels).add(MANGLED[name])
    assert len(pdl_kernels) >= 10
    waits = set()
    for o in sorted(glob.glob(os.path.join(os.path.dirname(HERE), "llmlb_b200", "_build", "*.o"))):
        txt = subprocess.run(["cuobjdump", "-sass", o], capture_output=True, text=True).stdout
        for f in re.split(r"\n\s*Function : ", txt)[1:]:
            if "ACQBULK" in f:
                waits.add(f.split("\n", 1)[0].strip())
    # Reviewed exception: tp_reduce_norm_kernel has no dependency wait on purpose — it must be resident while its producer
    # GEMM is still pushing.  It orders itself through the exchange instead: it reads the residual row only after THIS rank's
    # own words / end-of-grid flag of the collective arrived, which proves the local GEMM finished, whose own dependency wait
    # covers everything before it (csrc/tp_exchange.cu; DESIGN.md section 5, "what went wrong" item 3 is the bug this fixed).
    ordered_by_exchange = {k for k in pdl_kernels if "tp_reduce_norm_kernel" in k}
    assert len(ordered_by_exchange) == 2
    missing = sorted(k for k in pdl_kernels - ordered_by_exchange if k not in waits)
    assert not missing, "launched as programmatic dependents without a griddepcontrol.wait: %s" % missing


def test_op_gemm_accepts_arbitrary_shapes_within_the_same_limits(built_lib, tmp_path):
    """The public kernel-level entry point takes any (tokens, n_out, k) with k % 8 == 0 — ragged last tiles, n_out that is not a
    multiple of the 128-row tile, K shorter than one 64-wide slab: 6000 random shapes, each accepted, each launch within one
    wave for the K-split kernels, with its shared-memory opt-in and legal TMA descriptors (checked by the fake runtime)."""
    log = str(tmp_path / "op.log")
    env = dict(os.environ, LD_PRELOAD=HL.build_fake(), FAKE_CUDART_LAUNCH_LOG=log)
    r = subprocess.run([sys.executable, os.path.join(HERE, "support", "op_gemm_sweep.py"), "6000", "1"], env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    calls = launches = 0
    for line in open(log):
        if line.startswith("###"):
            calls += 1
            ctx = line
            continue
        p = line.split()
        launches += 1
        ctas = int(p[1]) * int(p[2]) * int(p[3])
        assert "gemm_tc" in p[0] and ctas <= SM_COUNT and int(p[7]) <= MAX_SMEM, (ctx, line)
    assert calls > 5000 and launches >= calls


def test_every_kernel_level_entry_point_survives_random_arguments(built_lib, tmp_path):
    """Every llmlb_op_* entry point with random pointers (valid or NULL) and integers from {0, 1, odd, model-sized, 2^32 - 1}:
    25000 calls, each returns OK or a negative error code — never a crash.  Found on the first run: a dimension near 2^32
    wrapped llmlb_op_gemm's 32-bit tile count to zero and the launch planner divided by it (SIGFPE); dimensions are
    bounded at the entry point now.  Launches whose configuration the device would refuse come back as errors through
    the fake runtime's cudaGetLastError, like on the GPU."""
    env = dict(os.environ, LD_PRELOAD=HL.build_fake(), FAKE_CUDART_LAUNCH_LOG=str(tmp_path / "opf.log"))
    for seed in ("1", "2"):
        r = subprocess.run([sys.executable, os.path.join(HERE, "support", "op_fuzz.py"), "12500", seed], env=env, capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, "seed %s rc %d\n%s" % (seed, r.returncode, r.stderr[-1500:])
        assert "calls 12500" in r.stdout and "(0, " in r.stdout and "(-1, " in r.stdout, r.stdout[-300:]


def test_engine_create_with_random_configurations_refuses_or_serves(built_lib, tmp_path):
    """llmlb_engine_create from a valid configuration with up to three fields knocked to odd values (zero, not a multiple of
    the page, more ranks than kv heads, a 2^20-page pool, NaN rope base, a foreign ABI version ...), 3000 times: every call
    either returns an error code and no engine, or an engine that then serves a request to completion and is destroyed."""
    env = dict(os.environ, LD_PRELOAD=HL.build_fake())
    r = subprocess.run([sys.executable, os.path.join(HERE, "support", "create_fuzz.py"), "3000", "1"], env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-500:] + r.stderr[-2500:]
    n_ok, n_err = [int(x) for x in re.search(r"engines (\d+) refused (\d+)", r.stdout).groups()]
    assert n_ok > 1000 and n_err > 500
