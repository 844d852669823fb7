"""CPU-side checks of the drop-in boundary: the C-ABI library builds, loads, exports every
symbol include/llmlb_b200.h declares, and refuses to run without a GPU (no CPU fallback)."""
import ctypes
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_functions():
    src = open(os.path.join(ROOT, "include", "llmlb_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(llmlb_[a-z0-9_]+)\s*\(", src)))


def test_header_declares_the_engine_and_kernel_entry_points():
    fns = header_functions()
    for must in ["llmlb_engine_create", "llmlb_engine_destroy", "llmlb_request_submit",
                 "llmlb_request_poll", "llmlb_request_cancel", "llmlb_engine_health",
                 "llmlb_engine_model_info", "llmlb_last_error", "llmlb_op_gemv", "llmlb_op_gemm",
                 "llmlb_op_decode_attention", "llmlb_op_prefill_attention_tc", "llmlb_op_sample"]:
        assert must in fns


def test_library_exports_every_declared_symbol(built_lib):
    lib = ctypes.CDLL(built_lib)
    missing = [f for f in header_functions() if not hasattr(lib, f)]
    assert not missing, missing


def test_ffi_prototypes_cover_header(built_lib):
    from llmlb_b200 import ffi
    assert sorted(ffi.PROTOTYPES) == header_functions()
    assert ffi.lib().llmlb_abi_version() == ffi.ABI_VERSION


def test_struct_sizes_match_c_layout(built_lib):
    """ctypes mirrors must have the C sizes (checked against a gcc-compiled probe)."""
    import subprocess
    import tempfile
    from llmlb_b200 import ffi
    probe = r'''
#include <stdio.h>
#include "llmlb_b200.h"
int main(void){printf("%zu %zu %zu %zu %zu %zu\n", sizeof(llmlb_model_config),
 sizeof(llmlb_engine_config), sizeof(llmlb_model_info), sizeof(llmlb_health),
 sizeof(llmlb_sampling), sizeof(llmlb_token_event));return 0;}'''
    with tempfile.TemporaryDirectory() as d:
        c = os.path.join(d, "p.c")
        open(c, "w").write(probe)
        exe = os.path.join(d, "p")
        subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), c, "-o", exe])
        sizes = [int(x) for x in subprocess.check_output([exe]).split()]
    mine = [ctypes.sizeof(t) for t in (ffi.ModelConfig, ffi.EngineConfig, ffi.ModelInfo,
                                       ffi.Health, ffi.Sampling, ffi.TokenEvent)]
    assert sizes == mine


def test_engine_create_fails_loudly_without_gpu(built_lib):
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from llmlb_b200 import ffi
    with pytest.raises(ffi.LlmlbError) as ei:
        ffi.Engine(ffi.LLAMA_TINY)
    assert ei.value.code == ffi.E_DEVICE
    assert "no CUDA device" in str(ei.value)


def test_argument_validation_without_gpu(built_lib):
    from llmlb_b200 import ffi
    L = ffi.lib()
    assert L.llmlb_engine_create(None, None) == ffi.E_INVALID_ARG
    assert L.llmlb_op_gemv(None, None, None, 0.0, None, 1, 8, 8, 0, 8, None) == ffi.E_INVALID_ARG
    assert L.llmlb_op_gemm(None, None, None, 1, 8, 8, 0, 8, 0, None) == ffi.E_INVALID_ARG
    assert b"bad argument" in L.llmlb_last_error()


def test_host_library_exports_every_declared_symbol():
    """include/llmlb_host.h (tokenizer + Anthropic translation) and include/llmlb_gateway.h (gateway rows a1.x,
    checkpoint readers, download contract) against libllmlb_host.so — in both directions: every declared function is
    exported, and the library exports nothing the headers do not declare — and both headers compile as plain C.
    The implementing .cpp files include the headers, so a signature that drifts fails the build itself."""
    import subprocess
    import tempfile
    from llmlb_b200 import build
    declared = {}
    for h in ("llmlb_host.h", "llmlb_gateway.h"):
        src = open(os.path.join(ROOT, "include", h)).read()
        src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
        declared[h] = sorted(set(re.findall(r"\b(llmlb_[a-z0-9_]+)\s*\(", src)))
    fns = declared["llmlb_host.h"]
    assert "llmlb_tok_encode" in fns and "llmlb_anthropic_stream_feed" in fns and len(fns) >= 20
    gw = declared["llmlb_gateway.h"]
    for must in ("llmlb_lm_select", "llmlb_lm_update_tps", "llmlb_lm_lease_begin", "llmlb_acc_feed", "llmlb_extract_usage", "llmlb_gate_try_begin",
                 "llmlb_classify_upstream_error", "llmlb_lb_error", "llmlb_frame", "llmlb_ckpt_open", "llmlb_dl_start"):
        assert must in gw
    assert not set(fns) & set(gw)
    path = build.build_host()
    lib = ctypes.CDLL(path)
    missing = [f for f in fns + gw if not hasattr(lib, f)]
    assert not missing, missing
    exported = {l.split()[-1] for l in subprocess.check_output(["nm", "-D", "--defined-only", path], text=True).splitlines() if " T llmlb_" in l}
    assert exported == set(fns) | set(gw), sorted(exported ^ (set(fns) | set(gw)))
    with tempfile.TemporaryDirectory() as d:
        c = os.path.join(d, "h.c")
        open(c, "w").write('#include "llmlb_host.h"\n#include "llmlb_gateway.h"\n#include "llmlb_b200.h"\n'
                           'void* (*probe)(void) = llmlb_tok_stream_create;\nvoid* (*probe2)(void) = llmlb_lm_create;\nint main(void){return 0;}\n')
        subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Werror", "-pedantic", "-c", "-I", os.path.join(ROOT, "include"), c, "-o", os.path.join(d, "h.o")])


def test_rust_ffi_crate_matches_the_header():
    """ffi/llmlb-b200-sys (source only: no cargo here): #[repr(C)] layouts, constants and the extern
    block against include/llmlb_b200.h, via gcc offsetof (tools/check_rust_layout.py)."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("check_rust_layout", os.path.join(ROOT, "tools", "check_rust_layout.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    assert mod.check() == []
