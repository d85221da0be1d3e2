"""The C-ABI library loads without a GPU, exports every symbol include/infltm.h declares, the ctypes
structures match the C layout, and the error convention (rc<0 + ltm_last_error) works -- no compute calls."""
import ctypes as C
import os
import re
import subprocess

import pytest

from infinite_video_b200 import _capi, build

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "infltm.h")


@pytest.fixture(scope="module")
def lib():
    build.build()
    return _capi.lib()


def _declared():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(ltm_[a-z0-9_]+)\s*\(", src)))


def test_every_declared_symbol_is_exported_and_bound(lib):
    names = _declared()
    assert len(names) >= 18
    out = subprocess.check_output(["nm", "-D", "--defined-only", _capi.LIB_PATH], text=True)
    exported = set(re.findall(r" T (ltm_[a-z0-9_]+)", out))
    assert set(names) <= exported, sorted(set(names) - exported)
    assert set(names) == set(_capi.EXPORTED)
    for n in names:
        assert getattr(lib, n) is not None


def test_version_and_error_convention(lib):
    assert lib.ltm_version() == 100
    rc = lib.ltm_pool_mean(None, None, 1, 1, 1, 4, 1, None)      # argument validation precedes any CUDA call
    assert rc < 0
    assert b"pool_mean" in lib.ltm_last_error()
    rc = lib.ltm_resample(None, 1, 127, 1, None, None, None, 0, None, None, None, None, None, 1, 512, None)
    assert rc < 0 and b"resample" in lib.ltm_last_error()
    g = _capi.GemmArgs()
    assert lib.ltm_gemm(C.byref(g), None) < 0
    # entry points added with the tensor-core attention / overlapped step: validation before any CUDA call
    rc = lib.ltm_cont_attn_rect_tc(None, None, None, 1536, None, None, 0.0, 0.0, None, None, None, None, None,
                                   1, 32, 256, 12, 64, None)
    assert rc < 0 and b"cont_attn_rect_tc" in lib.ltm_last_error()
    assert lib.ltm_attn_tc_supported(256, 64) == 1 and lib.ltm_attn_tc_supported(64, 64) == 1
    assert lib.ltm_attn_tc_supported(512, 64) == 0 and lib.ltm_attn_tc_split_supported(512, 64) == 1
    assert lib.ltm_attn_tc_split_supported(256, 64) == 0 and lib.ltm_attn_tc_split_workspace_floats(2, 40, 12) == 2 * 12 * 2 * 2 * 68 * 32
    assert lib.ltm_attn_tc_supported(256, 128) == 0
    a, o = _capi.RectStepArgs(), _capi.Overlap()
    rc = lib.ltm_rect_step_overlap(C.byref(a), C.byref(o), None, None, None, None)
    assert rc < 0 and b"rect_step_overlap" in lib.ltm_last_error()
    rc = lib.ltm_sticky_hist_gauss(None, None, None, None, 1, 384, 8, None)
    assert rc < 0 and b"sticky_hist_gauss" in lib.ltm_last_error()


def test_ctypes_structs_match_c_layout(tmp_path):
    prog = tmp_path / "sz.c"
    prog.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "infltm.h"\n'
                    'int main(){printf("%zu %zu %zu %zu %zu %zu %zu %zu %zu %zu %zu\\n", sizeof(ltm_gemm_args), offsetof(ltm_gemm_args, C),'
                    ' offsetof(ltm_gemm_args, impl), sizeof(ltm_rect_step_args), offsetof(ltm_rect_step_args, W_out),'
                    ' offsetof(ltm_rect_step_args, ctx_dev), offsetof(ltm_gemm_args, round_tf32),'
                    ' offsetof(ltm_rect_step_args, X), offsetof(ltm_rect_step_args, c_none),'
                    ' offsetof(ltm_rect_step_args, attn_part), offsetof(ltm_rect_step_args, hist_keep));return 0;}\n')
    exe = tmp_path / "sz"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(prog), "-o", str(exe)])
    got = [int(x) for x in subprocess.check_output([str(exe)], text=True).split()]
    want = [C.sizeof(_capi.GemmArgs), _capi.GemmArgs.C.offset, _capi.GemmArgs.impl.offset,
            C.sizeof(_capi.RectStepArgs), _capi.RectStepArgs.W_out.offset, _capi.RectStepArgs.ctx_dev.offset,
            _capi.GemmArgs.round_tf32.offset, _capi.RectStepArgs.X.offset, _capi.RectStepArgs.c_none.offset,
            _capi.RectStepArgs.attn_part.offset, _capi.RectStepArgs.hist_keep.offset]
    assert got == want


def test_product_refuses_cpu_tensors():
    import torch
    from infinite_video_b200 import ops
    with pytest.raises(ValueError):
        ops.pool_mean(torch.zeros(1, 2, 4, 8))
    from infinite_video_b200.batched import BatchedRectLTM
    with pytest.raises(ValueError):
        BatchedRectLTM(64, .75, torch.zeros(768, 768), None, torch.zeros(768, 768), None, device="cpu")
