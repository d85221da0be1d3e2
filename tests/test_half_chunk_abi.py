"""16-bit chunks at the C ABI, without a GPU: the chunk-storage fields of the step argument blocks sit where the header
puts them, and bad storage codes / widths are refused before any CUDA call."""
import ctypes as C
import os
import subprocess

import pytest

from infinite_video_b200 import _capi, build

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    build.build()
    return _capi.lib()


def test_dtype_fields_match_c_layout(tmp_path):
    prog = tmp_path / "off.c"
    prog.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "infltm.h"\n'
                    'int main(){printf("%zu %zu %zu %zu\\n", offsetof(ltm_rect_step_args, k_dtype),'
                    ' sizeof(ltm_rect_step_args), offsetof(ltm_overlap, next_dtype), sizeof(ltm_overlap));return 0;}\n')
    exe = tmp_path / "off"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(prog), "-o", str(exe)])
    got = [int(x) for x in subprocess.check_output([str(exe)], text=True).split()]
    assert got == [_capi.RectStepArgs.k_dtype.offset, C.sizeof(_capi.RectStepArgs),
                   _capi.Overlap.next_dtype.offset, C.sizeof(_capi.Overlap)]
    # appended last: a zero-initialised block keeps meaning fp32
    assert _capi.RectStepArgs.k_dtype.offset > _capi.RectStepArgs.hist_keep.offset
    assert _capi.Overlap.next_dtype.offset > _capi.Overlap.next_splits.offset
    assert _capi.RectStepArgs().k_dtype == 0 and _capi.Overlap().next_dtype == 0


FAKE = C.c_void_p(0x10000)           # aligned, never dereferenced: every call below fails its argument checks


@pytest.mark.parametrize("args, msg", [
    ((None, 0, FAKE, 1, 1, 1, 768, 1, 0, None), b"null pointer"),
    ((FAKE, 0, FAKE, 1, 1, 1, 772, 1, 0, None), b"multiple of 8"),
    ((FAKE, 1, FAKE, 0, 1, 1, 768, 1, 0, None), b"bad shape"),
    ((FAKE, 1, FAKE, 1, 1, 4, 768, 5, 0, None), b"splits"),
    ((FAKE, 1, FAKE, 1, 1, 4, 768, 1, -1, None), b"max_ctas"),
    ((C.c_void_p(0x10008), 1, FAKE, 1, 1, 4, 768, 1, 0, None), b"aligned"),
])
def test_pool_mean_16_grid_argument_errors(lib, args, msg):
    rc = lib.ltm_pool_mean_16_grid(*args)
    assert rc < 0
    err = lib.ltm_last_error()
    assert b"pool_mean_16_grid" in err and msg in err


def _step_args(k_dtype, e=768, binned=0):
    a = _capi.RectStepArgs()
    a.Bv, a.L, a.T, a.e, a.N, a.Q, a.H, a.d = 1, 8, 32, e, 64, 32, 12, 64
    a.k_dtype, a.binned = k_dtype, binned
    a.k_dev = a.q_dev = a.ctx_dev = FAKE
    return a


@pytest.mark.parametrize("k_dtype, e, binned, msg", [
    (3, 768, 0, b"k_dtype=3"),
    (-1, 768, 0, b"k_dtype=-1"),
    (1, 772, 0, b"e % 8"),
    (2, 772, 0, b"e % 8"),
    (1, 768, 1, b"per bin"),
])
def test_step_entry_points_refuse_bad_chunk_storage(lib, k_dtype, e, binned, msg):
    a = _step_args(k_dtype, e, binned)
    rc = lib.ltm_rect_step(C.byref(a), FAKE, FAKE, None, None, FAKE, None)
    assert rc < 0 and b"rect_step:" in lib.ltm_last_error() and msg in lib.ltm_last_error()
    rc = lib.ltm_rect_step_host(C.byref(a), FAKE, FAKE, None, None, FAKE, None)
    assert rc < 0 and b"rect_step_host" in lib.ltm_last_error() and msg in lib.ltm_last_error()
    o = _capi.Overlap()
    o.ev_fork = o.ev_join = FAKE
    rc = lib.ltm_rect_step_overlap(C.byref(a), C.byref(o), FAKE, None, None, FAKE)
    assert rc < 0 and b"rect_step_overlap" in lib.ltm_last_error() and msg in lib.ltm_last_error()


@pytest.mark.parametrize("next_dtype, e, next_binned, msg", [
    (5, 768, 0, b"next_dtype=5"),
    (1, 772, 0, b"e % 8"),
    (2, 768, 1, b"per bin"),
])
def test_overlap_refuses_bad_next_chunk_storage(lib, next_dtype, e, next_binned, msg):
    a = _step_args(0, e)
    o = _capi.Overlap()
    o.ev_fork = o.ev_join = FAKE
    o.k_next, o.xpart_next, o.ev_fork_pool, o.ev_pooled_next = FAKE, FAKE, FAKE, FAKE
    o.next_dtype, o.next_binned = next_dtype, next_binned
    rc = lib.ltm_rect_step_overlap(C.byref(a), C.byref(o), FAKE, None, None, FAKE)
    assert rc < 0 and b"rect_step_overlap" in lib.ltm_last_error() and msg in lib.ltm_last_error()
