"""Chunks given per video, without a GPU: the pointer-table fields of the step argument blocks sit where the header puts
them, the pointer pooling entry point and both step entry points refuse inconsistent arguments before any CUDA call,
and `split_videos` cuts whole videos into chunk views."""
import ctypes as C
import os
import subprocess

import pytest
import torch

from infinite_video_b200 import _capi, build
from infinite_video_b200.video import split_videos

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FAKE = C.c_void_p(0x10000)           # aligned, never dereferenced: every call below fails its argument checks


@pytest.fixture(scope="module")
def lib():
    build.build()
    return _capi.lib()


def test_table_fields_match_c_layout(tmp_path):
    prog = tmp_path / "off.c"
    prog.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "infltm.h"\n'
                    'int main(){printf("%zu %zu %zu %zu\\n", offsetof(ltm_rect_step_args, k_ptrs),'
                    ' sizeof(ltm_rect_step_args), offsetof(ltm_overlap, next_ptrs), sizeof(ltm_overlap));return 0;}\n')
    exe = tmp_path / "off"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(prog), "-o", str(exe)])
    got = [int(x) for x in subprocess.check_output([str(exe)], text=True).split()]
    assert got == [_capi.RectStepArgs.k_ptrs.offset, C.sizeof(_capi.RectStepArgs),
                   _capi.Overlap.next_ptrs.offset, C.sizeof(_capi.Overlap)]
    # appended after the chunk storage fields: a zero-initialised block means "no table"
    assert _capi.RectStepArgs.k_ptrs.offset > _capi.RectStepArgs.k_dtype.offset
    assert _capi.Overlap.next_ptrs.offset > _capi.Overlap.next_dtype.offset
    assert _capi.RectStepArgs().k_ptrs is None and _capi.Overlap().next_ptrs is None


def test_zero_block_keeps_todays_refusals(lib):
    # no table: the step still asks for its usual pointers, and says nothing about tables
    a, o = _capi.RectStepArgs(), _capi.Overlap()
    assert lib.ltm_rect_step(C.byref(a), None, None, None, None, None, None) < 0
    assert b"rect_step: null pointer" in lib.ltm_last_error()
    assert lib.ltm_rect_step_overlap(C.byref(a), C.byref(o), None, None, None, None) < 0
    assert b"rect_step_overlap: null pointer" in lib.ltm_last_error()


@pytest.mark.parametrize("args, msg", [
    ((None, 0, FAKE, FAKE, 2, 8, 32, 768, 1, 4, 0, None), b"null pointer"),
    ((FAKE, 0, FAKE, None, 2, 8, 32, 768, 1, 4, 0, None), b"null pointer"),
    ((FAKE, 0, None, FAKE, 2, 8, 32, 768, 1, 4, 0, None), b"null pointer"),
    ((FAKE, 0, FAKE, FAKE, 0, 8, 32, 768, 1, 4, 0, None), b"bad shape"),
    ((FAKE, 0, FAKE, FAKE, 2, 8, 32, 768, 1, 17, 0, None), b"bad shape"),
    ((FAKE, 3, FAKE, FAKE, 2, 8, 32, 768, 1, 4, 0, None), b"dtype=3"),
    ((FAKE, 1, FAKE, FAKE, 2, 8, 32, 772, 1, 4, 0, None), b"multiple of 8"),
    ((FAKE, 0, FAKE, FAKE, 2, 8, 32, 770, 1, 4, 0, None), b"multiple of 4"),
    ((FAKE, 0, FAKE, FAKE, 2, 8, 32, 768, 0, 4, 0, None), b"splits"),
    ((FAKE, 0, FAKE, FAKE, 2, 8, 32, 768, 33, 4, 0, None), b"splits"),
    ((FAKE, 0, FAKE, FAKE, 2, 8, 32, 768, 1, 4, -1, None), b"max_ctas"),
    ((C.c_void_p(0x10004), 0, FAKE, FAKE, 2, 8, 32, 768, 1, 4, 0, None), b"aligned"),
    ((FAKE, 0, C.c_void_p(0x10008), FAKE, 2, 8, 32, 768, 1, 4, 0, None), b"aligned"),
])
def test_pool_mean_ptrs_argument_errors(lib, args, msg):
    rc = lib.ltm_pool_mean_ptrs(*args)
    assert rc < 0
    err = lib.ltm_last_error()
    assert b"pool_mean_ptrs" in err and msg in err


def _step_args(table=True, lengths=True, binned=0):
    a = _capi.RectStepArgs()
    a.Bv, a.L, a.T, a.e, a.N, a.Q, a.H, a.d = 2, 8, 32, 768, 64, 32, 12, 64
    a.binned = binned
    a.k_ptrs = FAKE if table else None
    a.lengths, a.frame_offs = (FAKE, FAKE) if lengths else (None, None)
    return a


@pytest.mark.parametrize("chunk, lengths, binned, msg", [
    (FAKE, True, 0, b"k_ptrs and a chunk pointer are both set"),
    (None, False, 0, b"k_ptrs needs per-video lengths"),
    (None, True, 1, b"not pooled per bin"),
])
def test_step_refuses_inconsistent_table(lib, chunk, lengths, binned, msg):
    a = _step_args(lengths=lengths, binned=binned)
    rc = lib.ltm_rect_step(C.byref(a), chunk, FAKE, None, None, FAKE, None)
    err = lib.ltm_last_error()
    assert rc < 0 and b"rect_step:" in err and msg in err
    if chunk is None:
        o = _capi.Overlap()
        o.ev_fork = o.ev_join = FAKE
        rc = lib.ltm_rect_step_overlap(C.byref(a), C.byref(o), FAKE, None, None, FAKE)
        err = lib.ltm_last_error()
        assert rc < 0 and b"rect_step_overlap:" in err and msg in err


@pytest.mark.parametrize("k_next, lengths, binned, msg", [
    (FAKE, True, 0, b"next_ptrs and a chunk pointer are both set"),
    (None, False, 0, b"next_ptrs needs per-video lengths"),
    (None, True, 1, b"not pooled per bin"),
])
def test_overlap_refuses_inconsistent_next_table(lib, k_next, lengths, binned, msg):
    a = _step_args(table=False, lengths=False)
    o = _capi.Overlap()
    o.ev_fork = o.ev_join = FAKE
    o.next_ptrs, o.k_next, o.xpart_next, o.ev_fork_pool, o.ev_pooled_next = FAKE, k_next, FAKE, FAKE, FAKE
    if lengths:
        o.next_lengths = o.next_offs = FAKE
    o.next_binned = binned
    rc = lib.ltm_rect_step_overlap(C.byref(a), C.byref(o), FAKE, None, None, FAKE)
    err = lib.ltm_last_error()
    assert rc < 0 and b"rect_step_overlap:" in err and msg in err


def test_split_videos_chunks_are_views():
    T, e, L = 4, 8, 3
    videos = [torch.arange(F * T * e, dtype=torch.float32).view(F * T, e) for F in (8, 2, 9, 5)]
    chunks = split_videos(videos, L, T)
    assert len(chunks) == 3                                       # ceil(9 / 3)
    lens = [[0 if x is None else x.shape[0] // T for x in ch] for ch in chunks]
    # frames per chunk: min(L, F - c*L) while the video lasts, then None
    assert lens == [[3, 2, 3, 3], [3, 0, 3, 2], [2, 0, 3, 0]]
    for c, ch in enumerate(chunks):
        for v, x in enumerate(ch):
            if x is None:
                continue
            assert x.untyped_storage().data_ptr() == videos[v].untyped_storage().data_ptr()
            assert x.data_ptr() == videos[v].data_ptr() + c * L * T * e * 4
            assert x.stride() == (e, 1)
            assert torch.equal(x, videos[v][c * L * T:c * L * T + x.shape[0]])


def test_split_videos_refuses_one_frame_tail_and_bad_shapes():
    T, e = 4, 8
    with pytest.raises(ValueError, match="video 1 has 7 frames"):
        split_videos([torch.zeros(6 * T, e), torch.zeros(7 * T, e)], 3, T)
    with pytest.raises(ValueError, match="video 0"):
        split_videos([torch.zeros(6 * T + 1, e)], 3, T)
    with pytest.raises(ValueError, match="video 0"):
        split_videos([torch.zeros(6 * T)], 3, T)
    with pytest.raises(ValueError, match="frames_per_chunk"):
        split_videos([torch.zeros(6 * T, e)], 1, T)
    assert split_videos([torch.zeros(6 * T, e)], 3, T)[1][0].shape == (3 * T, e)
