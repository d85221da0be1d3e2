"""Host side of ragged batches (per-video chunk lengths), no GPU: the table bank slices back to the per-length tables
bit for bit, the new C-ABI fields sit where the header puts them, and malformed lengths are refused."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
import torch

from infinite_video_b200 import _capi, tables
from infinite_video_b200.batched import _as_lengths

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

LENGTHS = (2, 3, 7, 8, 30, 255, 256)


@pytest.mark.parametrize("spacing", ["linear", "log"])
@pytest.mark.parametrize("tau", [.5, .75])
@pytest.mark.parametrize("N", [64, 100, 256, 512])
def test_bank_entries_equal_rect_tables(N, tau, spacing):
    bank = tables.RectBank(256, N, tau, spacing=spacing)
    assert bank.fill(LENGTHS) == list(LENGTHS)
    assert bank.fill(LENGTHS) == []                                   # filled once
    for L in LENGTHS:
        t = tables.rect_tables(L, N, tau, spacing=spacing)
        got = bank.entry(L)
        for g, w in zip(got[:6], (t.seg_ptr0, t.seg_mem0, t.g0, t.seg_ptr1, t.seg_mem1, t.g1)):
            assert g.dtype == w.dtype and np.array_equal(g, w)
        assert got[6] == t.jf
        # the absolute offsets of an entry stay inside its fixed slot of the concatenated member lists
        assert bank.seg_ptr0[L][0] == bank.mem0_off(L) and bank.seg_ptr0[L][-1] <= bank.mem0_off(L + 1)
        assert bank.seg_ptr1[L][0] == bank.mem1_off(L) and bank.seg_ptr1[L][-1] <= bank.mem1_off(L + 1)


def test_bank_refuses_lengths_out_of_range():
    bank = tables.RectBank(16, 64, .75)
    for bad in (1, 17, -2):
        with pytest.raises(ValueError):
            bank.fill([bad])
    assert bank.fill([0, 16]) == [16]                                 # 0 = idle: no tables


def test_lengths_validation():
    assert _as_lengths([0, 2, 16], 3, 16) == (0, 2, 16)
    assert _as_lengths(torch.tensor([5, 0]), 2, 8) == (5, 0)
    for bad in ([1, 4], [4, 9], [-1, 4], [4], [4, 4, 4], [2.5, 4]):
        with pytest.raises(ValueError):
            _as_lengths(bad, 2, 8)
    with pytest.raises(ValueError):
        _as_lengths(torch.tensor([4.0, 4.0]), 2, 8)


def test_ragged_struct_fields_match_c_layout(tmp_path):
    fields = {"ltm_rect_step_args": (_capi.RectStepArgs, ["gemm_ctas", "lengths", "frame_offs", "frames", "n_idle",
                                                          "bank_seg_ptr0", "bank_seg_mem0", "bank_g0", "bank_seg_ptr1",
                                                          "bank_seg_mem1", "bank_g1", "hist_keep"]),
              "ltm_overlap": (_capi.Overlap, ["next_binned", "next_lengths", "next_offs", "next_frames",
                                              "next_splits"])}
    lines, want = [], []
    for st, (cls, names) in fields.items():
        lines.append(f'printf("%zu\\n", sizeof({st}));')
        want.append(C.sizeof(cls))
        for n in names:
            lines.append(f'printf("%zu\\n", offsetof({st}, {n}));')
            want.append(getattr(cls, n).offset)
    prog = tmp_path / "ragged.c"
    prog.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "infltm.h"\nint main(){' + "".join(lines) +
                    "return 0;}\n")
    exe = tmp_path / "ragged"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(prog), "-o", str(exe)])
    got = [int(x) for x in subprocess.check_output([str(exe)], text=True).split()]
    assert got == want


def test_ragged_pool_validates_before_any_cuda_call():
    from infinite_video_b200 import build
    build.build()
    lib = _capi.lib()
    assert lib.ltm_pool_mean_ragged(None, 0, None, None, 1, 2, 32, 768, 1, 2, 0, None) < 0
    assert b"pool_mean_ragged" in lib.ltm_last_error()
