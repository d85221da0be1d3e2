"""Host side of the cross-attention branch's encoder mask, no GPU: the shapes and dtypes `encoder_mask_rows` accepts
become one contiguous float32 row per video, and everything the softmax kernels would read out of bounds or from the
wrong video (a broadcast batch, per-query or per-head masks, a wrong L*T) is refused with ValueError."""
import pytest
import torch

from infinite_video_b200.cross_attention import CrossAttentionLTM, encoder_mask_rows

B, Q, H, LT = 3, 4, 2, 24


def _rows():
    g = torch.Generator().manual_seed(5)
    m = torch.zeros(B, LT)
    m[torch.rand(B, LT, generator=g) < .4] = -10000.0
    m[1] = torch.finfo(torch.float32).min
    return m


@pytest.mark.parametrize("dtype", [torch.float32, torch.float16, torch.bfloat16, torch.float64])
@pytest.mark.parametrize("shape", [(B, LT), (B, 1, LT), (B, 1, 1, LT)])
def test_accepted_shapes_give_one_float32_row_per_video(shape, dtype):
    rows = _rows()
    got = encoder_mask_rows(rows.to(dtype).reshape(shape), B, LT)
    assert got.shape == (B, LT) and got.dtype == torch.float32 and got.is_contiguous()
    assert torch.equal(got, rows.to(dtype).float())        # fp16 turns finfo(fp32).min into -inf: still a zero weight


def test_non_contiguous_mask_is_copied():
    rows = _rows()
    got = encoder_mask_rows(rows.t().contiguous().t().reshape(B, 1, 1, LT), B, LT)
    assert got.is_contiguous() and torch.equal(got, rows)


def test_float32_row_mask_is_passed_through():
    rows = _rows()
    assert encoder_mask_rows(rows, B, LT).data_ptr() == rows.data_ptr()
    assert encoder_mask_rows(None, B, LT) is None


@pytest.mark.parametrize("shape", [
    (1, 1, 1, LT),          # one mask broadcast over the batch: reshaped to [B, -1] it would send videos past its end
    (1, LT),
    (B, 1, Q, LT),          # per query: reshaped to [B, Q*LT] video v would use video 0's row v
    (B, Q, LT),
    (B, H, 1, LT),          # per head
    (B, H, Q, LT),
    (B, 1, 1, LT - 4),      # wrong L*T
    (B, 1, 1, LT + 4),
    (B, LT, 1),
    (B + 1, 1, 1, LT),
    (B * LT,),
    (B, 1, 1, 1, LT),
])
def test_rejected_shapes(shape):
    with pytest.raises(ValueError, match="encoder_attention_mask"):
        encoder_mask_rows(torch.zeros(shape), B, LT)


@pytest.mark.parametrize("dtype", [torch.bool, torch.int64, torch.int32, torch.uint8])
def test_rejected_dtypes(dtype):
    with pytest.raises(ValueError, match="float"):
        encoder_mask_rows(torch.zeros(B, 1, 1, LT, dtype=dtype), B, LT)


def test_batch_of_one_is_its_own_batch():
    m = torch.zeros(1, 1, 1, LT)
    assert encoder_mask_rows(m, 1, LT).shape == (1, LT)


def test_mask_on_another_device_is_refused():
    with pytest.raises(ValueError, match="is on cpu"):
        encoder_mask_rows(torch.zeros(B, LT), B, LT, device="meta")
    assert encoder_mask_rows(torch.zeros(B, LT), B, LT, device="cpu").shape == (B, LT)


def test_short_term_validates_the_mask_before_anything_else():
    """`short_term` refuses a malformed mask before it reaches any library call (on CPU tensors the first library
    call would raise a different error: the product refuses CPU tensors)."""
    torch.manual_seed(0)
    m = CrossAttentionLTM(torch.nn.Linear(32, 32), torch.nn.Linear(32, 32), torch.nn.Linear(32, 32), .5, 16, .75,
                          n_heads=H, tokens_per_frame=8)
    q, enc = torch.zeros(B, Q, 32), torch.zeros(B, LT, 32)
    for bad in (torch.zeros(1, 1, 1, LT), torch.zeros(B, 1, Q, LT), torch.zeros(B, 1, 1, LT // 2)):
        with pytest.raises(ValueError, match="encoder_attention_mask"):
            m.short_term(q, enc, bad)
    with pytest.raises(ValueError, match="CUDA"):
        m.short_term(q, enc, torch.zeros(B, 1, 1, LT))
