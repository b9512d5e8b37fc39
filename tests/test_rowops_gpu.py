"""Patchify / attention kernels through the C ABI vs fp32 PyTorch on the same inputs (the LayerNorm
forward is tested in test_train_rowops_gpu.py)."""
import math

import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("B,C,S,p", [(2, 3, 224, 16), (3, 3, 32, 16), (1, 3, 384, 16), (2, 1, 64, 8)])
def test_patchify(vitk, B, C, S, p):
    x = torch.randn(B, C, S, S, device="cuda")
    out = vitk.ops.patchify(x, p)
    g = S // p
    ref = x.reshape(B, C, g, p, g, p).permute(0, 2, 4, 1, 3, 5).reshape(B * g * g, C * p * p)
    assert torch.equal(out, ref.bfloat16())  # pure gather + round-to-nearest: bit exact


@pytest.fixture(params=[1, 2, 3, 4], ids=["flash", "tcgen05", "tcgen05-unpipelined", "tcgen05-long-seq"])
def attn_impl(request, vitk):
    vitk._lib.set_attention_impl(request.param)
    yield request.param
    vitk._lib.set_attention_impl(0)


def _attn_ref(qkv, B, N, H):
    D = qkv.shape[-1] // 3
    hd = D // H
    q, k, v = qkv.float().reshape(B, N, 3, H, hd).permute(2, 0, 3, 1, 4)
    s = (q @ k.transpose(-2, -1)) / math.sqrt(hd)
    p = torch.softmax(s, dim=-1)
    ctx = (p @ v).transpose(1, 2).reshape(B * N, D)
    lse = torch.logsumexp(s, dim=-1)
    return ctx, lse


@pytest.mark.parametrize("B,N,H", [(2, 197, 12), (1, 5, 1), (3, 17, 2), (2, 64, 3), (1, 198, 12),
                                   (1, 577, 4), (2, 16, 1), (1, 65, 2), (2, 128, 2), (1, 129, 1),
                                   (1, 256, 2), (40, 197, 12), (7, 224, 3), (5, 225, 2), (64, 100, 12),
                                   (33, 208, 16), (150, 1, 1), (2, 577, 12), (1, 640, 2), (3, 257, 1),
                                   (1, 513, 3), (20, 384, 4)])
def test_attention(vitk, attn_impl, B, N, H):
    if attn_impl == 3 and N > 256:
        pytest.skip("the unpipelined tcgen05 kernel covers N <= 256")
    g = torch.Generator(device="cuda").manual_seed(N)
    qkv = (torch.randn(B * N, 3 * H * 64, generator=g, device="cuda") * 1.5).bfloat16()
    ctx, lse = vitk.ops.attention(qkv, B, N, H, return_lse=True)
    ref, lse_ref = _attn_ref(qkv, B, N, H)
    torch.testing.assert_close(ctx.float(), ref, rtol=2e-2, atol=2e-2)
    torch.testing.assert_close(lse, lse_ref, rtol=1e-3, atol=1e-3)


def test_attention_peaked_softmax(vitk, attn_impl):
    # large logits: exercises the running-max rescale across key blocks
    B, N, H = 1, 197, 2
    g = torch.Generator(device="cuda").manual_seed(7)
    qkv = (torch.randn(B * N, 3 * H * 64, generator=g, device="cuda") * 6).bfloat16()
    ctx = vitk.ops.attention(qkv, B, N, H)
    ref, _ = _attn_ref(qkv, B, N, H)
    assert torch.isfinite(ctx.float()).all()
    torch.testing.assert_close(ctx.float(), ref, rtol=3e-2, atol=3e-2)


@pytest.mark.parametrize("gap", [40.0, 80.0, 300.0, -300.0])
def test_attention_late_peak(vitk, attn_impl, gap):
    """Scores whose maximum sits `gap` (natural-log units) above/below the first key chunk: the
    pipelined tcgen05 kernel takes its reference exponent from the first 32 keys and must rescale
    the row when a later chunk exceeds it by more than 2^64."""
    B, N, H = 2, 197, 2
    g = torch.Generator(device="cuda").manual_seed(3)
    qkv = torch.randn(B, N, 3, H, 64, generator=g, device="cuda") * 0.3
    u = torch.nn.functional.normalize(torch.randn(64, generator=g, device="cuda"), dim=0)
    qkv[:, :, 0] += 8.0 * u                      # every query has a large component along u
    amp = gap * 8.0 / 8.0                        # q.k / sqrt(64) ~= 8 * amp / 8 = gap
    qkv[:, 70:150, 1] += amp * u                 # keys 70..149 score ~gap higher than keys 0..31
    qkv[:, 190:, 1] += 0.5 * amp * u
    qkv = qkv.reshape(B * N, 3 * H * 64).bfloat16()
    ctx, lse = vitk.ops.attention(qkv, B, N, H, return_lse=True)
    ref, lse_ref = _attn_ref(qkv, B, N, H)
    assert torch.isfinite(ctx.float()).all()
    torch.testing.assert_close(ctx.float(), ref, rtol=3e-2, atol=3e-2)
    torch.testing.assert_close(lse, lse_ref, rtol=1e-3, atol=2e-2)


@pytest.mark.parametrize("N,gap", [(577, 12.0), (577, 60.0), (640, 25.0), (300, 200.0)])
def test_attention_long_sequence_moving_maximum(vitk, N, gap):
    """Long-sequence kernel (one pass over 128-key blocks with a lazily updated reference
    maximum): rows whose block maxima rise by `gap` (natural-log units) from block to block must
    rescale what they have accumulated, rows whose maxima fall must not, rows in between mix -
    all inside the same warps."""
    B, H = 2, 3
    g = torch.Generator(device="cuda").manual_seed(11)
    qkv = torch.randn(B, N, 3, H, 64, generator=g, device="cuda") * 0.3
    u = torch.nn.functional.normalize(torch.randn(64, generator=g, device="cuda"), dim=0)
    sign = torch.linspace(-1.0, 1.0, N, device="cuda").roll(17)[None, :, None, None]
    qkv[:, :, 0] += 8.0 * sign * u                # query component along u: -8 .. +8 over the rows
    blk = (torch.arange(N, device="cuda") // 128).float()[None, :, None, None]
    qkv[:, :, 1] += gap * blk * u                 # keys of block j score ~ sign * gap * j
    qkv = qkv.reshape(B * N, 3 * H * 64).bfloat16()
    vitk._lib.set_attention_impl(4)
    try:
        ctx, lse = vitk.ops.attention(qkv, B, N, H, return_lse=True)
    finally:
        vitk._lib.set_attention_impl(0)
    ref, lse_ref = _attn_ref(qkv, B, N, H)
    assert torch.isfinite(ctx.float()).all() and torch.isfinite(lse).all()
    torch.testing.assert_close(ctx.float(), ref, rtol=3e-2, atol=3e-2)
    torch.testing.assert_close(lse, lse_ref, rtol=1e-3, atol=2e-2)


def test_attention_rejects_other_head_dims(vitk):
    qkv = torch.zeros(10, 3 * 24, device="cuda").bfloat16()
    with pytest.raises(vitk.VitkError):
        vitk.ops.attention(qkv, 1, 10, 2)   # head_dim 12: not a multiple of 8


@pytest.mark.parametrize("rows,D,n_out", [(8, 768, 6), (3, 64, 6), (128, 1024, 256)])
def test_linear_rows_backward(vitk, rows, D, n_out):
    """vitk_linear_rows_backward against autograd of F.linear (the head on the CLS rows)."""
    import ctypes as C
    g = torch.Generator(device="cuda").manual_seed(0)
    x = torch.randn(rows, D, generator=g, device="cuda", requires_grad=True)
    w = (torch.randn(n_out, D, generator=g, device="cuda") / D ** 0.5).requires_grad_(True)
    b = torch.randn(n_out, generator=g, device="cuda", requires_grad=True)
    dy = torch.randn(rows, n_out, generator=g, device="cuda")
    torch.nn.functional.linear(x, w, b).backward(dy)
    dx, dw = torch.empty_like(x), torch.empty_like(w)
    db = torch.empty_like(b)
    vitk._lib.check(vitk._lib.lib().vitk_linear_rows_backward(
        x.data_ptr(), D, w.data_ptr(), dy.data_ptr(), dx.data_ptr(), dw.data_ptr(), db.data_ptr(),
        rows, D, n_out, torch.cuda.current_stream().cuda_stream))
    torch.testing.assert_close(dx, x.grad, rtol=1e-4, atol=1e-4)
    torch.testing.assert_close(dw, w.grad, rtol=1e-4, atol=1e-4)
    torch.testing.assert_close(db, b.grad, rtol=1e-4, atol=1e-4)
