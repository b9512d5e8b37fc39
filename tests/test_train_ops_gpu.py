"""Backward / optimizer kernels through the C ABI vs PyTorch autograd (fp32) on the same inputs (the
LayerNorm backward and the bias column sums are tested in test_train_rowops_gpu.py)."""

import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("B,N,H", [(2, 197, 12), (1, 5, 1), (3, 17, 2), (2, 64, 3), (1, 198, 4),
                                   (1, 129, 2), (1, 256, 1), (1, 128, 2), (30, 197, 12),
                                   # ragged 64-query sub-tiles of the pipelined tcgen05 kernel
                                   (1, 224, 2), (2, 160, 2), (1, 176, 1), (2, 65, 2), (1, 240, 1)])
@pytest.mark.parametrize("impl", [1, 2], ids=["mma_sync", "tcgen05"])
def test_attention_backward(vitk, impl, B, N, H):
    vitk._lib.set_attention_impl(impl)
    try:
        _attention_backward_case(vitk, B, N, H)
    finally:
        vitk._lib.set_attention_impl(0)


def _attention_backward_case(vitk, B, N, H):
    g = torch.Generator(device="cuda").manual_seed(N)
    D = H * 64
    qkv = torch.randn(B * N, 3 * D, generator=g, device="cuda").bfloat16()
    dctx = torch.randn(B * N, D, generator=g, device="cuda").bfloat16()
    ctx, lse = vitk.ops.attention(qkv, B, N, H, return_lse=True)
    dqkv = vitk.ops.attention_bwd(qkv, ctx, dctx, lse, B, N, H)
    ref_in = qkv.float().requires_grad_(True)
    q, k, v = ref_in.reshape(B, N, 3, H, 64).permute(2, 0, 3, 1, 4)
    s = (q @ k.transpose(-2, -1)) / 8.0
    o = (torch.softmax(s, dim=-1) @ v).transpose(1, 2).reshape(B * N, D)
    o.backward(dctx.float())
    err = (dqkv.float() - ref_in.grad).abs().max().item()
    scale = ref_in.grad.abs().max().item()
    assert err < 3e-2 * max(1.0, scale), (err, scale)
    cos = torch.nn.functional.cosine_similarity(dqkv.float().flatten(), ref_in.grad.flatten(), dim=0)
    assert cos > 0.999


@pytest.mark.parametrize("n", [1000, 4096 + 3, 1 << 20])
def test_adamw_matches_torch(vitk, n):
    g0 = torch.Generator(device="cuda").manual_seed(n)
    p = torch.randn(n, generator=g0, device="cuda")
    ref = p.clone().requires_grad_(True)
    opt = torch.optim.AdamW([ref], lr=1e-4, weight_decay=1e-4)   # train.py:1598-1602
    m, v = torch.zeros_like(p), torch.zeros_like(p)
    shadow = torch.empty(n, dtype=torch.bfloat16, device="cuda")
    for step in range(1, 4):
        grad = torch.randn(n, generator=g0, device="cuda") * 0.01
        ref.grad = grad.clone()
        opt.step()
        vitk.ops.adamw_step(p, grad, m, v, step, shadow=shadow)
        torch.testing.assert_close(p, ref.detach(), rtol=1e-6, atol=1e-7)
    assert torch.equal(shadow, p.bfloat16())
    st = opt.state[ref]
    torch.testing.assert_close(m, st["exp_avg"], rtol=1e-6, atol=1e-9)
    torch.testing.assert_close(v, st["exp_avg_sq"], rtol=1e-6, atol=1e-12)


@pytest.mark.parametrize("B,N,H,hd", [(2, 198, 25, 16),    # train.py's Config: D 400, 25 heads, DeiT
                                       (3, 50, 4, 32),
                                       (2, 197, 3, 96),
                                       (1, 197, 2, 128),
                                       (2, 577, 2, 64),     # 384 px: beyond the tcgen05 backward
                                       (1, 257, 1, 8),
                                       (2, 130, 3, 48), (2, 77, 2, 80), (1, 197, 2, 112)])
@pytest.mark.parametrize("impl", [0, 1], ids=["mma.sync-where-it-fits", "cuda-cores"])
def test_generic_attention_forward_and_backward(vitk, B, N, H, hd, impl):
    """The attention kernels behind every shape the tcgen05 kernels leave out - attention_xmma.cu
    (mma.sync; head_dim a multiple of 16, the head's rows in shared memory) and attention_gen.cu
    (CUDA cores; anything else, and everything under impl 1): context, log-sum-exp and d_qkv
    against autograd of the reference's formulation (train.py:536-549)."""
    g = torch.Generator(device="cuda").manual_seed(N + hd)
    D = H * hd
    qkv = torch.randn(B * N, 3 * D, generator=g, device="cuda").bfloat16()
    dctx = torch.randn(B * N, D, generator=g, device="cuda").bfloat16()
    vitk._lib.set_attention_impl(impl)
    try:
        ctx, lse = vitk.ops.attention(qkv, B, N, H, return_lse=True)
        dqkv = vitk.ops.attention_bwd(qkv, ctx, dctx, lse, B, N, H)
    finally:
        vitk._lib.set_attention_impl(0)
    ref_in = qkv.float().requires_grad_(True)
    q, k, v = ref_in.reshape(B, N, 3, H, hd).permute(2, 0, 3, 1, 4)
    s = (q @ k.transpose(-2, -1)) / hd ** 0.5
    o = (torch.softmax(s, dim=-1) @ v).transpose(1, 2).reshape(B * N, D)
    o.backward(dctx.float())
    assert (ctx.float() - o.detach()).abs().max() < 2e-2
    torch.testing.assert_close(lse, torch.logsumexp(s.detach(), dim=-1), rtol=1e-4, atol=1e-4)
    err = (dqkv.float() - ref_in.grad).abs().max().item()
    scale = ref_in.grad.abs().max().item()
    assert err < 3e-2 * max(1.0, scale), (err, scale)
    cos = torch.nn.functional.cosine_similarity(dqkv.float().flatten(), ref_in.grad.flatten(), dim=0)
    assert cos > 0.999


def test_batched_transpose(vitk):
    """vitk_transpose_bf16_batched (W^T copies for the input-gradient GEMMs): full 64 x 64 tiles take
    the 16-byte path, ragged / unaligned matrices the element-wise one; several jobs per launch."""
    import ctypes as C
    g = torch.Generator(device="cuda").manual_seed(0)
    shapes = [(768, 2304), (3072, 768), (100, 70), (64, 64), (130, 200), (8, 8)]
    srcs = [torch.randn(r, c, generator=g, device="cuda").bfloat16() for r, c in shapes]
    # an unaligned source: same data, shifted by one element
    buf = torch.zeros(128 * 128 + 1, device="cuda").bfloat16()
    buf[1:] = srcs[3].new_tensor(torch.randn(128 * 128, generator=torch.Generator().manual_seed(1)).tolist()).bfloat16()
    srcs.append(buf[1:].view(128, 128))
    shapes.append((128, 128))
    dsts = [torch.empty(c, r, dtype=torch.bfloat16, device="cuda") for r, c in shapes]
    n = len(shapes)
    vitk._lib.check(vitk._lib.lib().vitk_transpose_bf16_batched(
        n, (C.c_void_p * n)(*[t.data_ptr() for t in srcs]), (C.c_void_p * n)(*[t.data_ptr() for t in dsts]),
        (C.c_int * n)(*[r for r, _ in shapes]), (C.c_int * n)(*[c for _, c in shapes]),
        torch.cuda.current_stream().cuda_stream))
    for s_, d_ in zip(srcs, dsts):
        assert torch.equal(d_, s_.t().contiguous())
