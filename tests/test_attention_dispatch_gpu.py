"""Which attention kernels each entry point runs, for every row of the selection table in
csrc/attention.cu.  The numerical tests accept any kernel that computes the right values, so a
wrong dispatch (say 230 tokens sent to the key-block kernel instead of the single-block one)
passes them; here the kernel names recorded by torch.profiler are compared with the table.
`vitk_attention_set_impl` values: 0 automatic, 1 the mma.sync / CUDA-core kernels, 2-4 force
tcgen05 forward kernels at head_dim 64."""
import re

import pytest
import torch
from torch.profiler import ProfilerActivity, profile

from oracle import vit_oracle as O

pytestmark = pytest.mark.gpu

_KERNEL = re.compile(r"\b(attn_\w+?_kernel(?:<[^<>()]*>)?)")

TC2, TC, TC3, HD64 = ("attn_fwd_tc2_kernel<false>", "attn_fwd_tc_kernel", "attn_fwd_tc3_kernel",
                      "attn_fwd_hd64_kernel")
GEN_FWD, GEN_BWD = "attn_gen_fwd_kernel", "attn_gen_bwd_kernel"


def _ran(fn):
    """Base names (template arguments kept) of the attention kernels `fn` launches."""
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return {m.group(1) for e in prof.events() for m in [_KERNEL.search(e.name)] if m}


def _with_impl(vitk, impl, fn):
    vitk._lib.set_attention_impl(impl)
    try:
        return _ran(fn)
    finally:
        vitk._lib.set_attention_impl(0)


def _qkv(B, N, H, hd, seed=0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return torch.randn(B * N, 3 * H * hd, device="cuda", generator=g).to(torch.bfloat16)


def _fwd_hd64(impl, N):
    if impl == 1:
        return HD64
    if impl == 0 and N > 640:
        return HD64
    if impl == 4:
        return TC3
    if impl in (0, 2) and N <= 208:
        return TC2
    return TC if N <= 256 else TC3


@pytest.mark.parametrize("lse", [False, True], ids=["ctx", "lse"])
@pytest.mark.parametrize("impl", [0, 1, 2, 3, 4])
@pytest.mark.parametrize("N", [1, 208, 209, 256, 257, 640, 641])
def test_packed_forward_hd64(vitk, N, impl, lse):
    if impl in (2, 3, 4) and N > 640:
        pytest.skip("the forced tcgen05 kernels take at most 640 tokens")
    qkv = _qkv(2, N, 2, 64)
    got = _with_impl(vitk, impl, lambda: vitk.ops.attention(qkv, 2, N, 2, return_lse=lse))
    assert got == {_fwd_hd64(impl, N)}


@pytest.mark.parametrize("lse", [False, True], ids=["ctx", "lse"])
@pytest.mark.parametrize("impl", [0, 1])
@pytest.mark.parametrize("hd", [32, 48, 96, 128])
def test_packed_forward_other_head_dims(vitk, hd, impl, lse):
    N = 197
    qkv = _qkv(2, N, 2, hd)
    got = _with_impl(vitk, impl, lambda: vitk.ops.attention(qkv, 2, N, 2, return_lse=lse))
    if not lse and hd in (32, 96, 128):
        want = f"attn_x_kernel<{hd}>"
    else:
        want = GEN_FWD if impl == 1 else f"attn_xmma_fwd_kernel<{hd}>"
    assert got == {want}


@pytest.mark.parametrize("impl", [1, 2])
@pytest.mark.parametrize("N,hd,want", [
    (197, 64, ("attn_bwd_hd64_kernel", "attn_bwd_tc2_kernel<false>")),
    (256, 64, ("attn_bwd_hd64_kernel", "attn_bwd_tc_kernel<false>")),   # tc2's tiles do not fit
    (257, 64, (GEN_BWD, "attn_xmma_bwd_kernel<64>")),
    (577, 64, (GEN_BWD, GEN_BWD)),                                     # beyond the mma.sync tiles
    (197, 32, (GEN_BWD, "attn_xmma_bwd_kernel<32>")),
])
def test_packed_backward(vitk, N, hd, want, impl):
    B, H = 2, 2
    qkv = _qkv(B, N, H, hd)
    ctx, lse = vitk.ops.attention(qkv, B, N, H, return_lse=True)
    dctx = torch.randn_like(ctx)
    got = _with_impl(vitk, impl, lambda: vitk.ops.attention_bwd(qkv, ctx, dctx, lse, B, N, H))
    assert got == {want[0] if impl == 1 else want[1]}


@pytest.mark.parametrize("S,want", [
    (224, {"attn_fwd_tc2_kernel<true>", "attn_bwd_tc2_kernel<true>"}),   # 197 tokens
    (240, {GEN_FWD, "attn_bwd_tc2_kernel<true>"}),                      # 226 tokens
])
def test_train_step_with_dropout(vitk, S, want):
    kw = dict(image_size=S, patch_size=16, embed_dim=128, num_layers=1, num_heads=2, mlp_dim=256,
              dropout=0.1)
    torch.manual_seed(0)
    tuner = vitk.FineTuner(vitk.ViTClassifier(num_classes=6, **kw).cuda().train())
    x, y = O.synthetic_images(2, S).cuda(), O.synthetic_labels(2).cuda()
    assert _ran(lambda: tuner.step(x, y)) == want


def _head(vitk, D, Q):
    torch.manual_seed(0)
    head = vitk.ObjectDetectionHead(embed_dim=D, num_classes=6, num_queries=Q)
    for m in head.modules():
        if isinstance(m, torch.nn.Dropout):
            m.p = 0.0
        if isinstance(m, torch.nn.MultiheadAttention):
            m.dropout = 0.0
    return head.cuda()


# (D, Q, P): head_dim D / 8.  The tcgen05 decoder kernel takes <= 128 queries and <= 256 keys.
HEADS = [(768, 100, 196), (512, 130, 40)]


@pytest.mark.parametrize("impl", [0, 1])
@pytest.mark.parametrize("D,Q,P", HEADS)
def test_head_decode(vitk, D, Q, P, impl):
    head = _head(vitk, D, Q).eval()
    tokens = torch.randn(2, P + 1, D, device="cuda")
    with torch.no_grad():
        got = _with_impl(vitk, impl, lambda: head.decode(tokens, skip_tokens=1))
    hd = D // 8
    tc = impl == 0 and Q <= 128
    assert got == {f"attn_xtc_kernel<{hd}>" if tc else f"attn_x_kernel<{hd}>"}


@pytest.mark.parametrize("impl", [0, 1])
@pytest.mark.parametrize("D,Q,P", HEADS)
def test_head_train_forward_backward(vitk, D, Q, P, impl):
    head = _head(vitk, D, Q).train()
    tokens = torch.randn(2, P + 1, D, device="cuda", requires_grad=True)

    def step():
        out = head.decode(tokens, skip_tokens=1)
        (out["class_logits"].sum() + out["bbox_coords"].sum()).backward()

    got = _with_impl(vitk, impl, step)
    hd = D // 8
    if impl == 1:
        want = {"attn_xgen_fwd_kernel", "attn_xgen_bwd_kernel"}
    elif Q <= 128:
        want = {f"attn_xtc_kernel<{hd}>", f"attn_xmma_bwd_kernel<{hd}>"}
    else:
        want = {f"attn_xmma_fwd_kernel<{hd}>", f"attn_xmma_bwd_kernel<{hd}>"}
    assert got == want


@pytest.mark.parametrize("S,want", [
    (224, {TC2, "attn_xtc_kernel<64>"}),    # 197 tokens: one key block for the CLS query
    (384, {TC3, "attn_x_kernel<64>"}),      # 577 tokens
])
def test_forward_cls_tail(vitk, S, want):
    kw = dict(image_size=S, patch_size=16, embed_dim=128, num_layers=2, num_heads=2, mlp_dim=256,
              dropout=0.0)
    torch.manual_seed(0)
    model = vitk.ViTClassifier(num_classes=6, **kw).cuda().eval()
    x = O.synthetic_images(2, S).cuda()
    with torch.no_grad():
        assert _ran(lambda: model.classify_pruned(x)) == want
