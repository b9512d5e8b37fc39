"""Separate-source attention at every head_dim from 16 to 128 (the "xr" kernels of
csrc/attention_xr.cu and csrc/attention_xr_bwd.cu, chosen by csrc/attention.cu for head_dims other
than 32 / 64 / 96 / 128), through vitk_attention_src / vitk_attention_src_bwd, against fp64 torch:
forward with and without the log-sum-exp, backward, dropout with the library's own masks, and a
guard that every output column a call does not own keeps its value bit for bit."""
import ctypes as C
import math

import pytest
import torch
from torch.profiler import ProfilerActivity, profile

pytestmark = pytest.mark.gpu

H = 8
SENT = 12345.0          # sentinel in output columns / rows a call does not own
HDS = [16, 24, 40, 48, 49, 50, 72, 80, 100, 127, 128]
SHAPES = [(1, 198), (5, 5), (5, 196), (100, 100), (100, 196), (128, 256), (7, 1)]
pad16 = lambda n: (n + 15) // 16 * 16


class Case:
    """Operands laid out as the detection head lays them out: packed [3D] rows for the
    self-attention (Nq == Nk), a [D] query and K/V in layer 1 of [L*2D = 4D] rows for the
    cross-attention; outputs with a padded pitch and one spare row per image (sentinel-filled)."""

    def __init__(self, B, Nq, Nk, hd, seed=0, single=False, packed=None):
        self.B, self.Nq, self.Nk, self.hd, self.single = B, Nq, Nk, hd, single
        D = self.D = H * hd
        g = torch.Generator(device="cuda").manual_seed(seed)
        rnd = lambda *s: torch.randn(*s, device="cuda", generator=g).to(torch.bfloat16)
        self.packed = (Nq == Nk) if packed is None else packed
        if self.packed:
            self.x = rnd(B, Nq, 3 * D)
            self.q_off, self.k_off, self.v_off = 0, D, 2 * D
            self.qbuf = self.kvbuf = self.x
            self.ldq = self.ldkv = 3 * D
            self.q_img = self.kv_img = Nq * 3 * D
        else:
            self.qbuf = rnd(B, Nq, D)
            self.kvbuf = rnd(B, Nk, 4 * D)
            self.q_off, self.k_off, self.v_off = 0, 2 * D, 3 * D
            self.ldq, self.ldkv = D, 4 * D
            self.q_img, self.kv_img = Nq * D, Nk * 4 * D
        self.ldc = D + 8
        self.ctx_img = (Nq + 1) * self.ldc
        self.dctx = rnd(B, Nq + 1, self.ldc)

    def heads(self):
        """q, k, v as fp64 [B, H, N, hd]."""
        D, hd = self.D, self.hd
        q = self.qbuf[:, :, self.q_off:self.q_off + D]
        k = self.kvbuf[:, :, self.k_off:self.k_off + D]
        v = self.kvbuf[:, :, self.v_off:self.v_off + D]
        f = lambda t: t.double().cpu().reshape(self.B, t.shape[1], H, hd).transpose(1, 2)
        return f(q), f(k), f(v)

    def img(self, x):
        return 0 if self.single else x

    def ptr(self, t, off=0):
        return t.data_ptr() + 2 * off

    def new_ctx(self):
        return torch.full((self.B, self.Nq + 1, self.ldc), SENT, device="cuda", dtype=torch.bfloat16)


def _drop_args(p, seed=77, site=10, layer=1):
    return C.c_float(p), seed, site, layer


def fwd(vitk, c, lse=False, p=0.0, impl=0):
    ctx = c.new_ctx()
    l = torch.full((c.B, H, c.Nq), float("nan"), device="cuda") if lse else None
    st = torch.cuda.current_stream().cuda_stream
    vitk._lib.set_attention_impl(impl)
    try:
        vitk._lib.check(vitk._lib.lib().vitk_attention_src(
            c.ptr(c.qbuf, c.q_off), c.img(c.q_img), c.ldq, c.ptr(c.kvbuf, c.k_off),
            c.ptr(c.kvbuf, c.v_off), c.img(c.kv_img), c.ldkv, ctx.data_ptr(), c.img(c.ctx_img), c.ldc,
            l.data_ptr() if lse else None, c.B, c.Nq, c.Nk, H, c.hd, *_drop_args(p), st))
    finally:
        vitk._lib.set_attention_impl(0)
    torch.cuda.synchronize()
    return ctx, l


def bwd(vitk, c, ctx, lse, p=0.0, impl=0):
    """Returns dq, dk, dv as [B, N, D] plus the raw output buffers (for the guard)."""
    D = c.D
    st = torch.cuda.current_stream().cuda_stream
    if c.packed:
        ld = 3 * D + 8
        dx = torch.full((c.B, c.Nq + 1, ld), SENT, device="cuda", dtype=torch.bfloat16)
        dq_buf, dq_off, lddq, dq_img = dx, 0, ld, (c.Nq + 1) * ld
        dkv_buf, dk_off, dv_off, lddkv, dkv_img = dx, D, 2 * D, ld, (c.Nq + 1) * ld
        bufs = [dx]
    else:
        dq_buf = torch.full((c.B, c.Nq + 1, D + 8), SENT, device="cuda", dtype=torch.bfloat16)
        dq_off, lddq, dq_img = 0, D + 8, (c.Nq + 1) * (D + 8)
        lddkv = 4 * D + 8
        dkv_buf = torch.full((c.B, c.Nk + 1, lddkv), SENT, device="cuda", dtype=torch.bfloat16)
        dk_off, dv_off, dkv_img = 2 * D, 3 * D, (c.Nk + 1) * lddkv
        bufs = [dq_buf, dkv_buf]
    vitk._lib.set_attention_impl(impl)
    try:
        vitk._lib.check(vitk._lib.lib().vitk_attention_src_bwd(
            c.ptr(c.qbuf, c.q_off), c.img(c.q_img), c.ldq, c.ptr(c.kvbuf, c.k_off),
            c.ptr(c.kvbuf, c.v_off), c.img(c.kv_img), c.ldkv, ctx.data_ptr(), c.dctx.data_ptr(),
            c.img(c.ctx_img), c.ldc, lse.data_ptr(), c.ptr(dq_buf, dq_off), c.img(dq_img), lddq,
            c.ptr(dkv_buf, dk_off), c.ptr(dkv_buf, dv_off), c.img(dkv_img), lddkv, c.B, c.Nq, c.Nk,
            H, c.hd, *_drop_args(p), st))
    finally:
        vitk._lib.set_attention_impl(0)
    torch.cuda.synchronize()
    dq = dq_buf[:, :c.Nq, dq_off:dq_off + D]
    dk = dkv_buf[:, :c.Nk, dk_off:dk_off + D]
    dv = dkv_buf[:, :c.Nk, dv_off:dv_off + D]
    owned = [torch.zeros(b.shape, dtype=torch.bool, device="cuda") for b in bufs]
    owned[0][:, :c.Nq, dq_off:dq_off + D] = True
    owned[-1][:, :c.Nk, dk_off:dk_off + D] = True
    owned[-1][:, :c.Nk, dv_off:dv_off + D] = True
    return dq, dk, dv, list(zip(bufs, owned))


def masks(vitk, c, p, seed=77, site=10, layer=1):
    """The library's keep masks for the attention probabilities, scaled by 1 / (1 - p)."""
    n = c.B * H * c.Nq * pad16(c.Nk)
    out = torch.empty(n, dtype=torch.uint8, device="cuda")
    vitk._lib.check(vitk._lib.lib().vitk_dropout_keep_mask(
        C.c_float(p), seed, site, layer, n, out.data_ptr(), torch.cuda.current_stream().cuda_stream))
    t = int(p * 65536 + 0.5)
    m = out.view(c.B, H, c.Nq, pad16(c.Nk))[..., :c.Nk].double().cpu()
    return m * (65536.0 / (65536 - t))


def reference(c, mask=None, grads=False):
    q, k, v = c.heads()
    if grads:
        q, k, v = (t.requires_grad_(True) for t in (q, k, v))
    s = q @ k.transpose(-1, -2) / math.sqrt(c.hd)
    lse = torch.logsumexp(s, -1)
    pr = torch.softmax(s, -1)
    if mask is not None:
        pr = pr * mask
    o = pr @ v
    if not grads:
        return o, lse
    do = c.dctx[:, :c.Nq, :c.D].double().cpu().reshape(c.B, c.Nq, H, c.hd).transpose(1, 2)
    (o * do).sum().backward()
    back = lambda t: t.grad.transpose(1, 2).reshape(c.B, -1, c.D)
    return back(q), back(k), back(v)


def as_heads(c, ctx):
    return ctx[:, :c.Nq, :c.D].double().cpu().reshape(c.B, c.Nq, H, c.hd).transpose(1, 2)


def check_ctx_guard(c, ctx):
    """Columns past H*hd and the spare row of every image keep the sentinel."""
    assert (ctx[:, :c.Nq, c.D:] == SENT).all()
    assert (ctx[:, c.Nq, :] == SENT).all()


def rel(a, b):
    """Relative error, with an absolute floor (an RMS of 1e-2) for gradients that are zero in
    exact arithmetic: with a single key the softmax is constant and dq vanishes."""
    a, b = a.double().flatten().cpu(), b.double().flatten().cpu()
    return ((a - b).norm() / max(b.norm().item(), 1e-2 * b.numel() ** 0.5)).item()


@pytest.mark.parametrize("Nq,Nk", SHAPES)
@pytest.mark.parametrize("hd", HDS)
def test_forward_matches_fp64(vitk, hd, Nq, Nk):
    c = Case(3, Nq, Nk, hd, seed=hd * 1000 + Nq + Nk)
    o_ref, lse_ref = reference(c)
    ctx, _ = fwd(vitk, c)
    check_ctx_guard(c, ctx)
    err = (as_heads(c, ctx) - o_ref).abs().max().item()
    assert err < 3e-2, err
    ctx2, lse = fwd(vitk, c, lse=True)
    check_ctx_guard(c, ctx2)
    assert torch.equal(ctx2[:, :Nq, :c.D], ctx[:, :Nq, :c.D])   # same kernel, same arithmetic
    assert (lse.double().cpu() - lse_ref).abs().max().item() < 1e-2


@pytest.mark.parametrize("packed", [True, False], ids=["self", "cross"])
@pytest.mark.parametrize("hd", [24, 50, 100])
def test_single_image_without_image_stride(vitk, hd, packed):
    """batch 1 with q_img = kv_img = 0, as the head's layer-0 self-attention calls it."""
    Nq, Nk = (5, 5) if packed else (5, 196)
    c = Case(1, Nq, Nk, hd, seed=5, single=True, packed=packed)
    o_ref, lse_ref = reference(c)
    ctx, lse = fwd(vitk, c, lse=True)
    check_ctx_guard(c, ctx)
    assert (as_heads(c, ctx) - o_ref).abs().max().item() < 3e-2
    assert (lse.double().cpu() - lse_ref).abs().max().item() < 1e-2
    dq, dk, dv, guard = bwd(vitk, c, ctx, lse)
    for got, want in zip((dq, dk, dv), reference(c, grads=True)):
        assert rel(got, want) < 3e-2
    for buf, owned in guard:
        assert (buf[~owned] == SENT).all()


@pytest.mark.parametrize("Nq,Nk", [(5, 5), (5, 196), (100, 100), (100, 196), (128, 256), (1, 198), (7, 1)])
@pytest.mark.parametrize("hd", [16, 40, 49, 50, 80, 127, 128])
def test_backward_matches_fp64_autograd(vitk, hd, Nq, Nk):
    c = Case(2, Nq, Nk, hd, seed=hd + 7 * Nq + Nk)
    ctx, lse = fwd(vitk, c, lse=True)
    dq, dk, dv, guard = bwd(vitk, c, ctx, lse)
    for name, got, want in zip("qkv", (dq, dk, dv), reference(c, grads=True)):
        e = rel(got, want)
        assert e < 3e-2, (name, e)
    for buf, owned in guard:                   # padding, spare rows, the other layer's K/V half
        assert (buf[~owned] == SENT).all()


@pytest.mark.parametrize("Nq,Nk", [(5, 196), (100, 100), (128, 256)])
@pytest.mark.parametrize("hd", [50, 100])
def test_dropout_matches_fp64_with_the_library_masks(vitk, hd, Nq, Nk):
    p = 0.1
    c = Case(2, Nq, Nk, hd, seed=hd + Nq)
    m = masks(vitk, c, p)
    o_ref, lse_ref = reference(c, mask=m)
    ctx, lse = fwd(vitk, c, lse=True, p=p)
    check_ctx_guard(c, ctx)
    assert (as_heads(c, ctx) - o_ref).abs().max().item() < 3e-2
    assert (lse.double().cpu() - lse_ref).abs().max().item() < 1e-2   # the row sum counts every term
    plain, _ = fwd(vitk, c, lse=True)
    assert (plain[:, :Nq, :c.D].float() - ctx[:, :Nq, :c.D].float()).abs().max() > 1e-2
    dq, dk, dv, guard = bwd(vitk, c, ctx, lse, p=p)
    for name, got, want in zip("qkv", (dq, dk, dv), reference(c, mask=m, grads=True)):
        e = rel(got, want)
        assert e < 3e-2, (name, e)
    for buf, owned in guard:
        assert (buf[~owned] == SENT).all()


@pytest.mark.parametrize("Nq,Nk", [(5, 196), (100, 100)])
@pytest.mark.parametrize("hd", [48, 80])
def test_agrees_with_the_cuda_core_kernels(vitk, hd, Nq, Nk):
    """At head_dims the existing training kernels also take, impl 1 keeps them (attn_xgen_*):
    an independent implementation to compare the tcgen05 kernels with."""
    c = Case(2, Nq, Nk, hd, seed=hd)
    ctx0, lse0 = fwd(vitk, c, lse=True, impl=0)
    ctx1, lse1 = fwd(vitk, c, lse=True, impl=1)
    assert (ctx0[:, :Nq, :c.D].float() - ctx1[:, :Nq, :c.D].float()).abs().max() < 2e-2
    assert (lse0 - lse1).abs().max() < 1e-3
    g0 = bwd(vitk, c, ctx0, lse0, impl=0)[:3]
    g1 = bwd(vitk, c, ctx0, lse0, impl=1)[:3]
    for a, b in zip(g0, g1):
        assert rel(a, b) < 2e-2


_KERNEL_PREFIX = "attn_"


def _ran(fn):
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return {e.name for e in prof.events() if _KERNEL_PREFIX in e.name}


@pytest.mark.parametrize("hd", [24, 50, 100])
def test_ragged_head_dims_run_the_xr_kernels(vitk, hd):
    c = Case(2, 5, 196, hd)
    names = _ran(lambda: fwd(vitk, c))
    assert any("attn_xr_fwd_kernel" in n for n in names), names
    ctx, lse = fwd(vitk, c, lse=True)
    assert any("attn_xr_fwd_kernel" in n for n in _ran(lambda: fwd(vitk, c, lse=True, p=0.1)))
    names = _ran(lambda: bwd(vitk, c, ctx, lse))
    assert any("attn_xr_bwd_kernel" in n for n in names), names
    if hd % 8 != 0:   # impl 1 still needs xr where no other kernel takes the head_dim
        names = _ran(lambda: bwd(vitk, c, ctx, lse, impl=1))
        assert any("attn_xr_bwd_kernel" in n for n in names), names


def test_existing_head_dims_keep_their_kernels(vitk):
    c = Case(2, 100, 196, 64)
    names = _ran(lambda: fwd(vitk, c))
    assert any("attn_xtc_kernel" in n for n in names) and not any("xr" in n for n in names), names
    c = Case(2, 100, 196, 48)
    ctx, lse = fwd(vitk, c, lse=True)
    names = _ran(lambda: bwd(vitk, c, ctx, lse, impl=1))
    assert any("attn_xgen_bwd_kernel" in n for n in names), names


@pytest.mark.parametrize("Nq,Nk,hd", [(5, 257, 50), (129, 196, 50), (5, 196, 8)])
def test_unsupported_shapes_are_rejected_before_any_launch(vitk, Nq, Nk, hd):
    c = Case(1, Nq, Nk, hd)
    n0 = vitk.launch_count()
    with pytest.raises(vitk.VitkError):
        fwd(vitk, c)
    if hd != 8:   # (head_dim 8 with the log-sum-exp is the CUDA-core training kernels' shape)
        with pytest.raises(vitk.VitkError):
            fwd(vitk, c, lse=True)
    assert vitk.launch_count() == n0
