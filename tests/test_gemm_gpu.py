"""tcgen05 GEMM (vitk_gemm through the C ABI) vs an fp32 matmul of the same bf16 operands."""
import pytest
import torch

pytestmark = pytest.mark.gpu

SHAPES = [
    (128, 256, 64),      # one tile, one k-block
    (128, 256, 256),     # k pipeline wraps the 4-stage ring
    (256, 512, 768),     # 2x2 tiles
    (300, 768, 768),     # ragged M
    (1000, 400, 400),    # ragged N and K (train.py Config dims D=400)
    (197 * 32, 2304, 768),   # C1 qkv
    (197 * 8, 768, 3072),    # fc2 shape, long K
    (64, 128, 64),       # BLOCK_N=128 path, M < tile
]


@pytest.fixture(params=[(1, False), (2, False), (1, True), (2, True)],
                ids=["cta1-tma", "cta2-tma", "cta1-direct", "cta2-direct"], autouse=True)
def gemm_mode(request, vitk):
    """Every GEMM test runs with single-CTA and CTA-pair (cta_group::2) tiles, and with the
    TMA-store and the direct epilogue."""
    ctas, direct = request.param
    vitk._lib.set_gemm_cta_group(ctas)
    vitk._lib.set_gemm_direct_epilogue(direct)
    yield request.param
    vitk._lib.set_gemm_cta_group(0)
    vitk._lib.set_gemm_direct_epilogue(False)


def _ref(a, b):
    return a.float() @ b.float().t()


def _mk(M, N, K, seed=0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    a = torch.randn(M, K, generator=g, device="cuda").bfloat16()
    b = (torch.randn(N, K, generator=g, device="cuda") / K ** 0.5).bfloat16()
    bias = torch.randn(N, generator=g, device="cuda")
    return a, b, bias


@pytest.mark.parametrize("M,N,K", SHAPES)
def test_gemm_f32_epilogue(vitk, M, N, K):
    a, b, bias = _mk(M, N, K)
    out = vitk.ops.gemm(a, b, vitk._lib.EPI_F32, bias=bias)
    ref = _ref(a, b) + bias
    torch.testing.assert_close(out, ref, rtol=1e-4, atol=1e-4)


@pytest.mark.parametrize("M,N,K", SHAPES)
def test_gemm_bf16_epilogue(vitk, M, N, K):
    a, b, bias = _mk(M, N, K, seed=1)
    out = vitk.ops.gemm(a, b, vitk._lib.EPI_BF16, bias=bias)
    ref = (_ref(a, b) + bias).bfloat16()
    torch.testing.assert_close(out.float(), ref.float(), rtol=1e-2, atol=1e-2)


@pytest.mark.parametrize("M,N,K", SHAPES[:5])
def test_gemm_gelu_epilogue(vitk, M, N, K):
    a, b, bias = _mk(M, N, K, seed=2)
    pre = torch.empty(M, N, dtype=torch.bfloat16, device="cuda")
    out = vitk.ops.gemm(a, b, vitk._lib.EPI_GELU_BF16, bias=bias, out2=pre)
    x = _ref(a, b) + bias
    torch.testing.assert_close(pre.float(), x.bfloat16().float(), rtol=1e-2, atol=1e-2)
    ref = torch.nn.functional.gelu(x)  # erf form
    torch.testing.assert_close(out.float(), ref.bfloat16().float(), rtol=1e-2, atol=1e-2)


@pytest.mark.parametrize("M,N,K", SHAPES[:5])
def test_gemm_relu_epilogue(vitk, M, N, K):
    """linear1 + ReLU of the decoder feed-forward (nn.TransformerDecoderLayer, evaluation.py:170)."""
    a, b, bias = _mk(M, N, K, seed=7)
    out = vitk.ops.gemm(a, b, vitk._lib.EPI_RELU_BF16, bias=bias)
    ref = torch.relu(_ref(a, b) + bias)
    assert (out >= 0).all()
    torch.testing.assert_close(out.float(), ref.bfloat16().float(), rtol=1e-2, atol=1e-2)


@pytest.mark.parametrize("M,N,K", SHAPES[:5])
def test_gemm_residual_epilogue_inplace(vitk, M, N, K):
    a, b, bias = _mk(M, N, K, seed=3)
    resid = torch.randn(M, N, device="cuda")
    ref = _ref(a, b) + bias + resid
    x = resid.clone()
    out = vitk.ops.gemm(a, b, vitk._lib.EPI_RESID_F32, bias=bias, resid=x, out=x)
    assert out.data_ptr() == x.data_ptr()
    torch.testing.assert_close(x, ref, rtol=1e-4, atol=1e-4)


def test_gemm_alpha_beta(vitk):
    a, b, bias = _mk(256, 256, 128, seed=4)
    c0 = torch.randn(256, 256, device="cuda")
    out = vitk.ops.gemm(a, b, vitk._lib.EPI_F32, out=c0.clone(), alpha=0.5, beta=2.0)
    torch.testing.assert_close(out, 0.5 * _ref(a, b) + 2.0 * c0, rtol=1e-4, atol=1e-4)


def test_gemm_dgelu_epilogue(vitk):
    a, b, _ = _mk(256, 256, 128, seed=5)
    pre = torch.randn(256, 256, device="cuda").bfloat16()
    out = vitk.ops.gemm(a, b, vitk._lib.EPI_DGELU_BF16, aux=pre)
    x = pre.float().requires_grad_(True)
    torch.nn.functional.gelu(x).sum().backward()
    ref = _ref(a, b) * x.grad
    torch.testing.assert_close(out.float(), ref.bfloat16().float(), rtol=2e-2, atol=2e-2)


def test_gemm_rejects_bad_arguments(vitk):
    a, b, _ = _mk(128, 256, 64)
    with pytest.raises(vitk.VitkError):
        vitk.ops.gemm(a[:, :60], b[:, :60])          # K not a multiple of 8
    with pytest.raises(vitk.VitkError):
        vitk.ops.gemm(a.cpu(), b.cpu())              # no CPU fallback


def test_gemm_many_tiles_deterministic(vitk):
    a, b, bias = _mk(197 * 64, 768, 768, seed=6)
    o1 = vitk.ops.gemm(a, b, vitk._lib.EPI_F32, bias=bias)
    o2 = vitk.ops.gemm(a, b, vitk._lib.EPI_F32, bias=bias)
    assert torch.equal(o1, o2)
    torch.testing.assert_close(o1, _ref(a, b) + bias, rtol=1e-4, atol=1e-4)


@pytest.mark.parametrize("T,O,I,split", [(64, 128, 256, 1), (256, 128, 256, 1), (1000, 768, 768, 1),
                                         (197 * 16, 768, 3072, 4), (197 * 16, 2304, 768, 3),
                                         (5000, 400, 400, 2), (197 * 32, 3072, 768, 8)])
def test_gemm_wgrad_mn_major(vitk, T, O, I, split):
    """dW = dY^T X with both operands read in place (MN-major tcgen05 descriptors), split-K."""
    g = torch.Generator(device="cuda").manual_seed(T)
    dy = torch.randn(T, O, generator=g, device="cuda").bfloat16()
    x = torch.randn(T, I, generator=g, device="cuda").bfloat16()
    ref = dy.float().t() @ x.float()
    out = torch.zeros(O, I, device="cuda")
    vitk.ops.gemm_wgrad(dy, x, out, accumulate=(split > 1), split_k=split)
    torch.testing.assert_close(out, ref, rtol=2e-4, atol=2e-3 * (T / 256) ** 0.5)
    # accumulate on top of an existing gradient
    out2 = ref.clone()
    vitk.ops.gemm_wgrad(dy, x, out2, alpha=0.5, accumulate=True, split_k=split)
    torch.testing.assert_close(out2, 1.5 * ref, rtol=2e-4, atol=3e-3 * (T / 256) ** 0.5)


# ---- residual GEMM followed by its LayerNorm (train.py:586-591) ------------------------------
LN_SHAPES = [
    (15, 64, 64),          # tiny model of the smoke test: one partial row block, BLOCK_N = 128
    (128, 256, 256),       # exactly one row block
    (300, 768, 768),       # ragged M, three column tiles per row block
    (1000, 400, 1600),     # train.py Config dims (D = 400): ragged N tile, LayerNorm lanes past D
    (197 * 8, 768, 3072),  # linear2 of ViT-B/16
    (197 * 4, 1024, 1024),  # ViT-L width: four column tiles, 8 float4 per lane
    (129, 768, 768),       # second CTA of the pair owns a single row
    (197 * 256, 768, 768),  # configs[1] geometry: every CTA pair covers several row blocks
]


@pytest.mark.parametrize("M,N,K", LN_SHAPES)
def test_gemm_resid_layernorm_matches_gemm_then_layernorm(vitk, M, N, K, gemm_mode):
    """vitk_gemm_resid_layernorm == vitk_gemm(RESID_F32) followed by vitk_layernorm, bit for bit,
    and both match fp32 PyTorch."""
    a, w, bias = _mk(M, N, K, seed=7)
    g = torch.Generator(device="cuda").manual_seed(8)
    x0 = torch.randn(M, N, generator=g, device="cuda")
    gamma = 1.0 + 0.1 * torch.randn(N, generator=g, device="cuda")
    beta = 0.1 * torch.randn(N, generator=g, device="cuda")

    x_ref = x0.clone()
    vitk.ops.gemm(a, w, vitk._lib.EPI_RESID_F32, bias=bias, resid=x_ref, out=x_ref)
    y_ref, mean_ref, rstd_ref = vitk.ops.layernorm(x_ref, gamma, beta, return_stats=True)

    x = x0.clone()
    y, mean, rstd = vitk.ops.gemm_resid_layernorm(a, w, x, gamma, beta, bias=bias, return_stats=True)
    assert torch.equal(x, x_ref)
    assert torch.equal(y, y_ref)
    assert torch.equal(mean, mean_ref) and torch.equal(rstd, rstd_ref)

    xt = x0 + _ref(a, w) + bias
    torch.testing.assert_close(x, xt, rtol=1e-4, atol=2e-4)
    yt = torch.nn.functional.layer_norm(xt, (N,), gamma, beta, 1e-5)
    torch.testing.assert_close(y.float(), yt, rtol=1e-2, atol=2e-2)


