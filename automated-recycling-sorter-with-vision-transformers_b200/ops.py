"""Tensor-level wrappers over the per-operator C-ABI entry points (include/vitk.h).

Each function takes CUDA tensors, passes raw pointers + the current stream to libvitk and returns
the output tensor.  Used by the sub-module forwards and by the parity tests; `vitk_forward` (see
engine.py) runs the same kernels back to back without returning to Python.
"""
from __future__ import annotations

import torch

from . import _lib
from ._lib import check, lib


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _need_cuda(*ts: torch.Tensor) -> None:
    for t in ts:
        if t is not None and not t.is_cuda:
            raise _lib.VitkError("vitk operators need CUDA tensors (there is no CPU fallback)")


def _ptr(t) -> int | None:
    return None if t is None else t.data_ptr()


def cast_bf16(x: torch.Tensor) -> torch.Tensor:
    """fp32 -> bf16 (round to nearest even) with the library's own kernel."""
    _need_cuda(x)
    x = x.contiguous()
    assert x.dtype == torch.float32
    out = torch.empty(x.shape, dtype=torch.bfloat16, device=x.device)
    if x.numel():
        check(lib().vitk_cast_f32_to_bf16(x.data_ptr(), out.data_ptr(), x.numel(), _stream()))
    return out


def split3(x: torch.Tensor, is_weight: bool) -> torch.Tensor:
    """fp32 [R, K] -> bf16 [R, 6K] three-term split operand of the fp32-parity mode."""
    _need_cuda(x)
    assert x.dtype == torch.float32 and x.dim() == 2 and x.stride(1) == 1
    R, K = x.shape
    out = torch.empty((R, 6 * K), dtype=torch.bfloat16, device=x.device)
    check(lib().vitk_split3(x.data_ptr(), x.stride(0), out.data_ptr(), R, K, 1 if is_weight else 0,
                            _stream()))
    return out


def gemm(a: torch.Tensor, b: torch.Tensor, epilogue: int = _lib.EPI_BF16, *, bias=None, resid=None,
         aux=None, out=None, out2=None, alpha: float = 1.0, beta: float = 0.0) -> torch.Tensor:
    """out = epilogue(a @ b.T); a bf16 [M,K], b bf16 [N,K] (nn.Linear weight layout)."""
    _need_cuda(a, b)
    assert a.dtype == torch.bfloat16 and b.dtype == torch.bfloat16
    assert a.dim() == 2 and b.dim() == 2 and a.shape[1] == b.shape[1]
    assert a.stride(1) == 1 and b.stride(1) == 1
    M, K = a.shape
    N = b.shape[0]
    f32_out = epilogue in (_lib.EPI_RESID_F32, _lib.EPI_F32)
    if out is None:
        out = torch.empty((M, N), dtype=torch.float32 if f32_out else torch.bfloat16, device=a.device)
    assert out.stride(1) == 1
    ldr = resid.stride(0) if resid is not None else 0
    check(lib().vitk_gemm(a.data_ptr(), a.stride(0), b.data_ptr(), b.stride(0), M, N, K, epilogue,
                          _ptr(bias), _ptr(resid), ldr, _ptr(aux), out.data_ptr(), _ptr(out2),
                          out.stride(0), alpha, beta, _stream()))
    return out


def gemm_resid_layernorm(a: torch.Tensor, w: torch.Tensor, x: torch.Tensor, gamma: torch.Tensor,
                         beta: torch.Tensor, *, bias=None, eps: float = 1e-5,
                         return_stats: bool = False):
    """x += a @ w.T + bias (in place, fp32) and LN(x) * gamma + beta as bf16, two launches
    (train.py:586-591).  Returns the bf16 LayerNorm output (and mean / rstd)."""
    _need_cuda(a, w, x)
    assert a.dtype == torch.bfloat16 and w.dtype == torch.bfloat16 and x.dtype == torch.float32
    assert a.stride(1) == 1 and w.stride(1) == 1 and x.is_contiguous()
    M, K = a.shape
    N = w.shape[0]
    assert x.shape == (M, N)
    y = torch.empty((M, N), dtype=torch.bfloat16, device=x.device)
    mean = rstd = None
    if return_stats:
        mean = torch.empty(M, dtype=torch.float32, device=x.device)
        rstd = torch.empty(M, dtype=torch.float32, device=x.device)
    check(lib().vitk_gemm_resid_layernorm(a.data_ptr(), a.stride(0), w.data_ptr(), w.stride(0), M,
                                          N, K, _ptr(bias), x.data_ptr(), gamma.data_ptr(),
                                          beta.data_ptr(), eps, y.data_ptr(), _ptr(mean),
                                          _ptr(rstd), _stream()))
    return (y, mean, rstd) if return_stats else y


def fold_layernorm(weight: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, bias=None):
    """Linear(LayerNorm(.)) in the folded form (vitk_fold_layernorm): returns
    (w_ln bf16 [out, in] = weight * gamma with zero-sum rows, b_ln f32 [out] = bias + weight beta,
    rowsum f32 [out] = what bf16 rounding leaves of the row sums of w_ln)."""
    _need_cuda(weight, gamma, beta)
    weight = weight.detach().float().contiguous()
    N, K = weight.shape
    w_ln = torch.empty((N, K), dtype=torch.bfloat16, device=weight.device)
    rowsum = torch.empty(N, dtype=torch.float32, device=weight.device)
    b_ln = torch.empty(N, dtype=torch.float32, device=weight.device)
    g, b = gamma.detach().float().contiguous(), beta.detach().float().contiguous()
    bb = bias.detach().float().contiguous() if bias is not None else None
    check(lib().vitk_fold_layernorm(weight.data_ptr(), g.data_ptr(), b.data_ptr(), _ptr(bb),
                                    w_ln.data_ptr(), b_ln.data_ptr(), rowsum.data_ptr(), N, K,
                                    _stream()))
    return w_ln, b_ln, rowsum


def row_stats(x: torch.Tensor):
    """bf16 copy of the fp32 rows and their (sum, sum of squares): ([rows, D] bf16, [1, rows, 2])."""
    _need_cuda(x)
    assert x.dtype == torch.float32 and x.dim() == 2 and x.stride(1) == 1
    rows, D = x.shape
    xb = torch.empty((rows, D), dtype=torch.bfloat16, device=x.device)
    stats = torch.empty((1, rows, 2), dtype=torch.float32, device=x.device)
    check(lib().vitk_row_stats(x.data_ptr(), x.stride(0), xb.data_ptr(), D, stats.data_ptr(), rows,
                               D, _stream()))
    return xb, stats


def gemm_resid_stats(a: torch.Tensor, w: torch.Tensor, x: torch.Tensor, *, bias=None):
    """x += a @ w.T + bias in place (fp32); returns (bf16(x), stats [parts, M, 2]) - the partial
    (sum, sum of squares) of every updated row per column group (vitk_gemm_resid_stats)."""
    _need_cuda(a, w, x)
    assert a.dtype == torch.bfloat16 and w.dtype == torch.bfloat16 and x.dtype == torch.float32
    assert a.stride(1) == 1 and w.stride(1) == 1 and x.is_contiguous()
    M, K = a.shape
    N = w.shape[0]
    assert x.shape == (M, N)
    xb = torch.empty((M, N), dtype=torch.bfloat16, device=x.device)
    parts = lib().vitk_stats_parts(N)
    stats = torch.empty((parts, M, 2), dtype=torch.float32, device=x.device)
    check(lib().vitk_gemm_resid_stats(a.data_ptr(), a.stride(0), w.data_ptr(), w.stride(0), M, N, K,
                                      _ptr(bias), x.data_ptr(), xb.data_ptr(), stats.data_ptr(),
                                      _stream()))
    return xb, stats


def gemm_layernorm_folded(xb: torch.Tensor, w_ln: torch.Tensor, b_ln: torch.Tensor,
                          stats: torch.Tensor, *, eps: float = 1e-5,
                          epilogue: int = _lib.EPI_BF16) -> torch.Tensor:
    """epilogue(Linear(LayerNorm(x))) from bf16(x), the folded weights and the row statistics."""
    _need_cuda(xb, w_ln, stats)
    assert xb.dtype == torch.bfloat16 and w_ln.dtype == torch.bfloat16
    assert stats.dtype == torch.float32 and stats.is_contiguous() and stats.dim() == 3
    M, K = xb.shape
    N = w_ln.shape[0]
    assert stats.shape[1] == M and stats.shape[2] == 2
    out = torch.empty((M, N), dtype=torch.bfloat16, device=xb.device)
    check(lib().vitk_gemm_layernorm_folded(xb.data_ptr(), xb.stride(0), w_ln.data_ptr(),
                                           w_ln.stride(0), M, N, K, epilogue,
                                           b_ln.data_ptr(), stats.data_ptr(), stats.shape[0], eps,
                                           out.data_ptr(), out.stride(0), _stream()))
    return out


def gemm_wgrad(dy: torch.Tensor, x: torch.Tensor, out: torch.Tensor | None = None, *,
               alpha: float = 1.0, accumulate: bool = False, split_k: int = 1) -> torch.Tensor:
    """out[o, i] (+)= alpha * sum_t dy[t, o] * x[t, i]; dy bf16 [T, O], x bf16 [T, I], out f32."""
    _need_cuda(dy, x)
    assert dy.dtype == torch.bfloat16 and x.dtype == torch.bfloat16
    assert dy.shape[0] == x.shape[0] and dy.stride(1) == 1 and x.stride(1) == 1
    T, O = dy.shape
    I = x.shape[1]
    if out is None:
        out = torch.zeros((O, I), dtype=torch.float32, device=dy.device)
    check(lib().vitk_gemm_wgrad(dy.data_ptr(), dy.stride(0), x.data_ptr(), x.stride(0), O, I, T,
                                out.data_ptr(), out.stride(0), alpha, 1.0 if accumulate else 0.0,
                                split_k, _stream()))
    return out


def layernorm(x: torch.Tensor, weight: torch.Tensor, bias: torch.Tensor, eps: float = 1e-5,
              out_dtype: torch.dtype = torch.bfloat16, return_stats: bool = False):
    """nn.LayerNorm over the last dim of an fp32 [rows, D] tensor."""
    _need_cuda(x)
    assert x.dtype == torch.float32 and x.dim() == 2 and x.stride(1) == 1
    rows, D = x.shape
    y = torch.empty((rows, D), dtype=out_dtype, device=x.device)
    mean = rstd = None
    if return_stats:
        mean = torch.empty(rows, dtype=torch.float32, device=x.device)
        rstd = torch.empty(rows, dtype=torch.float32, device=x.device)
    check(lib().vitk_layernorm(x.data_ptr(), x.stride(0), weight.data_ptr(), bias.data_ptr(),
                               y.data_ptr(), 1 if out_dtype == torch.float32 else 0, D, _ptr(mean),
                               _ptr(rstd), rows, D, eps, _stream()))
    return (y, mean, rstd) if return_stats else y


def attention(qkv: torch.Tensor, batch: int, n_tokens: int, num_heads: int,
              return_lse: bool = False):
    """softmax(q k^T / sqrt(hd)) v on the packed [B*N, 3*D] bf16 qkv activation -> [B*N, D]."""
    _need_cuda(qkv)
    assert qkv.dtype == torch.bfloat16 and qkv.is_contiguous()
    D = qkv.shape[-1] // 3
    ctx = torch.empty((batch * n_tokens, D), dtype=torch.bfloat16, device=qkv.device)
    lse = None
    if return_lse:
        lse = torch.empty((batch, num_heads, n_tokens), dtype=torch.float32, device=qkv.device)
    check(lib().vitk_attention(qkv.data_ptr(), ctx.data_ptr(), _ptr(lse), batch, n_tokens,
                               num_heads, D // num_heads, _stream()))
    return (ctx, lse) if return_lse else ctx


def layernorm_bwd(dy: torch.Tensor, x: torch.Tensor, mean: torch.Tensor, rstd: torch.Tensor,
                  weight: torch.Tensor, dx_resid: torch.Tensor | None = None):
    """Backward of nn.LayerNorm: returns (dx f32 [= dx_resid + dLN], dx bf16 copy, dgamma, dbeta)."""
    _need_cuda(dy, x)
    rows, D = x.shape
    assert dy.shape == x.shape and dy.is_contiguous() and x.is_contiguous()
    dx = dx_resid.clone() if dx_resid is not None else torch.empty_like(x)
    dxb = torch.empty((rows, D), dtype=torch.bfloat16, device=x.device)
    dg = torch.zeros(D, dtype=torch.float32, device=x.device)
    db = torch.zeros(D, dtype=torch.float32, device=x.device)
    check(lib().vitk_layernorm_bwd(dy.data_ptr(), 1 if dy.dtype == torch.float32 else 0,
                                   x.data_ptr(), mean.data_ptr(), rstd.data_ptr(),
                                   weight.data_ptr(), dx.data_ptr(), 1 if dx_resid is not None else 0,
                                   dxb.data_ptr(), dg.data_ptr(), db.data_ptr(), rows, D, None,
                                   0.0, 0, 0, 0, _stream()))
    return dx, dxb, dg, db


def attention_bwd(qkv: torch.Tensor, ctx: torch.Tensor, dctx: torch.Tensor, lse: torch.Tensor,
                  batch: int, n_tokens: int, num_heads: int) -> torch.Tensor:
    """d_qkv (bf16 [B*N, 3D]) of the attention core given d_ctx and the saved log-sum-exp."""
    _need_cuda(qkv, ctx, dctx, lse)
    assert qkv.is_contiguous() and ctx.is_contiguous() and dctx.is_contiguous()
    D = ctx.shape[-1]
    dqkv = torch.empty_like(qkv)
    check(lib().vitk_attention_bwd(qkv.data_ptr(), ctx.data_ptr(), dctx.data_ptr(), lse.data_ptr(),
                                   dqkv.data_ptr(), batch, n_tokens, num_heads, D // num_heads,
                                   _stream()))
    return dqkv


def colsum(y: torch.Tensor, out: torch.Tensor | None = None) -> torch.Tensor:
    """out[n] += sum_m y[m, n] for a bf16 matrix (bias gradients)."""
    _need_cuda(y)
    assert y.dtype == torch.bfloat16 and y.stride(1) == 1
    if out is None:
        out = torch.zeros(y.shape[1], dtype=torch.float32, device=y.device)
    check(lib().vitk_colsum_bf16(y.data_ptr(), y.stride(0), y.shape[0], y.shape[1], out.data_ptr(),
                                 _stream()))
    return out


def adamw_step(p, g, m, v, step: int, lr=1e-4, betas=(0.9, 0.999), eps=1e-8, weight_decay=1e-4,
               shadow=None, grad_scale: float = 1.0) -> None:
    """In-place fused AdamW over flat fp32 tensors (torch.optim.AdamW update rule)."""
    _need_cuda(p, g, m, v)
    check(lib().vitk_adamw_step(p.data_ptr(), g.data_ptr(), m.data_ptr(), v.data_ptr(), _ptr(shadow),
                                p.numel(), lr, betas[0], betas[1], eps, weight_decay, step,
                                grad_scale, _stream()))


def patchify(images: torch.Tensor, patch_size: int) -> torch.Tensor:
    """f32 NCHW -> bf16 [B*P, C*p*p] rows in conv-weight column order."""
    _need_cuda(images)
    assert images.dtype == torch.float32 and images.dim() == 4
    images = images.contiguous()
    B, Cc, S, S2 = images.shape
    assert S == S2
    P = (S // patch_size) ** 2
    out = torch.empty((B * P, Cc * patch_size * patch_size), dtype=torch.bfloat16,
                      device=images.device)
    check(lib().vitk_patchify(images.data_ptr(), out.data_ptr(), B, Cc, S, patch_size, _stream()))
    return out


def postprocess_scores(logits: torch.Tensor, exclude_last: bool = False, return_probs: bool = False):
    """softmax(logits, -1) then max / argmax over the classes (evaluation.py:403-404) in one kernel:
    returns (scores f32 [...], labels i64 [...]) and optionally the probabilities."""
    _need_cuda(logits)
    assert logits.dtype == torch.float32
    lead, C_ = logits.shape[:-1], logits.shape[-1]
    flat = logits.reshape(-1, C_).contiguous()
    rows = flat.shape[0]
    scores = torch.empty(rows, dtype=torch.float32, device=logits.device)
    labels = torch.empty(rows, dtype=torch.int64, device=logits.device)
    probs = torch.empty_like(flat) if return_probs else None
    check(lib().vitk_postprocess_scores(flat.data_ptr(), rows, C_, 1 if exclude_last else 0,
                                        scores.data_ptr(), labels.data_ptr(), _ptr(probs), _stream()))
    out = (scores.reshape(lead), labels.reshape(lead))
    return out + (probs.reshape(logits.shape),) if return_probs else out
