"""The row and optimizer kernels of the training step (train_ops.cu, and the LayerNorm forward of
rowops.cu) against an fp64 reference computed from the same fp32 / bf16 inputs the kernel got, at
the dispatch, shape and fused-option edges: every layernorm_bwd instantiation with and without
the residual, the bf16 copy, the parameter gradients, the bias column sums, the dropout mask and
the in-place form; the classifier loss tail; the weighted cross-entropy across several blocks
with ignored targets; AdamW's vector body and scalar tail with the non-finite guard; the bf16
column sums.  Places a kernel must not write hold NaN sentinels whose bits must come back.

Every fp32 element is held to |out - ref| <= C_ROUND * 2^-24 * M, where M is the magnitude of
the terms that produce the element:
  - the reference evaluated on absolute values (|x| for sums, |a| |b| for products), which bounds
    the rounding of any evaluation order of depth <= C_ROUND;
  - plus, where a computed statistic feeds later terms, its own bound carried through the
    reference's derivative: the mean's error shifts every x - mean, and var' = var + dmean^2
    gives rstd a relative error of dmean^2 / (2 (var + eps)) on top of rsqrtf's 2 ulp;
  - plus, for a sum that one thread accumulates term by term over the classes (the softmax
    denominators), u times the sum of its partial sums in that order: the first-order error
    bound of recursive summation (Higham, Accuracy and Stability of Numerical Algorithms, 4.2),
    which a depth-independent multiple of the magnitude does not cover for 4096 terms;
  - plus, for an output that n atomic adds accumulate onto its initial value in an unknown order
    (one add per CTA or per image), u n (|initial| + sum |terms|): the same bound with every
    partial sum bounded by the total magnitude;
  - plus the documented error of the fast intrinsics: expf 2 ulp, logf 1 ulp, rsqrtf 2 ulp,
    __expf(y) 2 + floor(1.173 |y|) ulp, __logf(z) 2^-21.41 absolute on [0.5, 2] and 3 ulp
    elsewhere (CUDA C Programming Guide, mathematical functions), and the rounding of the
    argument y = l - max, u |y|, which exp turns into a relative error; __expf flushes results
    below 2^-126 to zero, an absolute 2^-126 per term.
Errors of inputs to a later stage (features into logits, logits into the softmax, ...) are
propagated with the absolute values of the reference's partial derivatives.  The worst
err / bound per kernel family is printed at the end of the module (pytest -s).  Every bf16 output
is the rounding of an fp32 value the kernel also returns, and must equal bf16() of that value
bit for bit (after the dropout mask and scale, where one applies).
"""
import math
import re
from pathlib import Path

import numpy as np
import pytest
import torch
import torch.nn.functional as F

# Observed worst err / bound on a B200 (1000 W power limit): 0.25 (classifier tail, dbeta), 0.20
# (weighted cross-entropy, dlogits), <= 0.084 elsewhere; printed per family at the end of the
# module with -s.
C_ROUND = 32
U24 = 2.0 ** -24
ULP = 2.0 ** -23          # one fp32 ulp, relative, upper bound
TINY = 2.0 ** -126        # __expf flushes results below the smallest normal float to zero
EPS = float(np.float32(1e-5))

ROOT = Path(__file__).resolve().parent.parent
CSRC = ROOT / "automated-recycling-sorter-with-vision-transformers_b200" / "csrc"

gpu = pytest.mark.gpu


# ---- shared helpers -----------------------------------------------------------------------------
_REPORT = {}


def _note(key, value):
    _REPORT[key] = max(_REPORT.get(key, 0.0), value)


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    if _REPORT:
        print("\nworst err / bound per kernel family (and per output):")
        for k in sorted(_REPORT):
            print(f"  {k:40s} {_REPORT[k]:.4g}")


def _gen(seed):
    return torch.Generator(device="cuda").manual_seed(seed)


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _p(t):
    return None if t is None else t.data_ptr()


def _bits(t):
    return t.view(torch.int32) if t.element_size() == 4 else t.view(torch.int16)


def _check(family, name, out, ref, bound):
    """|out - ref| <= bound elementwise; records the worst ratio under `family`."""
    out = out.double()
    ref = ref.double()
    assert torch.isfinite(out).all(), f"{name}: non-finite output"
    err = (out - ref).abs()
    ratio = torch.where(bound > 0, err / bound.clamp_min(1e-300),
                        torch.where(err > 0, torch.full_like(err, math.inf), torch.zeros_like(err)))
    worst = ratio.max().item() if ratio.numel() else 0.0
    _note(family, worst)
    _note(f"{family} / {name.split(',')[0]}", worst)
    if worst > 1.0:
        i = int(ratio.argmax())
        raise AssertionError(
            f"{name}: err / bound = {worst:.3g} at flat index {i}: out {out.flatten()[i].item()!r}, "
            f"ref {ref.flatten()[i].item()!r}, bound {bound.flatten()[i].item():.3g}; "
            f"{int((ratio > 1).sum())} of {ratio.numel()} elements out of bound")


def _same_bits(a, b, what):
    assert torch.equal(_bits(a), _bits(b)), f"{what}: bits differ"


def _nan(shape, dtype=torch.float32):
    return torch.full(shape, math.nan, dtype=dtype, device="cuda")


def _untouched(buf, before, keep_out, what):
    """The elements of `buf` where keep_out is True still hold the bits of `before`."""
    a, b = _bits(buf), _bits(before)
    assert torch.equal(a[keep_out], b[keep_out]), f"{what}: wrote where it must not"


class _Rows:
    """A [rows, D] operand inside a NaN-filled buffer of `pitch` columns, starting at column
    `off`; everything outside the operand must come back untouched."""

    def __init__(self, rows, D, dtype, pitch=None, off=0):
        self.D, self.off = D, off
        self.pitch = pitch if pitch is not None else D
        self.buf = _nan((rows, self.pitch), dtype)
        self.view = self.buf[:, off:off + D]
        self.outside = torch.ones(rows, self.pitch, dtype=torch.bool, device="cuda")
        self.outside[:, off:off + D] = False

    def fill(self, values):
        self.view.copy_(values)
        return self

    def snapshot(self):
        self.before = self.buf.clone()
        return self

    def check_outside(self, what):
        _untouched(self.buf, self.before, self.outside, what)


# ---- LayerNorm forward (vitk_layernorm) ----------------------------------------------------------
LN_D = [4, 124, 128, 132, 252, 256, 260, 392, 400, 508, 512, 516, 764, 768, 1020, 1024]
LN_ROWS = [1, 7, 8, 9, 6304]
LN_LAYOUTS = ["dense", "strided", "views"]


def _fwd_cases():
    cases = []
    for i, D in enumerate(LN_D):
        for k in range(2):
            cases.append((D, LN_ROWS[(i + 2 * k) % 5], LN_LAYOUTS[(i + k) % 3], (i + k) % 2 == 0))
    # shapes of the earlier fp32-parity test
    cases += [(D, rows, "dense", True) for rows, D in
              [(1, 768), (197, 768), (6304, 768), (50, 1024), (33, 400), (7, 64)]]
    return cases


FWD_CASES = _fwd_cases()


def _ln_fwd_layout(layout, D, f32):
    """(x pitch, x offset, y pitch, y offset) in elements; offsets are 16 bytes."""
    if layout == "dense":
        return D, 0, D, 0
    if layout == "strided":
        return D + 12, 0, D + 20, 0
    return (D + 8, 4, D + 8, 4) if f32 else (D + 8, 4, D + 16, 8)


def _ln_fwd_call(vitk, x, x_pitch, g, b, y, y_f32, y_pitch, mean, rstd, rows, D):
    vitk._lib.check(vitk._lib.lib().vitk_layernorm(
        x.data_ptr(), x_pitch, g.data_ptr(), b.data_ptr(), y.data_ptr(), 1 if y_f32 else 0, y_pitch,
        _p(mean), _p(rstd), rows, D, EPS, _stream()))


def _ln_fwd_ref(x, g, b):
    """fp64 LayerNorm of the fp32 rows and the bounds of mean, rstd and y (module docstring)."""
    c = C_ROUND * U24
    x64 = x.double()
    mu = x64.mean(1, keepdim=True)
    var = ((x64 - mu) ** 2).mean(1, keepdim=True)
    rstd = 1.0 / torch.sqrt(var + EPS)
    xh = (x64 - mu) * rstd
    g64, b64 = g.double(), b.double()
    y = xh * g64 + b64
    mu_err = c * x64.abs().mean(1, keepdim=True)
    rstd_rel = c + 2 * ULP + 0.5 * mu_err ** 2 / (var + EPS)
    y_bound = (c * ((xh * g64).abs() + b64.abs()) + mu_err * rstd * g64.abs()
               + rstd_rel * (xh * g64).abs())
    return dict(mean=mu[:, 0], var=var[:, 0], rstd=rstd[:, 0], y=y, mean_bound=mu_err[:, 0],
                rstd_bound=rstd_rel[:, 0] * rstd[:, 0], y_bound=y_bound, xh=xh)


def _ln_fwd_run(vitk, x_rows, g, b, D, rows, layout, stats, f32):
    x_pitch, _, y_pitch, y_off = _ln_fwd_layout(layout, D, f32)
    y = _Rows(rows, D, torch.float32 if f32 else torch.bfloat16, y_pitch, y_off).snapshot()
    mean = _nan((rows + 1,)) if stats else None
    rstd = _nan((rows + 1,)) if stats else None
    _ln_fwd_call(vitk, x_rows.view, x_pitch, g, b, y.view, f32, y_pitch, mean, rstd, rows, D)
    y.check_outside("layernorm y")
    if stats:
        assert math.isnan(mean[rows].item()) and math.isnan(rstd[rows].item()), \
            "layernorm: wrote past the last row's statistics"
    return y, mean, rstd


@gpu
@pytest.mark.parametrize("D,rows,layout,stats", FWD_CASES,
                         ids=[f"D{D}-r{r}-{l}-{'stats' if s else 'nostats'}" for D, r, l, s in FWD_CASES])
def test_layernorm_forward(vitk, D, rows, layout, stats):
    g_ = _gen(D * 31 + rows)
    x_pitch, x_off, _, _ = _ln_fwd_layout(layout, D, True)
    xv = torch.randn(rows, D, generator=g_, device="cuda") * 3 + 1.5
    if rows >= 8:
        xv[3] = 1e4 + torch.randn(D, generator=g_, device="cuda")     # common offset 1e4
    x = _Rows(rows, D, torch.float32, x_pitch, x_off).fill(xv).snapshot()
    gamma = torch.randn(D, generator=g_, device="cuda")
    beta = torch.randn(D, generator=g_, device="cuda")
    ref = _ln_fwd_ref(xv, gamma, beta)
    outs = {}
    for f32 in (True, False):
        y, mean, rstd = _ln_fwd_run(vitk, x, gamma, beta, D, rows, layout, stats, f32)
        y2, mean2, rstd2 = _ln_fwd_run(vitk, x, gamma, beta, D, rows, layout, stats, f32)
        _same_bits(y.buf, y2.buf, "layernorm y, two calls")
        if stats:
            _same_bits(mean, mean2, "layernorm mean, two calls")
            _same_bits(rstd, rstd2, "layernorm rstd, two calls")
            _check("layernorm_fwd", "mean", mean[:rows], ref["mean"], ref["mean_bound"])
            _check("layernorm_fwd", "rstd", rstd[:rows], ref["rstd"], ref["rstd_bound"])
        outs[f32] = y.view.clone()
    x.check_outside("layernorm x")
    _check("layernorm_fwd", "y f32", outs[True], ref["y"], ref["y_bound"])
    _same_bits(outs[False], outs[True].bfloat16(), "y bf16 against bf16(y f32)")


@gpu
@pytest.mark.parametrize("D", [4, 128, 400, 768, 1024])
def test_layernorm_forward_constant_rows(vitk, D):
    """Variance 0: y must be beta exactly and rstd 1 / sqrt(eps) (to rsqrtf's 2 ulp)."""
    g_ = _gen(D)
    rows = 9
    x = torch.randn(rows, D, generator=g_, device="cuda")
    x[0] = 0.75
    x[4] = -2.5
    x[8] = 0.0
    gamma = torch.randn(D, generator=g_, device="cuda")
    beta = torch.randn(D, generator=g_, device="cuda")
    for f32 in (True, False):
        y = torch.empty(rows, D, dtype=torch.float32 if f32 else torch.bfloat16, device="cuda")
        mean, rstd = _nan((rows,)), _nan((rows,))
        _ln_fwd_call(vitk, x, D, gamma, beta, y, f32, D, mean, rstd, rows, D)
        want = beta if f32 else beta.bfloat16()
        for r in (0, 4, 8):
            _same_bits(y[r], want, f"constant row {r}: y != beta")
            assert mean[r].item() == x[r, 0].item()
            r_ref = 1.0 / math.sqrt(EPS)
            assert abs(rstd[r].item() - r_ref) <= 2 * ULP * r_ref, (rstd[r].item(), r_ref)


@gpu
def test_layernorm_forward_rejects_bad_shapes_and_alignment(vitk):
    g_ = _gen(5)
    for D, off in ((1028, 0), (6, 0), (256, 1)):
        buf = torch.randn(4, D + 4, generator=g_, device="cuda")
        x = buf[:, off:off + D]
        gamma = torch.ones(D, device="cuda")
        beta = torch.zeros(D, device="cuda")
        y = _nan((4, D))
        with pytest.raises(vitk.VitkError):
            _ln_fwd_call(vitk, x, D + 4, gamma, beta, y, True, D, None, None, 4, D)
        assert torch.isnan(y).all(), "a rejected call wrote its output"


# ---- LayerNorm backward (vitk_layernorm_bwd) -----------------------------------------------------
# train_ops.cu, layernorm_bwd:
#     const int nv = (D / 4 + 31) / 32;
#     const bool fused = dgamma != nullptr && nv <= 6;
# fused: layernorm_bwd_fused_kernel<T, 2 | 4 | 6> (nv <= 2 | 4 | 6); otherwise
# layernorm_bwd_params_kernel<T> when dgamma is given, then layernorm_bwd_dx_kernel<T, 2|4|6|8>,
# then colsum_bf16_kernel when dx_colsum is given.
def ln_bwd_kernels(D, f32, params, colsum):
    T = "float" if f32 else "__nv_bfloat16"
    nv = (D // 4 + 31) // 32
    if params and nv <= 6:
        return {f"layernorm_bwd_fused_kernel<{T}, {2 if nv <= 2 else 4 if nv <= 4 else 6}>"}
    ks = {f"layernorm_bwd_dx_kernel<{T}, {2 if nv <= 2 else 4 if nv <= 4 else 6 if nv <= 6 else 8}>"}
    if params:
        ks.add(f"layernorm_bwd_params_kernel<{T}>")
    if colsum:
        ks.add("colsum_bf16_kernel")
    return ks


def ln_bwd_instantiations():
    out = set()
    for T in ("float", "__nv_bfloat16"):
        out |= {f"layernorm_bwd_fused_kernel<{T}, {nv}>" for nv in (2, 4, 6)}
        out |= {f"layernorm_bwd_dx_kernel<{T}, {nv}>" for nv in (2, 4, 6, 8)}
        out.add(f"layernorm_bwd_params_kernel<{T}>")
    return out


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _chunks(rows, strips, per_sm, min_rows):
    """Row chunks of the column-reduction grids (train_ops.cu: layernorm_bwd's params launch,
    colsum_bf16): one atomic add per chunk and column."""
    chunks = min(-(-_sms() * per_sm // strips), -(-rows // min_rows))
    chunks = max(chunks, 1)
    rpb = -(-rows // chunks)
    return -(-rows // rpb)


def ln_bwd_adds(D, rows, params):
    """Atomic adds per column of dgamma / dbeta / dx_colsum (train_ops.cu, layernorm_bwd)."""
    if _fused(D, params):
        return min(2 * _sms(), -(-rows // 8))
    return _chunks(rows, (D + 255) // 256, 6, 16)


def colsum_adds(M, N):
    return _chunks(M, (N + 511) // 512, 12, 32)


def _fused(D, params):
    return params and (D // 4 + 31) // 32 <= 6


# (D, rows, dy f32, params, add_resid, dx_bf16, colsum, dropout p, in place)
BWD_D = [64, 128, 132, 256, 260, 392, 400, 508, 512, 516, 764, 768, 772, 1020, 1024]
BWD_ROWS = [1, 9, 8 * 296 - 1, 8 * 296 + 1, 50432]   # 296 CTAs of 8 warps: the fused grid


def _bwd_cases():
    cases, i = [], 0
    for D in BWD_D:
        for f32 in (False, True):
            for params in (True, False):
                colsum = (_fused(D, params) or D % 8 == 0) and i % 3 != 1
                dxb = colsum or (i // 2) % 2 == 0
                cases.append((D, BWD_ROWS[i % 5], f32, params, i % 2, dxb, colsum, 0.0, False))
                i += 1
    # shapes of the earlier fp32-autograd test
    for rows, D in [(5, 64), (197, 768), (3000, 768), (40, 1024), (33, 400)]:
        for f32 in (False, True):
            cases.append((D, rows, f32, True, 1, True, False, 0.0, False))
    # dropout on the bf16 copy (fused kernel only), with and without the column sums
    for j, (D, rows) in enumerate([(64, 9), (260, 8 * 296 + 1), (400, 50432), (768, 1),
                                   (512, 8 * 296 - 1), (128, 2000)]):
        cases.append((D, rows, j % 2 == 1, True, j % 2, True, j % 3 != 2, (0.1, 0.25)[j % 2], False))
    # dy is dx_io (the detection head's norm_bwd)
    for D, colsum in ((256, True), (768, False), (1024, True)):
        cases.append((D, 8 * 296 + 1, True, True, 0, True, colsum, 0.0, True))
    return cases


BWD_CASES = _bwd_cases()


def _bwd_id(c):
    D, rows, f32, params, resid, dxb, colsum, p, inplace = c
    return (f"D{D}-r{rows}-{'f32' if f32 else 'bf16'}{'-params' if params else ''}"
            f"{'-resid' if resid else ''}{'-dxb' if dxb else ''}{'-colsum' if colsum else ''}"
            f"{f'-drop{p}' if p else ''}{'-inplace' if inplace else ''}")


_KERNEL = re.compile(r"\b((?:layernorm_bwd_\w+?_kernel|colsum_bf16_kernel)(?:<[^<>()]*>)?)")


def _ran(fn):
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return {m.group(1) for e in prof.events() for m in [_KERNEL.search(e.name)] if m}


def _drop_scale(p):
    t = int(np.float32(p) * np.float32(65536.0) + np.float32(0.5))
    return t, np.float32(65536.0) / np.float32(65536 - t)


def _keep_mask(vitk, p, seed, site, layer, n):
    keep = torch.empty(n, dtype=torch.uint8, device="cuda")
    vitk._lib.check(vitk._lib.lib().vitk_dropout_keep_mask(p, seed, site, layer, n, keep.data_ptr(),
                                                           _stream()))
    return keep.bool()


class _BwdInputs:
    def __init__(self, case, seed):
        D, rows, f32, params, resid, dxb, colsum, p, inplace = case
        g_ = _gen(seed)
        self.x = torch.randn(rows, D, generator=g_, device="cuda") * 2 + 0.5
        # statistics as the forward would save them (fp32); the reference takes them as given
        self.mean = self.x.mean(1)
        self.rstd = torch.rsqrt(self.x.var(1, unbiased=False) + EPS)
        self.gamma = torch.randn(D, generator=g_, device="cuda")
        self.dy = torch.randn(rows, D, generator=g_, device="cuda").to(
            torch.float32 if f32 else torch.bfloat16)
        self.resid = torch.randn(rows, D, generator=g_, device="cuda") if resid else None
        self.dg0 = torch.randn(D, generator=g_, device="cuda") if params else None
        self.db0 = torch.randn(D, generator=g_, device="cuda") if params else None
        self.cs0 = torch.randn(D, generator=g_, device="cuda") if colsum else None


def _bwd_call(vitk, inp, case, site=2, layer=3, seed=1234):
    """One vitk_layernorm_bwd call on fresh output buffers; returns them."""
    D, rows, f32, params, resid, dxb, colsum, p, inplace = case
    if inplace:
        dx = inp.dy.clone()
    elif resid:
        dx = inp.resid.clone()
    else:
        dx = _nan((rows, D))          # not read without add_resid
    dy = dx if inplace else inp.dy
    out = dict(dx=dx,
               dxb=_nan((rows, D), torch.bfloat16) if dxb else None,
               dg=inp.dg0.clone() if params else None, db=inp.db0.clone() if params else None,
               cs=None)
    if colsum:
        out["cs_buf"] = _nan((D + 8,))
        out["cs_buf"][:D] = inp.cs0
        out["cs"] = out["cs_buf"][:D]

    def call():
        vitk._lib.check(vitk._lib.lib().vitk_layernorm_bwd(
            dy.data_ptr(), 1 if f32 else 0, inp.x.data_ptr(), inp.mean.data_ptr(),
            inp.rstd.data_ptr(), inp.gamma.data_ptr(), dx.data_ptr(), resid, _p(out["dxb"]),
            _p(out["dg"]), _p(out["db"]), rows, D, _p(out["cs"]), p, seed, site, layer, _stream()))
    return out, call


def _ln_bwd_ref(inp):
    x64, dy64 = inp.x.double(), inp.dy.double()
    mu, rs = inp.mean.double()[:, None], inp.rstd.double()[:, None]
    g64 = inp.gamma.double()
    xh = (x64 - mu) * rs
    gg = dy64 * g64
    s1 = gg.mean(1, keepdim=True)
    s2 = (gg * xh).mean(1, keepdim=True)
    dx = rs * (gg - s1 - xh * s2)
    mag = rs * (gg.abs() + gg.abs().mean(1, keepdim=True)
                + xh.abs() * (gg * xh).abs().mean(1, keepdim=True))
    if inp.resid is not None:
        dx = dx + inp.resid.double()
        mag = mag + inp.resid.double().abs()
    dgam, dgam_mag = (dy64 * xh).sum(0), (dy64 * xh).abs().sum(0)
    dbet, dbet_mag = dy64.sum(0), dy64.abs().sum(0)
    return dx, mag, dgam, dgam_mag, dbet, dbet_mag


@gpu
@pytest.mark.parametrize("case", BWD_CASES, ids=[_bwd_id(c) for c in BWD_CASES])
def test_layernorm_backward(vitk, case):
    D, rows, f32, params, resid, dxb, colsum, p, inplace = case
    inp = _BwdInputs(case, D * 7 + rows + 3 * f32)
    out, call = _bwd_call(vitk, inp, case)
    call()
    family = ("layernorm_bwd_fused" if _fused(D, params) else "layernorm_bwd_dx")
    c = C_ROUND * U24
    dx_ref, mag, dgam, dgam_mag, dbet, dbet_mag = _ln_bwd_ref(inp)
    dx = out["dx"]
    _check(family, "dx_io", dx, dx_ref, c * mag)
    if dxb:
        if p:
            keep = _keep_mask(vitk, p, 1234, 2, 3, rows * D).view(rows, D)
            _, scale = _drop_scale(p)
            sc = torch.tensor(float(scale), dtype=torch.float32, device="cuda")
            want = torch.where(keep, dx * sc, torch.zeros_like(dx)).bfloat16()
        else:
            want = dx.bfloat16()
        _same_bits(out["dxb"], want, "dx_bf16 against bf16(mask(dx_io))")
    if params:
        pf = family if family == "layernorm_bwd_fused" else "layernorm_bwd_params"
        ca = c + U24 * ln_bwd_adds(D, rows, params)
        _check(pf, "dgamma", out["dg"], inp.dg0.double() + dgam, ca * (inp.dg0.double().abs() + dgam_mag))
        _check(pf, "dbeta", out["db"], inp.db0.double() + dbet, ca * (inp.db0.double().abs() + dbet_mag))
    if colsum:
        y = out["dxb"].double()
        ref = inp.cs0.double() + y.sum(0)
        _check(family if _fused(D, params) else "colsum", "dx_colsum", out["cs"], ref,
               (c + U24 * (ln_bwd_adds(D, rows, params) if _fused(D, params) else colsum_adds(rows, D)))
               * (inp.cs0.double().abs() + y.abs().sum(0)))
        assert torch.isnan(out["cs_buf"][D:]).all(), "dx_colsum: wrote past column D"


_DISPATCH_CHILD = """
import json, sys
sys.path.insert(0, sys.argv[1])
import vitk
from tests import test_train_rowops_gpu as T
ran = {}
for case in T.BWD_CASES:
    inp = T._BwdInputs(case, 0)
    _, call = T._bwd_call(vitk, inp, case)
    ran[T._bwd_id(case)] = sorted(T._ran(call))
print(json.dumps(ran))
"""


@gpu
def test_layernorm_backward_runs_the_predicted_kernels():
    """The kernels torch.profiler records for every case of test_layernorm_backward are the ones
    ln_bwd_kernels predicts.  Profiled in a process of its own: after the rest of the suite has
    run in the same process, torch.profiler has been seen to record no kernels at all."""
    import json
    import subprocess
    import sys
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + ["-c", _DISPATCH_CHILD,
                                                                           str(ROOT)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-4000:]
    ran = json.loads(r.stdout.strip().splitlines()[-1])
    for case in BWD_CASES:
        want = sorted(ln_bwd_kernels(case[0], case[2], case[3], case[6]))
        assert ran[_bwd_id(case)] == want, f"{_bwd_id(case)}: ran {ran[_bwd_id(case)]}"


@gpu
@pytest.mark.parametrize("D,params", [(1024, True), (256, False), (768, False)])
def test_layernorm_backward_rejects_dropout_outside_the_fused_kernel(vitk, D, params):
    case = (D, 9, False, params, 0, True, False, 0.1, False)
    inp = _BwdInputs(case, D)
    out, call = _bwd_call(vitk, inp, case)
    with pytest.raises(vitk.VitkError):
        call()
    assert torch.isnan(out["dx"]).all() and torch.isnan(out["dxb"].float()).all()
    if params:
        _same_bits(out["dg"], inp.dg0, "dgamma")
        _same_bits(out["db"], inp.db0, "dbeta")


@gpu
@pytest.mark.parametrize("f32", [False, True], ids=["bf16", "f32"])
def test_layernorm_backward_colsum_outside_the_fused_kernel_at_d772(vitk, f32):
    """D = 772 takes the two-kernel path, whose column sums need D % 8 == 0: the call must be
    refused before anything is written."""
    case = (772, 33, f32, True, 1, True, True, 0.0, False)
    inp = _BwdInputs(case, 772)
    out, call = _bwd_call(vitk, inp, case)
    with pytest.raises(vitk.VitkError):
        call()
    _same_bits(out["dx"], inp.resid, "dx_io")
    _same_bits(out["dg"], inp.dg0, "dgamma")
    _same_bits(out["db"], inp.db0, "dbeta")
    _same_bits(out["cs"], inp.cs0, "dx_colsum")
    assert torch.isnan(out["dxb"].float()).all()


def test_layernorm_backward_cases_cover_every_instantiation():
    """CPU: the dispatch rule ln_bwd_kernels restates is the one in train_ops.cu, and the case
    list reaches all 16 kernel instantiations."""
    text = (CSRC / "train_ops.cu").read_text()
    assert "const int nv = (D / 4 + 31) / 32;" in text
    assert "const bool fused = dgamma != nullptr && nv <= 6;" in text
    assert "if (nv <= 2) VITK_LN_FUSED(float, dyf, 2);" in text
    assert "else if (nv <= 6) VITK_LN_BWD(float, dyf, 6);" in text
    # the launch geometry ln_bwd_adds and colsum_adds restate
    assert "int fgrid = sm_count() * 2;" in text
    assert "int chunks = (sm_count() * 6 + strips - 1) / strips;" in text
    assert "int chunks = (sm_count() * 12 + strips - 1) / strips;" in text
    hit = set()
    for D, rows, f32, params, resid, dxb, colsum, p, inplace in BWD_CASES:
        hit |= ln_bwd_kernels(D, f32, params, colsum)
    want = ln_bwd_instantiations()
    assert len(want) == 16
    assert not want - hit, f"no case runs {sorted(want - hit)}"
    assert "colsum_bf16_kernel" in hit
    # dropout, dx_colsum on both paths, in place, every row count
    assert any(c[7] for c in BWD_CASES) and any(c[8] for c in BWD_CASES)
    assert any(c[6] and _fused(c[0], c[3]) for c in BWD_CASES)
    assert any(c[6] and not _fused(c[0], c[3]) for c in BWD_CASES)
    assert set(BWD_ROWS) <= {c[1] for c in BWD_CASES}


# ---- classifier loss tail (vitk_classifier_head_loss_backward) ---------------------------------
CLS_D = [64, 100, 400, 768, 1024]
CLS_C = [1, 2, 6, 81, 1000]
CLS_B = [1, 3, 8, 33, 257]


def _cls_cases():
    cases = []
    for i, D in enumerate(CLS_D):
        for j, Cn in enumerate(CLS_C):
            B = CLS_B[(i + j) % 5]
            cases.append((D, Cn, B, 197 if (i + j) % 2 == 0 else 198,
                          1.0 / B if j % 2 == 0 else 1.0 / 64, (i + 2 * j) % 3 != 0))
    return cases


CLS_CASES = _cls_cases()


@gpu
@pytest.mark.parametrize("D,n_cls,B,N,scale,with_dw", CLS_CASES,
                         ids=[f"D{D}-C{c}-B{b}-N{n}-s{s:.3g}{'-dw' if w else ''}"
                              for D, c, b, n, s, w in CLS_CASES])
def test_classifier_head_loss_backward(vitk, D, n_cls, B, N, scale, with_dw):
    g_ = _gen(D * 1009 + n_cls * 7 + B)
    c = C_ROUND * U24
    scale = float(np.float32(scale))
    # inputs: only the CLS rows (b * N) of x hold values
    xc = torch.randn(B, D, generator=g_, device="cuda") * 1.5 + 0.3
    tie = 2 if B >= 3 else None
    if tie is not None:
        xc[tie] = 0.5                     # constant row: feat = beta, logits = head_w beta + b
    gamma = 1 + 0.2 * torch.randn(D, generator=g_, device="cuda")
    beta = 0.3 * torch.randn(D, generator=g_, device="cuda")
    W = torch.randn(n_cls, D, generator=g_, device="cuda") * (2.0 / math.sqrt(D))
    # head bias: nearly tied logits for the constant row, one class 40 below the rest
    hb = (-(W.double() @ beta.double()) + 1e-3 * torch.randn(n_cls, generator=g_, device="cuda",
                                                               dtype=torch.float64)).float()
    k40 = n_cls // 2
    if n_cls >= 2:
        hb[k40] -= 40.0
    labels = torch.randint(0, n_cls, (B,), generator=g_, device="cuda")
    labels[0] = 0
    labels[-1] = n_cls - 1
    if B >= 3 and n_cls >= 2:
        labels[1] = k40                   # label logit ~40 below the maximum
    x = _Rows(B * N, D, torch.float32)
    x.view.view(B, N, D)[:, 0] = xc
    dx = _Rows(B * N, D, torch.float32).snapshot()
    dxb = _Rows(B * N, D, torch.bfloat16).snapshot()
    cls_rows = torch.zeros(B * N, D, dtype=torch.bool, device="cuda")
    cls_rows.view(B, N, D)[:, 0] = True
    logits = _nan((B, n_cls))
    loss = torch.full((1,), 0.25, device="cuda")
    feat = _nan((B, D))
    dl = _nan((B, n_cls))
    dg0 = torch.randn(D, generator=g_, device="cuda")
    db0 = torch.randn(D, generator=g_, device="cuda")
    dg, db = dg0.clone(), db0.clone()
    dW0 = torch.randn(n_cls, D, generator=g_, device="cuda") if with_dw else None
    dhb0 = torch.randn(n_cls, generator=g_, device="cuda") if with_dw else None
    dW = dW0.clone() if with_dw else None
    dhb = dhb0.clone() if with_dw else None
    vitk._lib.check(vitk._lib.lib().vitk_classifier_head_loss_backward(
        x.buf.data_ptr(), N * D, gamma.data_ptr(), beta.data_ptr(), W.data_ptr(), hb.data_ptr(),
        labels.data_ptr(), scale, EPS, B, D, n_cls, logits.data_ptr(), loss.data_ptr(),
        feat.data_ptr(), dl.data_ptr(), dx.buf.data_ptr(), dxb.buf.data_ptr(), dg.data_ptr(),
        db.data_ptr(), _p(dW), _p(dhb), _stream()))
    _untouched(dx.buf, dx.before, ~cls_rows, "dx outside the CLS rows")
    _untouched(dxb.buf, dxb.before, ~cls_rows, "dx_bf16 outside the CLS rows")
    dx_cls = dx.buf.view(B, N, D)[:, 0]
    _same_bits(dxb.buf.view(B, N, D)[:, 0], dx_cls.bfloat16(), "dx_bf16 against bf16(dx)")

    # fp64 autograd of LayerNorm -> Linear -> scale * summed cross-entropy
    x64 = xc.double().requires_grad_(True)
    g64 = gamma.double().requires_grad_(True)
    be64 = beta.double().requires_grad_(True)
    W64 = W.double().requires_grad_(True)
    hb64 = hb.double().requires_grad_(True)
    mu = x64.mean(1, keepdim=True)
    var = ((x64 - mu) ** 2).mean(1, keepdim=True)
    rstd = 1.0 / torch.sqrt(var + EPS)
    xh = (x64 - mu) * rstd
    f64 = xh * g64 + be64
    f64.retain_grad()
    lg64 = f64 @ W64.t() + hb64
    lg64.retain_grad()
    loss64 = scale * F.cross_entropy(lg64, labels, reduction="sum")
    loss64.backward()

    # bounds, stage by stage (module docstring)
    with torch.no_grad():
        xh, f, lg, rstd, var = xh.detach(), f64.detach(), lg64.detach(), rstd.detach(), var.detach()
        ga, Wa = gamma.double().abs(), W.double().abs()
        mu_err = c * xc.double().abs().mean(1, keepdim=True)
        rstd_rel = c + 2 * ULP + 0.5 * mu_err ** 2 / (var + EPS)
        e_xh = c * xh.abs() + mu_err * rstd + rstd_rel * xh.abs()
        e_feat = c * (xh.abs() * ga + beta.double().abs()) + e_xh * ga
        e_lg = c * (f.abs() @ Wa.t() + hb.double().abs()) + e_feat @ Wa.t()
        m = lg.max(1, keepdim=True).values
        lse = torch.logsumexp(lg, 1, keepdim=True)
        logz = lse - m
        pr = torch.softmax(lg, 1)
        # expf 2 ulp per term, logf 1 ulp, rounding of l - max inside the exponent
        # z = sum_c expf(l_c - m), accumulated by one thread in class order
        ez = torch.exp(lg - m)
        z_partials = torch.cumsum(ez, 1).sum(1, keepdim=True) / ez.sum(1, keepdim=True)
        e_lse = ((pr * e_lg).sum(1, keepdim=True) + c * (m.abs() + logz.abs() + 1) + U24 * z_partials
                 + c * (pr * (lg - m).abs()).sum(1, keepdim=True) + 2 * ULP + ULP * logz.abs())
        onehot = F.one_hot(labels, n_cls).double()
        lab_lg = lg.gather(1, labels[:, None])
        e_lab = e_lg.gather(1, labels[:, None])
        e_loss = (scale * (e_lse + e_lab).sum() + c * scale * (lse.abs() + lab_lg.abs()).sum()
                  + c * 0.25 + U24 * B * (0.25 + scale * (lse - lab_lg).abs().sum()))
        e_p = pr * (e_lg + e_lse + c * (lg.abs() + lse.abs()) + 2 * ULP)
        dl64 = lg64.grad
        e_dl = scale * (e_p + c * (pr + onehot))
        df = f64.grad
        e_df = c * (dl64.abs() @ Wa) + e_dl @ Wa
        ca = c + U24 * B         # one atomic add per image
        e_dg = (ca * (dg0.double().abs() + (df * xh).abs().sum(0))
                + (e_df * xh.abs() + df.abs() * e_xh).sum(0))
        e_db = ca * (db0.double().abs() + df.abs().sum(0)) + e_df.sum(0)
        gg = df * gamma.double()
        e_gg = e_df * ga + c * gg.abs()
        s2 = (gg * xh).mean(1, keepdim=True)
        e_s1 = e_gg.mean(1, keepdim=True) + c * gg.abs().mean(1, keepdim=True)
        e_s2 = (e_gg * xh.abs() + gg.abs() * e_xh).mean(1, keepdim=True) \
            + c * (gg * xh).abs().mean(1, keepdim=True)
        dx_ref = x64.grad
        e_dx = (rstd * (e_gg + e_s1 + e_xh * s2.abs() + xh.abs() * e_s2) + rstd_rel * dx_ref.abs()
                + c * rstd * (gg.abs() + gg.abs().mean(1, keepdim=True)
                              + xh.abs() * (gg * xh).abs().mean(1, keepdim=True)))

    fam = "cls_loss_bwd"
    _check(fam, "feat", feat, f, e_feat)
    _check(fam, "logits", logits, lg, e_lg)
    _check(fam, "loss", loss, 0.25 + loss64.detach().reshape(1), e_loss.reshape(1))
    _check(fam, "dlogits", dl, dl64, e_dl)
    _check(fam, "dx", dx_cls, dx_ref, e_dx)
    _check(fam, "dgamma", dg, dg0.double() + g64.grad, e_dg)
    _check(fam, "dbeta", db, db0.double() + be64.grad, e_db)
    if with_dw:
        e_dW = (c * (dW0.double().abs() + dl64.abs().t() @ f.abs()) + e_dl.t() @ f.abs()
                + dl64.abs().t() @ e_feat)
        e_dhb = c * (dhb0.double().abs() + dl64.abs().sum(0)) + e_dl.sum(0)
        _check("head_wgrad", "dhead_w", dW, dW0.double() + W64.grad, e_dW)
        _check("head_wgrad", "dhead_b", dhb, dhb0.double() + hb64.grad, e_dhb)


# ---- weighted cross-entropy (vitk_weighted_cross_entropy) -------------------------------------
WCE_ROWS = [1, 255, 256, 257, 6400]
WCE_C = [1, 2, 7, 81, 4096]


def _wce_cases():
    cases = []
    for i, rows in enumerate(WCE_ROWS):
        for j, Cn in enumerate(WCE_C):
            cases.append((rows, Cn, (i + j) % 2 == 0, 1.0 if j % 2 == 0 else 0.5,
                          ("none", "loss", "dlogits")[(i + 2 * j) % 3]))
    return cases


WCE_CASES = _wce_cases()


def _wce_call(vitk, logits, targets, weight, loss, dl, gs):
    rows, Cn = logits.shape
    sums = torch.empty(2, device="cuda")
    vitk._lib.check(vitk._lib.lib().vitk_weighted_cross_entropy(
        logits.data_ptr(), targets.data_ptr(), _p(weight), rows, Cn, _p(loss), sums.data_ptr(),
        _p(dl), gs, _stream()))


@gpu
@pytest.mark.parametrize("rows,n_cls,weighted,gs,null", WCE_CASES,
                         ids=[f"r{r}-C{c}{'-w' if w else ''}-gs{g}-no_{n}" for r, c, w, g, n in WCE_CASES])
def test_weighted_cross_entropy(vitk, rows, n_cls, weighted, gs, null):
    g_ = _gen(rows * 13 + n_cls)
    c = C_ROUND * U24
    logits = torch.randn(rows, n_cls, generator=g_, device="cuda") * 3
    wide = torch.arange(rows, device="cuda") % 4 == 3
    logits[wide] = (torch.rand(int(wide.sum()), n_cls, generator=g_, device="cuda") * 2 - 1) * 1e4
    targets = torch.randint(0, n_cls, (rows,), generator=g_, device="cuda")
    ign = torch.rand(rows, generator=g_, device="cuda") < 0.2
    ign[0] = False
    targets[ign] = -100
    weight = None
    if weighted:
        weight = 0.5 + torch.rand(n_cls, generator=g_, device="cuda")
        weight[-1] = 0.1                 # background
    loss = None if null == "loss" else _nan((1,))
    dl = None if null == "dlogits" else _nan((rows, n_cls))
    _wce_call(vitk, logits, targets, weight, loss, dl, gs)

    l64 = logits.double().requires_grad_(True)
    w64 = weight.double() if weighted else None
    ref = F.cross_entropy(l64, targets, weight=w64, ignore_index=-100)
    ref.backward()
    with torch.no_grad():
        l = l64.detach()
        valid = targets >= 0
        t = targets.clamp_min(0)
        wt = (w64[t] if weighted else torch.ones(rows, dtype=torch.float64, device="cuda")) * valid
        m = l.max(1, keepdim=True).values
        y = l - m
        ez = torch.exp(y)
        e_term = ez * ((2 + torch.floor(1.173 * y.abs())) * ULP + U24 * y.abs()) + TINY  # __expf
        z = ez.sum(1, keepdim=True)
        e_z = e_term.sum(1, keepdim=True) + c * z + U24 * torch.cumsum(ez, 1).sum(1, keepdim=True)
        logz = torch.log(z)
        e_logf = torch.where((z >= 0.5) & (z <= 2), torch.full_like(z, 2.0 ** -21.41),
                             3 * ULP * logz.abs())                                   # __logf
        lt = l.gather(1, t[:, None])
        nll = m + logz - lt
        e_nll = (e_z / z + e_logf + c * (m.abs() + logz.abs() + lt.abs()))[:, 0]
        sw = wt.sum()
        e_sw = c * sw
        e_loss = ((wt * e_nll).sum() + c * (wt * nll[:, 0].abs()).sum()) / sw \
            + ref.detach().abs() * (e_sw / sw + U24)
        p = ez / z
        onehot = F.one_hot(t, n_cls).double() * valid[:, None]
        k = gs * wt / sw
        e_p = e_term / z + p * (e_z / z + 2 * U24)
        dl_ref = gs * l64.grad
        e_dl = k[:, None] * (e_p + c * (p + onehot)) + dl_ref.abs() * (e_sw / sw + 2 * U24)
    if loss is not None:
        _check("wce", "loss", loss, ref.detach().reshape(1), e_loss.reshape(1))
    if dl is not None:
        _check("wce", "dlogits", dl, dl_ref, e_dl)
        assert (_bits(dl[~valid]) == 0).all(), "dlogits of an ignored row must be +0"


@gpu
def test_weighted_cross_entropy_all_ignored(vitk):
    """Every target ignored: the loss is 0 / 0 = NaN, as in torch, and the gradient is zero."""
    rows, n_cls = 300, 7
    logits = torch.randn(rows, n_cls, generator=_gen(3), device="cuda")
    targets = torch.full((rows,), -100, dtype=torch.long, device="cuda")
    loss, dl = _nan((1,)), _nan((rows, n_cls))
    _wce_call(vitk, logits, targets, None, loss, dl, 1.0)
    assert math.isnan(F.cross_entropy(logits.double(), targets, ignore_index=-100).item())
    assert math.isnan(loss.item())
    assert (_bits(dl) == 0).all()


# ---- AdamW and the non-finite guard ------------------------------------------------------------
ADAM_N = [1, 2, 3, 4, 5, 1023, 4099, (1 << 20) + 3]
ADAM_STEPS = [1, 2, 1000]
LR, BETAS, ADAM_EPS, WD = 1e-3, (0.9, 0.999), 1e-8, 1e-2


def _adam_cases():
    return [(n, s, 1.0 if (i + j) % 2 == 0 else 2.0 ** -16, (i + j) % 3 != 0)
            for i, n in enumerate(ADAM_N) for j, s in enumerate(ADAM_STEPS)]


ADAM_CASES = _adam_cases()


def _f32(v):
    return float(np.float32(v))


def _adam_state(n, step, gs, seed):
    g_ = _gen(seed)
    p = torch.randn(n, generator=g_, device="cuda")
    g = torch.randn(n, generator=g_, device="cuda") * (0.01 / gs)     # gradients of a scaled loss
    if step == 1:
        m, v = torch.zeros(n, device="cuda"), torch.zeros(n, device="cuda")
    else:
        m = torch.randn(n, generator=g_, device="cuda") * 1e-3
        v = (torch.randn(n, generator=g_, device="cuda") * 1e-2) ** 2
    return p, g, m, v


def _adam_call(vitk, p, g, m, v, shadow, step, gs, guard=None):
    L = vitk._lib.lib()
    args = (p.data_ptr(), g.data_ptr(), m.data_ptr(), v.data_ptr(), _p(shadow), p.numel(), LR,
            BETAS[0], BETAS[1], ADAM_EPS, WD, step, gs)
    if guard is None:
        vitk._lib.check(L.vitk_adamw_step(*args, _stream()))
    else:
        vitk._lib.check(L.vitk_adamw_step_guarded(*args, guard.data_ptr(), _stream()))


def _adam_ref(p, g, m, v, t, gs):
    """fp64 AdamW with the fp32 constants the launcher hands the kernel; bounds of p, m, v."""
    c = C_ROUND * U24
    decay = _f32(1.0 - LR * WD)
    b1, b2, omb1, omb2 = _f32(BETAS[0]), _f32(BETAS[1]), _f32(1 - BETAS[0]), _f32(1 - BETAS[1])
    step_size = _f32(LR / (1.0 - BETAS[0] ** t))
    isb = _f32(1.0 / math.sqrt(1.0 - BETAS[1] ** t))
    gr = g.double() * _f32(gs)
    m64, v64, p64 = m.double(), v.double(), p.double()
    m1 = b1 * m64 + omb1 * gr
    v1 = b2 * v64 + omb2 * gr * gr
    den = torch.sqrt(v1) * isb + _f32(ADAM_EPS)
    upd = step_size * m1 / den
    p1 = p64 * decay - upd
    M_m = b1 * m64.abs() + omb1 * gr.abs()
    M_p = (p64 * decay).abs() + upd.abs() + 2 * step_size * M_m / den
    return p1, c * M_p, m1, c * M_m, v1, c * v1


@gpu
@pytest.mark.parametrize("n,step,gs,with_shadow", ADAM_CASES,
                         ids=[f"n{n}-t{s}-gs{g:g}{'-shadow' if w else ''}" for n, s, g, w in ADAM_CASES])
def test_adamw(vitk, n, step, gs, with_shadow):
    p, g, m, v = _adam_state(n, step, gs, n + step)
    p1, m1, v1 = p.clone(), m.clone(), v.clone()
    shadow = _nan((n,), torch.bfloat16) if with_shadow else None
    _adam_call(vitk, p1, g, m1, v1, shadow, step, gs)
    pr, pb, mr, mb, vr, vb = _adam_ref(p, g, m, v, step, gs)
    _check("adamw", "p", p1, pr, pb)
    _check("adamw", "exp_avg", m1, mr, mb)
    _check("adamw", "exp_avg_sq", v1, vr, vb)
    if with_shadow:
        _same_bits(shadow, p1.bfloat16(), "shadow against bf16(p)")


@gpu
@pytest.mark.parametrize("n", [5, 4099, (1 << 20) + 3])
def test_adamw_guarded(vitk, n):
    gs = 2.0 ** -16
    p, g, m, v = _adam_state(n, 2, gs, n)
    # flag set: nothing moves
    p1, m1, v1 = p.clone(), m.clone(), v.clone()
    shadow = _nan((n,), torch.bfloat16)
    guard = torch.tensor([1, 0], dtype=torch.int32, device="cuda")
    _adam_call(vitk, p1, g, m1, v1, shadow, 7, gs, guard)
    for a, b, what in ((p1, p, "p"), (m1, m, "exp_avg"), (v1, v, "exp_avg_sq")):
        _same_bits(a, b, f"guarded step with the flag set changed {what}")
    assert torch.isnan(shadow.float()).all()
    assert guard.tolist() == [1, 0]
    # k skipped steps: the bias corrections of step - k, evaluated on the device
    for step, k in ((1000, 3), (2, 1), (5, 4)):
        p1, m1, v1 = p.clone(), m.clone(), v.clone()
        shadow = _nan((n,), torch.bfloat16)
        guard = torch.tensor([0, k], dtype=torch.int32, device="cuda")
        _adam_call(vitk, p1, g, m1, v1, shadow, step, gs, guard)
        p2, m2, v2 = p.clone(), m.clone(), v.clone()
        _adam_call(vitk, p2, g, m2, v2, None, step - k, gs)
        _same_bits(m1, m2, "exp_avg of a guarded step")
        _same_bits(v1, v2, "exp_avg_sq of a guarded step")
        pr, pb, *_ = _adam_ref(p, g, m, v, step - k, gs)
        _check("adamw", f"p, step {step} with {k} skipped", p1, pr, pb)
        _same_bits(shadow, p1.bfloat16(), "shadow against bf16(p)")
        assert guard.tolist() == [0, k]


def _scan(vitk, g, guard, reset):
    vitk._lib.check(vitk._lib.lib().vitk_grad_guard_scan(g.data_ptr(), g.numel(), guard.data_ptr(),
                                                         reset, _stream()))


@gpu
@pytest.mark.parametrize("n", [1, 3, 4, 5, 7, 8, 4099, (1 << 20) + 3])
def test_grad_guard_scan(vitk, n):
    g0 = torch.randn(n, generator=_gen(n), device="cuda") * 100
    nvec = n // 4
    pos = {0, n - 1}
    if nvec:
        j = nvec // 2
        pos |= {4 * j, 4 * j + 1, 4 * j + 2, 4 * j + 3}
    if n % 4:
        pos |= set(range(4 * nvec, n))
    guard = torch.zeros(2, dtype=torch.int32, device="cuda")
    for i in sorted(pos):
        for val in (math.inf, -math.inf, math.nan):
            g = g0.clone()
            g[i] = val
            _scan(vitk, g, guard, 1)
            assert guard[0].item() == 1, f"{val} at {i} of {n} not flagged"
    _scan(vitk, g0, guard, 1)
    assert guard[0].item() == 0
    fmax = torch.full((n,), torch.finfo(torch.float32).max, device="cuda")
    fmax[::2] *= -1
    _scan(vitk, fmax, guard, 1)
    assert guard[0].item() == 0, "FLT_MAX flagged as non-finite"
    # reset = 0 keeps an earlier flag; finish counts flagged steps only
    guard.zero_()
    bad = g0.clone()
    bad[n - 1] = math.nan
    L = vitk._lib.lib()
    for flagged in (True, False, True, True, False):
        _scan(vitk, bad if flagged else g0, guard, 1)
        _scan(vitk, g0, guard, 0)
        assert guard[0].item() == int(flagged)
        vitk._lib.check(L.vitk_grad_guard_finish(guard.data_ptr(), _stream()))
    assert guard.tolist() == [0, 3]


# ---- bias-gradient column sums (vitk_colsum_bf16) ------------------------------------------------
COLSUM_CASES = [(M, N, (i + j) % 2 == 1) for i, M in enumerate([1, 31, 32, 33, 6304])
                for j, N in enumerate([8, 504, 512, 520, 2304])]
COLSUM_CASES += [(100, 768, False), (6304, 3072, False), (37, 2304, True), (5000, 400, False)]


@gpu
@pytest.mark.parametrize("M,N,pitched", COLSUM_CASES,
                         ids=[f"M{M}-N{N}{'-ld' if p else ''}" for M, N, p in COLSUM_CASES])
def test_colsum(vitk, M, N, pitched):
    g_ = _gen(M + N)
    ld = N + 8 if pitched else N
    y = _Rows(M, N, torch.bfloat16, ld).fill(torch.randn(M, N, generator=g_, device="cuda") * 3)
    out0 = torch.randn(N, generator=g_, device="cuda")
    out_buf = _nan((N + 8,))
    out_buf[:N] = out0
    vitk._lib.check(vitk._lib.lib().vitk_colsum_bf16(y.buf.data_ptr(), ld, M, N, out_buf.data_ptr(),
                                                     _stream()))
    y64 = y.view.double()
    _check("colsum", "out", out_buf[:N], out0.double() + y64.sum(0),
           (C_ROUND + colsum_adds(M, N)) * U24 * (out0.double().abs() + y64.abs().sum(0)))
    assert torch.isnan(out_buf[N:]).all(), "colsum wrote past column N"


@gpu
def test_colsum_rejects_a_misaligned_view(vitk):
    buf = torch.randn(16, 528, device="cuda").bfloat16()
    out = torch.zeros(512, device="cuda")
    with pytest.raises(vitk.VitkError):
        vitk.ops.colsum(buf[:, 4:516], out)       # 8 bytes past a 16-byte boundary
    assert (out == 0).all()
