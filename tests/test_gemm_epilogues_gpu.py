"""Every epilogue of the tcgen05 GEMM (gemm_sm100.cu) against an fp64 reference of the same bf16
operands, at the tile, layout and activation edges: both BLOCK_N widths with ragged last tiles,
M around the CTA-pair boundaries, K below one k-block and across many turns of the stage ring,
strided operands, outputs at 16-byte aligned and unaligned column offsets, out-of-place
residuals, bias=None, alpha / beta, the MN-major weight-gradient form with split-K, the residual
epilogue with row statistics and the LayerNorm-folded consumer.

Each element is held to |out - ref| <= acc_tol + approx(x) + out_rounding (`_bound`):
  acc_tol      = C_ACC * 2^-24 * (|alpha| |A| @ |B|^T + |bias| + |beta C0| + |resid|), times the
                 activation's largest slope (1.13 for the GELUs and gelu');
  approx(x)    = the documented error of the epilogue's activation (`_approx`);
  out_rounding = one bf16 ulp of |ref| for bf16 outputs (either neighbour), 0 for fp32 outputs.
The activation sweeps feed exactly known pre-activations, so there the bound is approx + rounding
alone and the saturated tails must come out exact.
"""
import math
from pathlib import Path

import pytest
import torch

# acc_tol in units of 2^-24 of the magnitude sum.  Observed worst on a B200 (1000 W) over this
# file: err / (2^-24 * magnitude) = 9.95 (EPI_F32, K = 4104, BLOCK_N 128); the worst per path is
# printed at the end of the module with -s.
C_ACC = 16
U24 = 2.0 ** -24
GELU_SLOPE = 1.13           # max of d/dx [x Phi(x)] (at x = sqrt 2)
SAT = 9.0                   # |x| from which the activations must have saturated

MODES = [(1, False), (2, False), (1, True), (2, True)]
MODE_IDS = ["cta1-tma", "cta2-tma", "cta1-direct", "cta2-direct"]

EPI_IDS = {"bf16": 0, "gelu": 1, "resid": 2, "f32": 3, "dgelu": 4, "gelu_tanh": 6, "relu": 7,
           "resid_stats": 8}
GELU_FAMILY = ("gelu", "gelu_tanh", "relu")


@pytest.fixture(params=MODES, ids=MODE_IDS)
def gemm_mode(request, vitk):
    """Single-CTA and CTA-pair tiles, with the TMA-staged and the direct epilogue requested."""
    ctas, direct = request.param
    vitk._lib.set_gemm_cta_group(ctas)
    vitk._lib.set_gemm_direct_epilogue(direct)
    yield request.param
    vitk._lib.set_gemm_cta_group(0)
    vitk._lib.set_gemm_direct_epilogue(False)


# ---- which kernel instantiation a call runs ----------------------------------------------------
# gemm_sm100.cu:1207-1210 (dispatch_tile):
#     // 256-wide tiles unless they would waste more than a 128-wide tiling does.
#     const int waste256 = ((p.N + 255) / 256) * 256 - p.N;
#     const int waste128 = ((p.N + 127) / 128) * 128 - p.N;
#     const bool n128 = waste128 < waste256;
# A tie goes to 256 (N = 136, 200, 744).
def block_n(N):
    waste256 = -(-N // 256) * 256 - N
    waste128 = -(-N // 128) * 128 - N
    return 128 if waste128 < waste256 else 256


def _out_align_ok(layout):
    return layout != "ldo_unaligned"


def predict(case, mode):
    """(epilogue, BLOCK_N, CTAS, TMA_EPI, MN) of gemm_tn_kernel that `case` runs under `mode`,
    following gemm_bf16_tn, dispatch, tma_epilogue_ok and dispatch_tile."""
    ctas, direct = mode
    kind = case[0]
    if kind == "wgrad":                 # MN-major: TMA store / reduce-add only, whatever is forced
        _, T, O, I, split, alpha, acc = case
        return ("f32", block_n(I), ctas, True, True)
    if kind == "stats":                 # TMA only
        _, M, N, K, layout = case
        return ("resid_stats", block_n(N), ctas, True, False)
    if kind == "folded":                # TMA only; the folded path of the bf16 instantiations
        _, epi, M, N, K = case
        return (epi, block_n(N), ctas, True, False)
    _, epi, M, N, K, layout, opt = case
    tma = not direct and _out_align_ok(layout)
    if epi == "resid":
        tma = tma and layout != "oop"            # out-of-place residual: direct
    if epi == "f32":
        tma = tma and opt[1] in (0.0, 1.0)       # beta outside {0, 1}: direct
    if epi == "dgelu" and ctas == 1:
        tma = False                               # kTma1: no room for the third slab
    return (epi, block_n(N), ctas, tma, False)


def reachable_instantiations():
    """The 62 gemm_tn_kernel instantiations gemm_bf16_tn can launch."""
    out = set()
    for epi in ("bf16", "gelu", "gelu_tanh", "relu", "resid", "f32", "dgelu"):
        for bn in (128, 256):
            for ctas in (1, 2):
                for tma in (False, True):
                    if epi == "dgelu" and ctas == 1 and tma:
                        continue
                    out.add((epi, bn, ctas, tma, False))
    for bn in (128, 256):
        for ctas in (1, 2):
            out.add(("resid_stats", bn, ctas, True, False))
            out.add(("f32", bn, ctas, True, True))
    return out


# ---- the case lists ----------------------------------------------------------------------------
# N: 8 (one partial 32-column chunk), 264 (third 128-wide tile has 8 columns), 384 (three full
# 128-wide tiles), 1600 (fc1 of the reference config: 13 tiles of 128) pick BLOCK_N = 128;
# 136, 200 (ties: one partial 256-wide tile), 744 (three 256-wide tiles, ragged), 768 pick 256.
N_LIST = [8, 264, 384, 1600, 136, 200, 744, 768]
M_LIST = [1, 127, 128, 129, 255, 257, 1000]
K_LIST = [8, 40, 72, 4104]      # below one k-block, one extra 8-wide k-block, many ring turns
LAYOUTS = ["plain", "views", "ldo_aligned", "ldo_unaligned", "no_bias"]
AB_LIST = [(1.0, 0.0), (0.5, 1.0), (0.5, 0.25)]   # EPI_F32: TMA store, TMA reduce-add, direct


def _matrix():
    cases = []
    for e, epi in enumerate(("bf16", "gelu", "gelu_tanh", "relu", "resid", "f32", "dgelu")):
        layouts = LAYOUTS + (["oop"] if epi == "resid" else [])
        for i, N in enumerate(N_LIST):
            M = M_LIST[(i + e) % len(M_LIST)]
            K = K_LIST[(i + 2 * e) % len(K_LIST)]
            layout = layouts[(i + e) % len(layouts)]
            if epi == "f32":
                opt = AB_LIST[i % len(AB_LIST)]
            elif epi in GELU_FAMILY:
                opt = (i % 2 == 0,)            # with out2
            else:
                opt = ()
            cases.append(("gemm", epi, M, N, K, layout, opt))
    return cases


MATRIX = _matrix()
STATS = [("stats", M_LIST[i % 7], N, K_LIST[i % 4], ("views" if i % 3 == 1 else
                                                       "no_bias" if i % 3 == 2 else "plain"))
         for i, N in enumerate(N_LIST)]
FOLDED = [("folded", epi, M, N, K) for epi, M, N, K in [
    ("bf16", 129, 384, 72), ("bf16", 257, 744, 40),
    ("gelu", 1, 8, 8), ("gelu", 1000, 768, 4104),
    ("gelu_tanh", 255, 1600, 136), ("gelu_tanh", 127, 200, 64),
    ("relu", 128, 264, 40), ("relu", 300, 136, 72)]]
# (T, O, I, split_k, alpha, accumulate): I = 136 picks BLOCK_N 256, 384 and 8 pick 128; split_k 3
# with T = 1000 (16 k-blocks) splits 6 + 6 + 4, with T = 65 (2 k-blocks) it is clamped to 2, and
# 40 > 16 k-blocks gives 16 splits of one k-block.
WGRAD = [("wgrad", T, O, I, s, a, acc) for T, O, I, s, a, acc in [
    (1, 8, 136, 1, 1.0, False), (8, 200, 384, 1, 0.5, True), (63, 744, 8, 1, 1.0, False),
    (65, 8, 136, 3, 1.0, True), (1000, 200, 384, 3, 0.5, True), (1000, 744, 8, 40, 1.0, True),
    (1000, 8, 136, 1, 0.5, True), (63, 200, 384, 8, 1.0, True), (8, 744, 8, 3, 1.0, True)]]
SWEEP_N = {128: 3968, 256: 4096}   # 31 full 128-wide tiles / 16 full 256-wide tiles


def _case_id(c):
    if c[0] == "gemm":
        _, epi, M, N, K, layout, opt = c
        o = "" if not opt else ("-out2" if opt == (True,) else "" if opt == (False,) else
                                f"-a{opt[0]}b{opt[1]}")
        return f"{epi}-{M}x{N}x{K}-{layout}{o}"
    return "-".join(str(x) for x in c)


# ---- reference and bound -------------------------------------------------------------------------
_REPORT = {}    # name -> worst err / bound; "c:<epi>" -> worst err / (2^-24 magnitude)


def _note(key, value):
    _REPORT[key] = max(_REPORT.get(key, 0.0), value)


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    if _REPORT:
        print("\nworst err / bound, and err / (2^-24 magnitude) where the output is fp32:")
        for k in sorted(_REPORT):
            print(f"  {k:28s} {_REPORT[k]:.4g}")


def gelu64(x):
    return 0.5 * x * (1.0 + torch.special.erf(x / math.sqrt(2.0)))


def dgelu64(x):
    return (0.5 * (1.0 + torch.special.erf(x / math.sqrt(2.0)))
            + x * torch.exp(-0.5 * x * x) / math.sqrt(2.0 * math.pi))


def bf16_ulp(ref):
    """One bf16 ulp of |ref| (8 significant bits); 0 where ref is 0."""
    _, e = torch.frexp(ref.abs())
    return torch.where(ref == 0, torch.zeros_like(ref), torch.ldexp(torch.ones_like(ref), e - 8))


def _approx(epi, x, g=None, tma=False):
    """Documented per-element error of the epilogue's activation against the exact erf form."""
    if epi == "gelu":
        return torch.full_like(x, 9e-5)            # erf-fitted logistic (gelu_fast[_pair])
    if epi == "gelu_tanh":
        return 3.3e-5 + 2.5e-4 * x.abs()           # 3.2e-5 fit + tanh.approx's ~2^-11 in t
    if epi == "dgelu":
        if tma:                                    # dgelu_tanh_pair: 1.21e-4 fit at x = 1.66
            return g.abs() * (1.3e-4 + 2.0 ** -11 * (0.5 + 2.0 * x.abs()))
        return g.abs() * 1e-5                      # erff / __expf
    return torch.zeros_like(x)


def _bound(mag, slope, approx, ref, bf16_out):
    b = C_ACC * U24 * mag * slope + approx
    return b + bf16_ulp(ref) if bf16_out else b


def _check(name, out, ref, bound, mag=None):
    """Asserts |out - ref| <= bound elementwise; records the worst ratio (and, for fp32 outputs,
    the worst err / (2^-24 mag), the measured accumulation constant)."""
    out = out.double()
    assert torch.isfinite(out).all(), f"{name}: non-finite output"
    err = (out - ref).abs()
    ratio = torch.where(bound > 0, err / bound.clamp_min(1e-300),
                        torch.where(err > 0, torch.full_like(err, math.inf), torch.zeros_like(err)))
    worst = ratio.max().item() if ratio.numel() else 0.0
    _note(name, worst)
    if mag is not None and err.numel():
        _note("c:" + name,(err / (U24 * mag).clamp_min(1e-300)).max().item())
    if worst > 1.0:
        i = int(ratio.argmax())
        r, c = divmod(i, ref.shape[-1]) if ref.dim() == 2 else (0, i)
        raise AssertionError(
            f"{name}: err / bound = {worst:.3g} at [{r}, {c}]: out {out.flatten()[i].item()!r}, "
            f"ref {ref.flatten()[i].item()!r}, bound {bound.flatten()[i].item():.3g}; "
            f"{int((ratio > 1).sum())} of {ratio.numel()} elements out of bound")
    return worst


def _bits(t):
    return t.view(torch.int32) if t.dtype == torch.float32 else t.view(torch.int16)


def _assert_same_bits(a, b, what):
    assert torch.equal(_bits(a), _bits(b)), f"{what}: two identical calls differ"


def _gen(seed):
    return torch.Generator(device="cuda").manual_seed(seed)


def _operand(rows, K, g, pad, scale=1.0):
    """bf16 [rows, K]; a column slice of a [rows, K + pad] buffer when pad > 0 (lda = K + pad)."""
    t = (torch.randn(rows, K + pad, generator=g, device="cuda") * scale).bfloat16()
    return t[:, :K] if pad else t


SENTINEL = -7.75


class _Placed:
    """An [M, N] output inside a buffer: plain, or a view at a column offset of a buffer N + 8 wide
    (ldo = N + 8).  The rest of the buffer holds SENTINEL and must come back untouched."""

    def __init__(self, M, N, dtype, layout):
        eb = 4 if dtype == torch.float32 else 2
        if layout in ("ldo_aligned", "ldo_unaligned"):
            self.off = (16 if layout == "ldo_aligned" else 8) // eb
            self.width = N + 8
        else:
            self.off, self.width = 0, N
        self.M, self.N, self.dtype = M, N, dtype

    def make(self, init=None):
        buf = torch.full((self.M, self.width), SENTINEL, dtype=self.dtype, device="cuda")
        view = buf[:, self.off:self.off + self.N]
        view.copy_(init if init is not None else torch.full_like(view, math.nan))
        return buf, view

    def check_pad(self, buf, what):
        mask = torch.ones(self.width, dtype=torch.bool, device="cuda")
        mask[self.off:self.off + self.N] = False
        if mask.any():
            assert (buf[:, mask].float() == SENTINEL).all(), f"{what}: wrote outside its columns"


# ---- the shape / layout / instantiation matrix ------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("case", MATRIX, ids=[_case_id(c) for c in MATRIX])
def test_gemm_epilogue(vitk, gemm_mode, case):
    _, epi, M, N, K, layout, opt = case
    _, bn, ctas, tma, _ = predict(case, gemm_mode)
    g = _gen(M * 7919 + N * 31 + K)
    views = layout == "views"
    a = _operand(M, K, g, 64 if views else 0)
    w = _operand(N, K, g, 8 if views else 0, 1.0 / math.sqrt(K))
    bias = None if layout == "no_bias" else torch.randn(N, generator=g, device="cuda")
    f32_out = epi in ("resid", "f32")
    place = _Placed(M, N, torch.float32 if f32_out else torch.bfloat16, layout)
    alpha, beta = opt if epi == "f32" else (1.0, 0.0)
    with_out2 = epi in GELU_FAMILY and opt[0]
    init = None
    if epi == "resid" or (epi == "f32" and beta != 0.0):
        init = torch.randn(M, N, generator=g, device="cuda")
    resid_sep = None
    if epi == "resid" and layout == "oop":      # resid != out, ldr = N + 16 != ldo = N
        resid_sep = torch.randn(M, N + 16, generator=g, device="cuda")[:, :N]
    aux = None
    if epi == "dgelu":                            # the pre-activation shares out's pitch / offset
        aux_place = _Placed(M, N, torch.bfloat16, layout)
        _, aux = aux_place.make((torch.randn(M, N, generator=g, device="cuda") * 1.5).bfloat16())

    def call():
        buf, out = place.make(init if resid_sep is None else None)
        buf2 = out2 = None
        if with_out2:
            buf2, out2 = place.make()
        resid = None
        if epi == "resid":
            resid = resid_sep if resid_sep is not None else out
        vitk.ops.gemm(a, w, EPI_IDS[epi], bias=bias, resid=resid, aux=aux, out=out, out2=out2,
                      alpha=alpha, beta=beta)
        return buf, out, buf2, out2

    buf, out, buf2, out2 = call()
    buf_b, _, buf2_b, _ = call()                 # the other tile sweep direction (sweep_next)
    _assert_same_bits(buf, buf_b, "out")
    if with_out2:
        _assert_same_bits(buf2, buf2_b, "out2")
    place.check_pad(buf, "out")
    if with_out2:
        place.check_pad(buf2, "out2")

    a64, w64 = a.double(), w.double()
    S = a64 @ w64.t()
    mag = a64.abs() @ w64.abs().t()
    b64 = bias.double() if bias is not None else torch.zeros(N, dtype=torch.float64, device="cuda")
    name = f"{epi}:{'tma' if tma else 'direct'}:bn{bn}"
    if epi == "f32":
        pre = alpha * S + b64
        mag = abs(alpha) * mag + b64.abs()
        if beta != 0.0:
            pre = pre + beta * init.double()
            mag = mag + abs(beta) * init.double().abs()
        _check(name, out, pre, _bound(mag, 1.0, 0.0, pre, False), mag)
        return
    if epi == "resid":
        r = (resid_sep if resid_sep is not None else init).double()
        pre = S + b64 + r
        mag = mag + b64.abs() + r.abs()
        _check(name, out, pre, _bound(mag, 1.0, 0.0, pre, False), mag)
        return
    pre = S + b64
    mag = mag + b64.abs()
    if epi == "bf16":
        _check(name, out, pre, _bound(mag, 1.0, 0.0, pre, True))
    elif epi == "relu":
        ref = pre.clamp_min(0.0)
        assert (out >= 0).all()
        _check(name, out, ref, _bound(mag, 1.0, 0.0, ref, True))
    elif epi in ("gelu", "gelu_tanh"):
        ref = gelu64(pre)
        _check(name, out, ref, _bound(mag, GELU_SLOPE, _approx(epi, pre), ref, True))
    else:   # dgelu: out = (acc + bias) * gelu'(aux)
        x = aux.double()
        ref = pre * dgelu64(x)
        _check(name, out, ref, _bound(mag, GELU_SLOPE, _approx(epi, x, pre, tma), ref, True))
    if with_out2:
        _check(name + ":out2", out2, pre, _bound(mag, 1.0, 0.0, pre, True))


# ---- activation sweeps with an exactly known pre-activation ------------------------------------
def _exact_operands(M, N, g):
    """A [M, 64], W [N, 64] with entries in {-1, 0, 1} in the first four columns and zeros after:
    A W^T is a small integer, exact in fp32, in one k-block."""
    a = torch.zeros(M, 64, device="cuda")
    w = torch.zeros(N, 64, device="cuda")
    a[:, :4] = torch.randint(-1, 2, (M, 4), generator=g, device="cuda").float()
    w[:, :4] = torch.randint(-1, 2, (N, 4), generator=g, device="cuda").float()
    return a.bfloat16(), w.bfloat16()


def _ramp(N):
    """-16 + odd multiples of 1/256: exact in fp32 after adding a small integer, and never a bf16
    rounding tie where |x| >= 8 (ties there are even multiples of 1/256)."""
    n = torch.arange(N, device="cuda", dtype=torch.float64)
    return -16.0 + (2.0 * n + 1.0) / 256.0


@pytest.mark.gpu
@pytest.mark.parametrize("bn", [128, 256], ids=["bn128", "bn256"])
@pytest.mark.parametrize("epi", ["gelu", "gelu_tanh", "relu", "dgelu"])
def test_activation_sweep(vitk, gemm_mode, epi, bn):
    """Dense ramp of pre-activations over [-20, 20] through every activation epilogue.  The
    saturated tails must be exact: gelu(x) == bf16(x) and gelu'(x) g == bf16(g) for x >= 9,
    |gelu(x)| <= 1e-6 |x| (times |g| for gelu') for x <= -9."""
    M, N = 256, SWEEP_N[bn]
    assert block_n(N) == bn
    _, _, ctas, tma, _ = predict(("gemm", epi, M, N, 64, "plain", (True, 1.0)), gemm_mode)
    g = _gen(11 + bn)
    a, w = _exact_operands(M, N, g)
    acc = a.double() @ w.double().t()
    name = f"sweep:{epi}:{'tma' if tma else 'direct'}:bn{bn}"

    if epi == "dgelu":
        bias = torch.full((N,), 0.5, device="cuda")         # g = acc + 0.5: never 0, exact
        xa = _ramp(N).float().bfloat16().expand(M, N).contiguous()
        calls = [vitk.ops.gemm(a, w, EPI_IDS[epi], bias=bias, aux=xa) for _ in range(2)]
        _assert_same_bits(calls[0], calls[1], name)
        out = calls[0].double()
        gg = acc + 0.5
        x = xa.double()
        ref = gg * dgelu64(x)
        hi, lo = x >= SAT, x <= -SAT
        mid = ~(hi | lo)
        assert torch.equal(out[hi], gg[hi].float().bfloat16().double()), f"{name}: x >= 9 not exact"
        tail = (out[lo].abs() / (x[lo].abs() * gg[lo].abs())).max().item()
        assert tail <= 1e-6, f"{name}: |out| / (|x| |g|) = {tail:.3g} for x <= -9"
        _note(name + ":tail<=-9", tail)
        _note(name + ":tail<=-9 nonzero", float((out[lo] != 0).sum().item()))
        bound = _approx(epi, x, gg, tma) + bf16_ulp(ref)
        _check(name, out[mid], ref[mid], bound[mid])
        return

    bias64 = _ramp(N)
    bias = bias64.float()
    pre = acc + bias64                                       # exact in fp32
    calls = []
    for _ in range(2):
        out2 = torch.empty(M, N, dtype=torch.bfloat16, device="cuda")
        out = vitk.ops.gemm(a, w, EPI_IDS[epi], bias=bias, out2=out2)
        calls.append((out, out2))
    _assert_same_bits(calls[0][0], calls[1][0], name)
    _assert_same_bits(calls[0][1], calls[1][1], name + ":out2")
    out, out2 = calls[0]
    pre_bf16 = pre.float().bfloat16()
    assert torch.equal(_bits(out2), _bits(pre_bf16)), f"{name}: out2 != bf16(acc + bias)"
    if epi == "relu":
        assert torch.equal(_bits(out), _bits(pre.clamp_min(0.0).float().bfloat16())), \
            f"{name}: relu not exact"
        return
    out = out.double()
    ref = gelu64(pre)
    hi, lo = pre >= SAT, pre <= -SAT
    mid = ~(hi | lo)
    bad = out[hi] != pre_bf16.double()[hi]
    assert not bad.any(), (f"{name}: gelu(x) != bf16(x) for x >= 9 at "
                           f"x = {pre[hi][bad][:4].tolist()}: {out[hi][bad][:4].tolist()}")
    tail = (out[lo].abs() / pre[lo].abs()).max().item()
    assert tail <= 1e-6, f"{name}: |gelu(x)| / |x| = {tail:.3g} for x <= -9"
    _note(name + ":tail<=-9", tail)
    _note(name + ":tail<=-9 nonzero", float((out[lo] != 0).sum().item()))
    _check(name, out[mid], ref[mid], _approx(epi, pre, tma=tma)[mid] + bf16_ulp(ref)[mid])


# ---- residual GEMM with row statistics, and the LayerNorm-folded consumer ----------------------
@pytest.mark.gpu
@pytest.mark.parametrize("case", STATS, ids=[_case_id(c) for c in STATS])
def test_gemm_resid_stats_epilogue(vitk, gemm_mode, case):
    _, M, N, K, layout = case
    _, bn, _, _, _ = predict(case, gemm_mode)
    g = _gen(M + N + K)
    views = layout == "views"
    a = _operand(M, K, g, 64 if views else 0)
    w = _operand(N, K, g, 8 if views else 0, 1.0 / math.sqrt(K))
    bias = None if layout == "no_bias" else torch.randn(N, generator=g, device="cuda")
    x0 = torch.randn(M, N, generator=g, device="cuda") * 2 + 0.3
    runs = []
    for _ in range(2):
        x = x0.clone()
        xb, st = vitk.ops.gemm_resid_stats(a, w, x, bias=bias)
        runs.append((x, xb, st))
    for i, what in enumerate(("x", "bf16(x)", "stats")):
        _assert_same_bits(runs[0][i], runs[1][i], what)
    x, xb, st = runs[0]
    a64, w64 = a.double(), w.double()
    b64 = bias.double() if bias is not None else 0.0
    ref = x0.double() + a64 @ w64.t() + b64
    mag = a64.abs() @ w64.abs().t() + x0.double().abs() + (b64.abs() if bias is not None else 0.0)
    name = f"resid_stats:tma:bn{bn}"
    _check(name, x, ref, _bound(mag, 1.0, 0.0, ref, False), mag)
    assert torch.equal(_bits(xb), _bits(x.bfloat16()))
    # partial p covers columns [p * cols, (p + 1) * cols): half a tile; fp32 sums of the stored x
    cols = bn // 2
    assert st.shape[0] == -(-N // cols)
    x64 = x.double()
    for p in range(st.shape[0]):
        seg = x64[:, p * cols:(p + 1) * cols]
        n = seg.shape[1]
        _check(name + ":sum", st[p, :, 0], seg.sum(1), 2 * n * U24 * seg.abs().sum(1))
        _check(name + ":sumsq", st[p, :, 1], (seg * seg).sum(1), 2 * (n + 1) * U24 * (seg * seg).sum(1))


@pytest.mark.gpu
@pytest.mark.parametrize("case", FOLDED, ids=[_case_id(c) for c in FOLDED])
def test_gemm_layernorm_folded_epilogue(vitk, gemm_mode, case):
    """out = act(rstd * (xb @ w^T) + b), rstd from three partial (sum, sum of squares) per row."""
    _, epi, M, N, K = case
    _, bn, _, _, _ = predict(case, gemm_mode)
    g = _gen(M * 3 + N + K)
    x = torch.randn(M, K, generator=g, device="cuda") * 2 + 0.3
    xb = x.bfloat16()
    w = _operand(N, K, g, 0, 1.0 / math.sqrt(K))
    b = torch.randn(N, generator=g, device="cuda") * 0.5
    edges = [0, K // 3, 2 * K // 3, K]
    st = torch.stack([torch.stack([x[:, lo:hi].sum(1), (x[:, lo:hi] ** 2).sum(1)], -1)
                      for lo, hi in zip(edges, edges[1:])]).contiguous()
    outs = [vitk.ops.gemm_layernorm_folded(xb, w, b, st, eps=1e-5, epilogue=EPI_IDS[epi])
            for _ in range(2)]
    _assert_same_bits(outs[0], outs[1], "out")
    s = st.double().sum(0)
    mean = s[:, 0] / K
    ex2 = s[:, 1] / K
    var = ex2 - mean * mean
    rstd = (1.0 / torch.sqrt(var + 1e-5))[:, None]
    # fp32 statistics: cancellation in E[x^2] - mean^2, rsqrtf
    rel_rstd = (2.0 ** -21 + 8 * U24 * ex2 / var)[:, None]
    S = xb.double() @ w.double().t()
    mag = rstd * (xb.double().abs() @ w.double().abs().t()) + b.double().abs()
    pre = rstd * S + b.double()
    slope = GELU_SLOPE if epi in ("gelu", "gelu_tanh") else 1.0
    ref = gelu64(pre) if epi in ("gelu", "gelu_tanh") else pre.clamp_min(0.0) if epi == "relu" else pre
    bound = _bound(mag, slope, _approx(epi, pre), ref, True) + slope * rel_rstd * (rstd * S).abs()
    _check(f"folded:{epi}:tma:bn{bn}", outs[0], ref, bound)


# ---- MN-major weight gradient ------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("case", WGRAD, ids=[_case_id(c) for c in WGRAD])
def test_gemm_wgrad_epilogue(vitk, gemm_mode, case):
    """out[O, I] = alpha dy^T x (+ out), out a view with ldo = I + 8 > I."""
    _, T, O, I, split, alpha, accumulate = case
    _, bn, _, _, _ = predict(case, gemm_mode)
    g = _gen(T * 13 + O + I)
    dy = torch.randn(T, O, generator=g, device="cuda").bfloat16()
    x = torch.randn(T, I, generator=g, device="cuda").bfloat16()
    place = _Placed(O, I, torch.float32, "ldo_aligned")
    c0 = torch.randn(O, I, generator=g, device="cuda") if accumulate else None
    outs = []
    for _ in range(2 if split == 1 else 1):
        buf, out = place.make(c0)
        vitk.ops.gemm_wgrad(dy, x, out, alpha=alpha, accumulate=accumulate, split_k=split)
        outs.append((buf, out))
    if split == 1:
        _assert_same_bits(outs[0][0], outs[1][0], "out")
    buf, out = outs[0]
    place.check_pad(buf, "out")
    d64, x64 = dy.double(), x.double()
    ref = alpha * (d64.t() @ x64)
    mag = abs(alpha) * (d64.abs().t() @ x64.abs())
    if accumulate:
        ref = ref + c0.double()
        mag = mag + c0.double().abs()
    # split-K: every split's partial is reduce-added into out, one more fp32 rounding each
    splits = min(split, -(-T // 64))
    bound = (C_ACC + splits) * U24 * mag
    _check(f"f32:mn:bn{bn}", out, ref, bound, mag)


# ---- CPU: the cases reach every instantiation --------------------------------------------------
def test_cases_cover_every_reachable_instantiation():
    src = (Path(__file__).resolve().parent.parent /
           "automated-recycling-sorter-with-vision-transformers_b200" / "csrc" / "gemm_sm100.cu")
    text = src.read_text()
    # the width rule block_n() restates
    assert "const bool n128 = waste128 < waste256;" in text
    assert "constexpr bool kTma1 = TMA_EPI && (EPI != EPI_DGELU_BF16);" in text
    hit = {}
    for mode in MODES:
        for case in MATRIX + STATS + FOLDED + WGRAD:
            hit.setdefault(predict(case, mode), (case, mode))
        for epi in ("gelu", "gelu_tanh", "relu", "dgelu"):
            for bn in (128, 256):
                case = ("gemm", epi, 256, SWEEP_N[bn], 64, "plain", (True,))
                hit.setdefault(predict(case, mode), (case, mode))
    reachable = reachable_instantiations()
    assert len(reachable) == 62
    assert not set(hit) - reachable, f"predicted unreachable tuples {set(hit) - reachable}"
    missing = reachable - set(hit)
    assert not missing, f"no case runs {sorted(missing)}"
