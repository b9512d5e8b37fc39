"""The detection head and the CLS-only classifier tail at embed widths whose head_dim is not 32, 64,
96 or 128 (SURVEY.md 0 divergence 2: train.py's Config is DeiT at D = 400, and ObjectDetectionHead
hard-codes 8 heads, so its decoder attention has head_dim 50), against the oracle in fp64 with the
bars of test_detection_gpu.py / test_detection_train_gpu.py / test_model_gpu.py."""
import pytest
import torch
import torch.nn.functional as F

from oracle import ref_loader
from oracle import vit_oracle as O

pytestmark = pytest.mark.gpu


def _head(vitk, D, Q, seed=1, layers=None):
    torch.manual_seed(0)
    head = vitk.ObjectDetectionHead(embed_dim=D, num_classes=6, num_queries=Q)
    if layers is not None:
        head.decoder.layers = torch.nn.ModuleList(list(head.decoder.layers)[:layers])
        head.decoder.num_layers = layers
    sd = O.randomize_head_state(head.state_dict(), seed)
    head.load_state_dict(sd)
    return head, sd


def _no_dropout(module):
    for m in module.modules():
        if isinstance(m, torch.nn.Dropout):
            m.p = 0.0
        if isinstance(m, torch.nn.MultiheadAttention):
            m.dropout = 0.0


def _rel(a, b):
    a, b = a.double().flatten(), b.double().flatten()
    return ((a - b).norm() / b.norm().clamp_min(1e-30)).item(), \
        (torch.dot(a, b) / (a.norm() * b.norm()).clamp_min(1e-30)).item()


@pytest.mark.parametrize("Q,P,B,skip", [(100, 196, 2, 1), (5, 196, 3, 2)])
@pytest.mark.parametrize("D", [192, 384, 392, 400, 640])
def test_head_inference_matches_oracle(vitk, D, Q, P, B, skip):
    head, sd = _head(vitk, D, Q, seed=100 + D)
    head = head.cuda().eval()
    tokens = torch.randn(B, P + skip, D, generator=torch.Generator().manual_seed(9))
    with torch.no_grad():
        ref = O.detection_head_forward(sd, tokens[:, skip:, :], dtype=torch.float64)
        out = head.decode(tokens.cuda(), skip_tokens=skip)
    lg, bx = out["class_logits"].cpu().double(), out["bbox_coords"].cpu().double()
    assert torch.isfinite(lg).all() and torch.isfinite(bx).all()
    # At 5 queries the head's bf16 error alone straddles test_detection_gpu.py's 2e-2, whichever
    # attention kernel runs: over six seeds (B200) the existing head_dim 32 / 64 kernels reach a
    # worst logit error of 0.0195 / 0.0218, head_dim 49 / 50 on the new ones 0.0199 / 0.0208.
    assert (lg - ref["class_logits"]).abs().max().item() < (2e-2 if Q == 100 else 3e-2)
    assert (bx - ref["bbox_coords"]).abs().max().item() < 1e-2


def _train_check(vitk, head, sd, tokens, skip, Q, masks=None):
    g = torch.Generator().manual_seed(3)
    B = tokens.shape[0]
    r_logits = torch.randn(B, Q, 7, generator=g)
    r_boxes = torch.randn(B, Q, 4, generator=g)
    sd64 = {k: v.double().clone().requires_grad_(True) for k, v in sd.items()}
    tok64 = tokens.double().clone().requires_grad_(True)
    ref = O.detection_head_forward(sd64, tok64[:, skip:, :], dtype=torch.float64, masks=masks)
    ((ref["class_logits"] * r_logits.double()).sum() + (ref["bbox_coords"] * r_boxes.double()).sum()).backward()
    tok = tokens.cuda().requires_grad_(True)
    out = head.decode(tok, skip_tokens=skip)
    ((out["class_logits"] * r_logits.cuda()).sum() + (out["bbox_coords"] * r_boxes.cuda()).sum()).backward()
    torch.cuda.synchronize()
    assert (out["class_logits"].detach().cpu().double() - ref["class_logits"]).abs().max() < 3e-2
    assert (out["bbox_coords"].detach().cpu().double() - ref["bbox_coords"]).abs().max() < 1e-2
    worst = (0.0, "")
    for name, prm in head.named_parameters():
        assert prm.grad is not None, name
        rel, cos = _rel(prm.grad.cpu(), sd64[name].grad)
        worst = max(worst, (rel, name))
        assert cos > 0.995 and rel < 9e-2, (name, rel, cos)
    rel, cos = _rel(tok.grad.cpu(), tok64.grad)
    print("worst parameter gradient error", worst, "d tokens", rel, cos)
    assert cos > 0.995 and rel < 9e-2
    return out


@pytest.mark.parametrize("D,Q,P,B,skip,L", [
    (400, 5, 196, 3, 2, 6),      # train.py's Config: head_dim 50, 5 queries, DeiT slicing
    (384, 100, 196, 2, 1, 2),    # ViT-S width: head_dim 48, 100 queries
])
def test_head_backward_matches_oracle_autograd(vitk, D, Q, P, B, skip, L):
    head, sd = _head(vitk, D, Q, layers=L)
    _no_dropout(head)
    head = head.cuda().train()
    tokens = torch.randn(B, P + skip, D, generator=torch.Generator().manual_seed(3))
    _train_check(vitk, head, sd, tokens, skip, Q)


def test_head_with_dropout_at_width_400(vitk):
    """The library's masks (the six dropout sites of every decoder layer) injected into the oracle."""
    from tests.test_detection_train_gpu import _head_masks
    p, D, Q, P, B, skip, L = 0.1, 400, 5, 196, 2, 2, 2
    head, sd = _head(vitk, D, Q, layers=L)
    for ly in head.decoder.layers:
        for m in (ly.dropout, ly.dropout1, ly.dropout2, ly.dropout3):
            m.p = p
        ly.self_attn.dropout = ly.multihead_attn.dropout = p
    head = head.cuda().train()
    seed = 4242
    head.__dict__["_vitk_forced_seed"] = seed
    F_ = head.decoder.layers[0].linear1.out_features
    masks = _head_masks(vitk, p, seed, B, Q, P, D, F_, 8, L)
    tokens = torch.randn(B, P + skip, D, generator=torch.Generator().manual_seed(3))
    out = _train_check(vitk, head, sd, tokens, skip, Q, masks=masks)
    with torch.no_grad():
        ev = head.eval().decode(tokens.cuda(), skip_tokens=skip)
    assert (ev["class_logits"] - out["class_logits"].detach()).abs().max() > 1e-2


TRAIN_PY = dict(image_size=224, embed_dim=400, num_layers=12, num_heads=25, mlp_dim=1600,
                num_classes=6, num_queries=5, dropout=0.1)


def test_train_py_detector_trains(vitk):
    """vitk.DeiTObjectDetector at train.py's own Config, batch 32, AdamW as train.py:1598-1602:
    eval forward works, every parameter gets a gradient and the loss goes down."""
    torch.manual_seed(0)
    model = vitk.DeiTObjectDetector(**TRAIN_PY).cuda()
    x = O.synthetic_images(32, 224).cuda()
    with torch.no_grad():
        ev = model.eval()(x[:8])
    assert ev["class_logits"].shape == (8, 5, 7) and torch.isfinite(ev["class_logits"]).all()
    model.train()
    opt = torch.optim.AdamW(model.parameters(), lr=1e-4, weight_decay=1e-4)
    tgt_cls = torch.randint(0, 7, (32, 5), generator=torch.Generator().manual_seed(1)).cuda()
    tgt_box = torch.rand(32, 5, 4, generator=torch.Generator().manual_seed(2)).cuda()
    w = torch.ones(7, device="cuda")
    w[-1] = 0.1
    losses = []
    for step in range(6):
        opt.zero_grad(set_to_none=True)
        pred, triplet = model(x)
        loss = vitk.weighted_cross_entropy(pred["class_logits"], tgt_cls, w) + \
            F.l1_loss(pred["bbox_coords"], tgt_box) + 0.01 * triplet.pow(2).sum()
        loss.backward()
        if step == 0:
            missing = [n for n, p in model.named_parameters() if p.grad is None]
            assert not missing, missing
        opt.step()
        losses.append(loss.item())
    assert all(map(lambda v: v == v, losses)), losses
    assert losses[-1] < losses[0], losses


@pytest.mark.skipif(not ref_loader.reference_available(), reason="reference scripts not shipped")
def test_reference_train_one_epoch_at_width_400(vitk, monkeypatch):
    """train.py's own train_one_epoch on the vitk detector at D = 400 with 25 encoder heads (head
    head_dim 50), two layers, against the reference's DeiTObjectDetector."""
    from tests import test_reference_loop_gpu as R
    kw = dict(R.KW, image_size=64, embed_dim=400, num_heads=25, mlp_dim=800)
    monkeypatch.setattr(R, "KW", kw)
    R.test_reference_train_one_epoch_runs_on_the_vitk_detector(vitk, monkeypatch)


def test_cls_tail_at_train_py_width(vitk):
    """vitk_forward_cls at D = 400, 25 heads (head_dim 16): the CLS-only attention is 1 query
    against 197 tokens."""
    kw = dict(image_size=224, patch_size=16, embed_dim=400, num_layers=2, num_heads=25, mlp_dim=1600)
    torch.manual_seed(1)
    model = vitk.ViTClassifier(num_classes=6, deit=True, dropout=0.0, **kw)
    sd = {k: v.clone() for k, v in model.state_dict().items()}
    x = O.synthetic_images(5, 224)
    with torch.no_grad():
        _, l_ref = O.classifier_forward(sd, x, kw["num_heads"], dtype=torch.float64)
    model = model.cuda().eval()
    with torch.no_grad():
        full = model(x.cuda())
        pruned = model.classify_pruned(x.cuda())
    assert (pruned - full).abs().max() < 4e-3
    assert (pruned.cpu().double() - l_ref).abs().max() < 2e-2
    assert torch.equal(pruned.cpu().double().argmax(-1), l_ref.argmax(-1))
