"""CPU tier: pins oracle/vit_oracle.py against the golden vectors produced by the reference's own
classes (oracle/gen_golden.py), and - when /root/reference is present - against the live classes.
Also checks the drop-in contract of the module mirrors (state_dict keys / seeded init)."""
import pytest
import torch

from oracle import ref_loader
from oracle import vit_oracle as O
from tests import helpers as H

FULL = ["tiny_vit_full", "tiny_deit_full", "small_deit_full"]


@pytest.mark.parametrize("name", FULL)
def test_oracle_matches_reference_golden(name):
    z, cfg = H.load(name)
    sd = H.weights(z)
    x = torch.from_numpy(z["images"])
    with torch.no_grad():
        t64, l64 = O.classifier_forward(sd, x, cfg["num_heads"], dtype=torch.float64)
        t32, l32 = O.classifier_forward(sd, x, cfg["num_heads"], dtype=torch.float32)
    assert (t64 - torch.from_numpy(z["tokens_f64"])).abs().max() < 1e-10
    assert (l64 - torch.from_numpy(z["logits_f64"])).abs().max() < 1e-10
    assert (t32 - torch.from_numpy(z["tokens_f32"])).abs().max() < 2e-5
    assert (l32 - torch.from_numpy(z["logits_f32"])).abs().max() < 2e-5


@pytest.mark.parametrize("name", ["vitb16_vit", "vitb16_deit"])
def test_oracle_matches_reference_vitb16(vitk, name):
    z, cfg = H.load(name)
    model = H.build_classifier(vitk, z, cfg, seed_rebuild=True)   # also checks the SHA-256
    x = O.synthetic_images(2, cfg["image_size"], seed=int(z["image_seed"]))  # first 2 of the 8
    with torch.no_grad():
        t, l = O.classifier_forward(model.state_dict(), x, cfg["num_heads"], dtype=torch.float32)
    assert (l.double() - torch.from_numpy(z["logits_f64"])[:2]).abs().max() < 1e-4
    assert (t[:, :4, :32].double() - torch.from_numpy(z["tokens_f64_head"])[:2]).abs().max() < 1e-3


@pytest.mark.parametrize("name", ["trainstep_tiny_vit", "trainstep_small_deit"])
def test_oracle_train_step_matches_reference(name):
    z, cfg = H.load(name)
    sd = H.weights(z, "w:")
    x = torch.from_numpy(z["images"])
    y = torch.from_numpy(z["labels"])
    loss, grads, new = O.train_step(sd, x, y, cfg["num_heads"], dtype=torch.float64)
    assert abs(float(loss) - float(z["loss_f64"])) < 1e-6   # weights were stored in fp32
    g_ref, n_ref = H.weights(z, "g:"), H.weights(z, "n:")
    for k in sd:
        assert (grads[k].float() - g_ref[k]).abs().max() <= 1e-5 * (1 + g_ref[k].abs().max()), k
        assert (new[k].float() - n_ref[k]).abs().max() < 1e-6, k


def test_module_mirrors_reproduce_reference_state_dict(vitk):
    """Same constructor order => same RNG stream => identical random init; same keys/shapes.
    Checked for the ViT and the DeiT mirror against the weights (in the reference's key order)
    that the reference's own constructors produced for each *_full fixture."""
    for name in FULL:
        z, cfg = H.load(name)
        torch.manual_seed(int(z["seed"]))
        m = vitk.ViTClassifier(num_classes=6, deit=str(z["kind"]) == "deit", **cfg)
        ref = H.weights(z)
        sd = m.state_dict()
        assert list(sd.keys()) == list(ref.keys()), name
        for k in ref:
            assert torch.equal(sd[k], ref[k]), (name, k)


@pytest.mark.skipif(not ref_loader.reference_available(), reason="reference only in the build box")
@pytest.mark.parametrize("kind", ["vit", "deit"])
def test_oracle_matches_live_reference(vitk, kind):
    kw = dict(image_size=48, patch_size=16, embed_dim=128, num_layers=2, num_heads=2, mlp_dim=256,
              dropout=0.1)
    torch.manual_seed(11)
    ref_cls = (ref_loader.load("evaluation").VisionTransformer if kind == "vit"
               else ref_loader.load("train").DataEfficientImageTransformer)
    ref = ref_cls(**kw).eval()
    torch.manual_seed(11)
    mine = (vitk.VisionTransformer if kind == "vit" else vitk.DataEfficientImageTransformer)(**kw)
    assert list(ref.state_dict().keys()) == list(mine.state_dict().keys())
    for a, b in zip(ref.state_dict().values(), mine.state_dict().values()):
        assert torch.equal(a, b)
    x = O.synthetic_images(3, 48)
    with torch.no_grad():
        want = ref(x)
        got = O.backbone_forward(ref.state_dict(), x, kw["num_heads"])
    assert (want - got).abs().max() < 2e-5
    # a reference checkpoint loads into the mirror (drop-in contract, SURVEY.md 8b)
    mine.load_state_dict(ref.state_dict(), strict=True)


@pytest.mark.parametrize("name", ["det_head_small", "det_head_vitb"])
def test_head_oracle_matches_reference_golden(vitk, name):
    """Detection head restatement vs the outputs of the reference's ObjectDetectionHead."""
    z = H.np.load(H.GOLDEN / f"{name}.npz", allow_pickle=True)
    _, sd = H.build_head(vitk, z)          # also: mirror keys == reference keys, SHA-256
    tokens = H.head_tokens(z)
    with torch.no_grad():
        o64 = O.detection_head_forward(sd, tokens[:, 1:, :], dtype=torch.float64)
        o32 = O.detection_head_forward(sd, tokens[:, 1:, :], dtype=torch.float32)
    assert (o64["class_logits"] - torch.from_numpy(z["class_logits_f64"])).abs().max() < 1e-10
    assert (o64["bbox_coords"] - torch.from_numpy(z["bbox_f64"])).abs().max() < 1e-10
    assert (o32["class_logits"] - torch.from_numpy(z["class_logits_f32"])).abs().max() < 2e-5
    assert (o32["bbox_coords"] - torch.from_numpy(z["bbox_f32"])).abs().max() < 2e-5


@pytest.mark.skipif(not ref_loader.reference_available(), reason="reference only in the build box")
def test_head_oracle_and_mirror_match_live_reference(vitk):
    ev = ref_loader.load("evaluation")
    torch.manual_seed(21)
    ref = ev.ViTObjectDetector(image_size=32, embed_dim=64, num_layers=1, num_heads=2, mlp_dim=64,
                               num_classes=6, num_queries=5).eval()
    torch.manual_seed(21)
    mine = vitk.ViTObjectDetector(image_size=32, embed_dim=64, num_layers=1, num_heads=2, mlp_dim=64,
                                  num_classes=6, num_queries=5)
    assert list(ref.state_dict().keys()) == list(mine.state_dict().keys())
    for (k, a), b in zip(ref.state_dict().items(), mine.state_dict().values()):
        assert torch.equal(a, b), k                      # same constructor order, same RNG stream
    mine.load_state_dict(ref.state_dict(), strict=True)  # a reference checkpoint loads
    mem = torch.randn(2, 4, 64, generator=torch.Generator().manual_seed(5))
    with torch.no_grad():
        want = ref.detection_head(mem)
        got = O.detection_head_forward(ref.state_dict(), mem, prefix="detection_head.")
    assert (want["class_logits"] - got["class_logits"]).abs().max() < 2e-5
    assert (want["bbox_coords"] - got["bbox_coords"]).abs().max() < 2e-5


@pytest.mark.skipif(not ref_loader.reference_available(), reason="reference only in the build box")
def test_post_process_and_triplet_oracles_match_live_reference():
    ev, tr = ref_loader.load("evaluation"), ref_loader.load("train")
    g = torch.Generator().manual_seed(0)
    out = {"class_logits": torch.randn(4, 50, 7, generator=g) * 2,
           "bbox_coords": torch.rand(4, 50, 4, generator=g)}
    out["class_logits"][2, :, -1] += 30.0
    for thr in (0.3, 0.5):
        want, got = ev.post_process_predictions(out, thr), O.post_process_predictions(out, thr)
        for a, b in zip(want, got):
            assert a["boxes"].shape == b["boxes"].shape
            assert torch.equal(a["labels"], b["labels"]) and torch.allclose(a["scores"], b["scores"])
            assert torch.equal(a["boxes"], b["boxes"])
    torch.manual_seed(2)
    det = tr.DeiTObjectDetector(image_size=32, embed_dim=64, num_layers=1, num_heads=2, mlp_dim=64,
                                num_classes=6, num_queries=3).eval()
    x = O.synthetic_images(2, 32)
    with torch.no_grad():
        _, trip = det(x, return_features=True)
        toks = det.backbone(x)
    ref = O.triplet_features(toks[:, 0], det.triplet_projection.weight, det.triplet_projection.bias)
    assert (trip - ref).abs().max() < 1e-6


def test_synthetic_inputs_are_deterministic():
    a, b = O.synthetic_images(2, 32), O.synthetic_images(2, 32)
    assert torch.equal(a, b) and a.shape == (2, 3, 32, 32) and a.dtype == torch.float32
    assert -2.2 < a.min() < -1.9 and 2.4 < a.max() < 2.7   # ImageNet-normalised 8-bit range
