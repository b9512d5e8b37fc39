"""Device timing of train.py's own detector, vitk.DeiTObjectDetector at its Config (DeiT, D = 400,
12 layers, 25 encoder heads of 16, MLP 1600, 6 classes, 5 object queries; the head's decoder
attention has 8 heads of 50):

    python tests/bench_detector_config.py [train_batch] [eval_batch] [out.json]

  * a training step at batch 32: forward, loss, backward, AdamW (train.py:1441-1460, 1598-1602)
  * an eval forward at batch 8 (evaluation.py's batch)
  * the detection head's time by kernel class, from the library's event profiler, for the eval
    forward and for the head's training forward + backward; the attention class there is the
    decoder attention alone (the encoder is outside the head)

CUDA events around `iters` back-to-back calls after warm-up.  The card's name and power limit are
read in the same run and printed with the numbers."""
import json
import subprocess
import sys
from pathlib import Path

import torch
import torch.nn.functional as F

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import vitk  # noqa: E402
from oracle import vit_oracle as O  # noqa: E402

CONFIG = dict(image_size=224, embed_dim=400, num_layers=12, num_heads=25, mlp_dim=1600,
              num_classes=6, num_queries=5, dropout=0.1)


def timed(fn, iters=20, warm=5):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm",
                              "--format=csv,noheader", "-i", "0"], capture_output=True, text=True,
                             timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = ""
    return out or torch.cuda.get_device_name(0)


def profiled(fn):
    torch.cuda.synchronize()
    vitk._lib.profile_collect()          # drop anything recorded before
    vitk._lib.profile_enable(True)
    try:
        fn()
        torch.cuda.synchronize()
        prof = vitk._lib.profile_collect()
    finally:
        vitk._lib.profile_enable(False)
    return {k: {"ms": round(v["ms"], 4), "launches": v["launches"]} for k, v in prof.items()
            if v["launches"]}


def main():
    Bt = int(sys.argv[1]) if len(sys.argv) > 1 else 32
    Be = int(sys.argv[2]) if len(sys.argv) > 2 else 8
    out_path = sys.argv[3] if len(sys.argv) > 3 else None
    if not torch.cuda.is_available():
        raise SystemExit("bench_detector_config needs a CUDA device")
    torch.manual_seed(0)
    model = vitk.DeiTObjectDetector(**CONFIG).cuda()
    opt = torch.optim.AdamW(model.parameters(), lr=1e-4, weight_decay=1e-4)
    x = O.synthetic_images(Bt, 224).cuda()
    xe = x[:Be].contiguous()
    Q = CONFIG["num_queries"]
    tgt_cls = torch.randint(0, 7, (Bt, Q), generator=torch.Generator().manual_seed(1)).cuda()
    tgt_box = torch.rand(Bt, Q, 4, generator=torch.Generator().manual_seed(2)).cuda()
    w = torch.ones(7, device="cuda")
    w[-1] = 0.1

    def train_step():
        opt.zero_grad(set_to_none=True)
        pred, triplet = model(x)
        loss = vitk.weighted_cross_entropy(pred["class_logits"], tgt_cls, w) + \
            F.l1_loss(pred["bbox_coords"], tgt_box) + 0.01 * triplet.pow(2).sum()
        loss.backward()
        opt.step()

    model.train()
    t_train = timed(train_step)
    model.eval()
    with torch.no_grad():
        t_eval = timed(lambda: model(xe))

    # the head alone, on the encoder's tokens (CLS and DIST dropped, as the detector does)
    head = model.detection_head
    with torch.no_grad():
        toks_e = model.backbone(xe)
    res = {"card": card(), "train_batch": Bt, "eval_batch": Be, "config": CONFIG,
           "train_step_ms": round(t_train, 3), "train_images_per_s": round(Bt / t_train * 1e3, 1),
           "eval_forward_ms": round(t_eval, 3), "eval_images_per_s": round(Be / t_eval * 1e3, 1)}
    with torch.no_grad():
        res["head_eval_profile"] = profiled(lambda: head.decode(toks_e, 2))
    model.train()
    toks_t = model.backbone(x).detach().requires_grad_(True)

    def head_train():
        out = head.decode(toks_t, 2)
        (out["class_logits"].float().sum() + out["bbox_coords"].float().sum()).backward()

    head_train()
    res["head_train_profile"] = profiled(head_train)
    for key in ("head_eval_profile", "head_train_profile"):
        prof = res[key]
        total = sum(v["ms"] for v in prof.values())
        attn = prof.get("attention", {}).get("ms", 0.0)
        res[key.replace("profile", "attention_share")] = round(attn / total, 4) if total else None
    print(json.dumps(res, indent=1))
    if out_path:
        Path(out_path).parent.mkdir(parents=True, exist_ok=True)
        Path(out_path).write_text(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
