#!/usr/bin/env python
"""Headline benchmark: ViT-B/16 224px bf16 inference images/sec (BASELINE.json configs[1]).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl vitk|reference] [--batch B]
                    [--dump-outputs DIR]

One "step" = one pass of the hot path (vitk_forward: patch-embed GEMM, 12 pre-LN blocks, CLS
LayerNorm + 6-class head) over one batch of 256 synthetic images per GPU.  Prints ONE JSON line.
For N>1 launch under torchrun (one rank per GPU); the batch shards across ranks with no data-path
collective (weak scaling); time = max over ranks of the device-timed region.

`--dump-outputs DIR` writes what the timed path returned in its last timed step to DIR/logits.npy
(float32, one row per image of the timed batch; for N>1 the ranks' shards in rank order).  Weights
and images are seeded, so two builds run with the same arguments can be compared output for output.
bench_outputs/ in the repository is git-ignored for such dumps.  The two --impl arms run different
batches (256 seeded images per GPU against 32 for the CPU arm), so only dumps of the same --impl
compare.

Next to the headline the same line carries, each device-timed with its own TFLOP/s and fraction
of the measured burst peak: the other BASELINE.json configurations (`configs`: ViT-L/16 weak and
strong sharding, ViT-B/16 at 384 px), the fine-tune step, the detector, a parity check of the
TIMED batch against the oracle (`parity_check`), the reference's own classes run by PyTorch eager
on the same GPU under bf16 autocast (`gpu_eager_baseline`) and, for N > 1, a data-parallel
equivalence check (`dp_check`).

`--impl reference` times the reference's own classes on the host CPU cores - byte-compiled into
oracle/_ref by oracle/build_ref.py, since /root/reference does not exist on the GPU box (kind
"reference"; the oracle port, kind "port", only if oracle/_ref is absent) - on a bounded sample of
the same workload.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

VIT_B16 = dict(image_size=224, patch_size=16, in_channels=3, embed_dim=768, num_layers=12,
               num_heads=12, mlp_dim=3072)
VIT_L16 = dict(image_size=224, patch_size=16, in_channels=3, embed_dim=1024, num_layers=24,
               num_heads=16, mlp_dim=4096)
VIT_B16_384 = dict(VIT_B16, image_size=384)
N_CLASSES = 6
METRIC = "vit_b16_224_inference_images_per_sec"
UNIT = "images/s"


def fwd_flops_per_image(cfg=VIT_B16, n_prefix=1, n_classes=N_CLASSES) -> float:
    """SURVEY.md 8d / BASELINE.md 4: 2*P*Kp*D + L*(2*N*D*3D + 4*N^2*D + 2*N*D^2 + 4*N*D*M) + 2*D*C."""
    P = (cfg["image_size"] // cfg["patch_size"]) ** 2
    N = P + n_prefix
    D, L, M = cfg["embed_dim"], cfg["num_layers"], cfg["mlp_dim"]
    Kp = cfg["in_channels"] * cfg["patch_size"] ** 2
    return 2 * P * Kp * D + L * (2 * N * D * 3 * D + 4 * N * N * D + 2 * N * D * D + 4 * N * D * M) \
        + 2 * D * n_classes


def dump_outputs(out_dir: str, arrays: dict) -> None:
    """Writes each tensor as <out_dir>/<name>.npy in float32."""
    import numpy as np
    d = Path(out_dir)
    d.mkdir(parents=True, exist_ok=True)
    for name, t in arrays.items():
        np.save(d / f"{name}.npy", t.detach().float().cpu().numpy())


def measured_peaks() -> tuple[dict, str]:
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        return json.loads(p.read_text()), "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


# ------------------------------------------------------------------------------------------------
# clocks / throttle reasons sampled DURING the timed region
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    REASONS = {
        0x0000000000000004: "sw_power_cap",
        0x0000000000000008: "hw_slowdown",
        0x0000000000000020: "sw_thermal_slowdown",
        0x0000000000000040: "hw_thermal_slowdown",
        0x0000000000000080: "hw_power_brake_slowdown",
    }

    def __init__(self, index: int):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thr = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self._nv = pynvml
            self._h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self._nv = None

    def _loop(self):
        nv = self._nv
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self._h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self._h)
                for bit, name in self.REASONS.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop.wait(0.05)

    def __enter__(self):
        if self._nv is not None:
            self._thr = threading.Thread(target=self._loop, daemon=True)
            self._thr.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self._thr is not None:
            self._thr.join()

    def summary(self) -> dict:
        return {"sm_mhz": statistics.median(self.samples) if self.samples else None,
                "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


# ------------------------------------------------------------------------------------------------
# CPU arm: the oracle port on the host cores
# ------------------------------------------------------------------------------------------------
def reference_classifier(kw: dict, n_classes: int = N_CLASSES, seed: int = 0, dropout: float = 0.0):
    """(backbone, head, kind): the reference's own VisionTransformer (evaluation.py:120-157, from
    oracle/_ref or /root/reference) + the oracle wrapper's nn.Linear head (SURVEY.md 8c), built
    under `seed` exactly as vitk.ViTClassifier is - or (None, None, "port") when the reference
    cannot be loaded here."""
    import torch
    try:
        from oracle import ref_loader
        if not ref_loader.reference_available():
            return None, None, "port"
        ev = ref_loader.load("evaluation")
    except Exception:
        return None, None, "port"
    torch.manual_seed(seed)
    bb = ev.VisionTransformer(dropout=dropout, **kw)
    head = torch.nn.Linear(kw["embed_dim"], n_classes)
    return bb, head, "reference"


def _cpu_forward_fn(batch: int):
    """A closure running one CPU forward of the classifier on `batch` synthetic images, the
    reference's classes when present, else the oracle port; plus its kind / description."""
    import torch
    from oracle import vit_oracle as O
    x = O.synthetic_images(batch, VIT_B16["image_size"])
    bb, head, kind = reference_classifier(VIT_B16)
    if bb is not None:
        bb.eval()

        def run():
            return head(bb(x)[:, 0])
        what = ("the reference's VisionTransformer (evaluation.py:120-157, oracle/_ref) + "
                "Linear(768, 6) on the CLS row, eval(), no_grad, torch CPU fp32")
    else:
        import vitk
        torch.manual_seed(0)
        model = vitk.ViTClassifier(num_classes=N_CLASSES, dropout=0.0, **VIT_B16)  # parameter container
        sd = {k: v.detach() for k, v in model.state_dict().items()}

        def run():
            return O.classifier_forward(sd, x, VIT_B16["num_heads"])[1]
        what = "reference algorithm restated in oracle/vit_oracle.py, torch CPU fp32"
    return run, kind, what


def cpu_forward_rate(batch: int, budget_s: float, min_iters: int = 1) -> dict:
    import torch
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    run, kind, what = _cpu_forward_fn(batch)
    with torch.no_grad():
        run()  # warm-up
        times = []
        t_end = time.perf_counter() + budget_s
        while len(times) < min_iters or (time.perf_counter() < t_end and len(times) < 50):
            t0 = time.perf_counter()
            run()
            times.append(time.perf_counter() - t0)
    best = min(times)
    return {"value": batch / best, "unit": UNIT, "cores": cores, "kind": kind,
            "threads": torch.get_num_threads(),
            "sample": f"{what}; batch {batch}, best of {len(times)} "
                      f"(median {batch / statistics.median(times):.1f} img/s), 1 warm-up"}


def run_reference(args) -> None:
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    batch = 32  # configs[0]: the reference's own CPU-runnable case
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    run, kind, what = _cpu_forward_fn(batch)
    steps = args.steps
    warm = min(args.warmup, 1)
    with torch.no_grad():
        for _ in range(max(warm, 1)):
            run()
        t0 = time.perf_counter()
        for _ in range(steps):
            logits = run()
        dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"logits": logits})
    val = batch * steps / dt
    sample = f"{what}, {cores} threads; {steps} steps x batch {batch} of the ViT-B/16 workload"
    _emit(json.dumps({
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus,
        "steps": steps, "warmup": max(warm, 1), "ms_per_step": 1e3 * dt / steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": "ViT-B/16 224px 6-class inference", "batch_per_step": batch,
                   "device": "host CPU"},
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
TRAIN_BATCH = 128


def measure_train_step(vitk, O, dev, world, rank, barrier, steps: int = 8, warmup: int = 3,
                       dropout: float = 0.1) -> dict:
    """BASELINE.json configs[2]: ViT-B/16 6-class fine-tune step (forward saving activations ->
    cross-entropy -> hand-written backward -> NCCL gradient all-reduce -> fused AdamW), bf16,
    128 images per GPU, data parallel. Reported next to the headline inference metric."""
    import torch
    import torch.distributed as dist
    B = TRAIN_BATCH
    torch.manual_seed(0)
    model = vitk.ViTClassifier(num_classes=N_CLASSES, dropout=dropout, **VIT_B16).to(dev).train()
    overlap = os.environ.get("VITK_DP_OVERLAP", "1") != "0"
    reserve = int(os.environ.get("VITK_DP_RESERVE_SMS", "0"))
    tuner = vitk.FineTuner(model, lr=1e-4, weight_decay=1e-4, overlap_allreduce=overlap,
                           reserve_sms=reserve, seed=1000 * rank)
    x = O.synthetic_images(B, VIT_B16["image_size"], seed=99 + rank).to(dev)
    y = O.synthetic_labels(B, N_CLASSES, seed=5 + rank).to(dev)
    for _ in range(warmup):
        loss, _ = tuner.step(x, y)
    barrier()
    n0 = vitk.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(steps):
        loss, _ = tuner.step(x, y)
    ev1.record()
    barrier()
    launches = vitk.launch_count() - n0
    ms = ev0.elapsed_time(ev1)
    if world > 1:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    vitk._lib.profile_enable(True)
    for _ in range(2):
        tuner.step(x, y)
    torch.cuda.synchronize()
    prof = vitk._lib.profile_collect()
    vitk._lib.profile_enable(False)
    ips = world * B * steps / (ms * 1e-3)
    flops = 3.0 * fwd_flops_per_image()
    peaks, _ = measured_peaks()
    tuner_overlap, tuner_sync = tuner.overlap, tuner.grad_sync
    tuner_mc = bool(tuner.peer is not None and tuner.peer.multicast)
    del tuner, model
    torch.cuda.empty_cache()
    return {"metric": "vit_b16_224_finetune_images_per_sec", "value": ips, "unit": UNIT,
            "ms_per_step": ms / steps, "batch_per_gpu": B, "global_batch": B * world,
            "steps": steps, "warmup": warmup, "gpu_launches": int(launches),
            "loss_after": float(loss.item()) * world,
            "tflops": ips / world * flops / 1e12,
            "frac_of_burst_peak": ips / world * flops / 1e12 / float(peaks["bf16_tflops"]),
            "by_kind_ms_per_step": {k: v["ms"] / 2 for k, v in prof.items() if v["launches"]},
            "optimizer": "fused AdamW lr 1e-4 wd 1e-4 (train.py:1598-1602)",
            "dropout": dropout,
            "grad_allreduce": ("none (1 GPU)" if world == 1 else
                               (("sharded reduce + AdamW + broadcast over symmetric memory "
                                 "(csrc/peer_optim.cu; " + ("multimem.ld_reduce / multimem.st through "
                                 "the NVSwitch" if tuner_mc else "peer loads / stores over NVLink") +
                                 "), Adam moments sharded over the ranks") if tuner_sync == "peer" else
                                ("NCCL sum over 14 flat fp32 slices, each started when the backward "
                                 "has produced it (overlapped)" if tuner_overlap else
                                 "NCCL sum over 14 flat fp32 slices after the backward")))}


def measure_detector(vitk, dev, world, barrier, batch: int, steps: int = 6, warmup: int = 3) -> dict:
    """SURVEY.md 8 row f1: evaluation.py's real model call, ViTObjectDetector(images) = ViT-B/16
    backbone + 6-layer detection head (100 queries, 6 + 1 classes), batch-sharded like the
    headline; device-resident inputs, CUDA events, max over ranks."""
    import torch
    import torch.distributed as dist
    torch.manual_seed(0)
    det = vitk.ViTObjectDetector(num_classes=N_CLASSES, num_queries=100, **VIT_B16).to(dev).eval()
    x = torch.randn(batch, 3, VIT_B16["image_size"], VIT_B16["image_size"], device=dev)
    with torch.no_grad():
        for _ in range(warmup):
            out = det(x)
        toks = det.backbone(x)
        barrier()
        n0 = vitk.launch_count()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        ev[0].record()
        for _ in range(steps):
            out = det(x)
        ev[1].record()
        launches = vitk.launch_count() - n0
        for _ in range(steps):
            out = det.detection_head.decode(toks, 1)
        ev[2].record()
        barrier()
    ms, ms_head = ev[0].elapsed_time(ev[1]), ev[1].elapsed_time(ev[2])
    if world > 1:
        t = torch.tensor([ms, ms_head], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, ms_head = float(t[0].item()), float(t[1].item())
    # end to end: pinned host images in, the prediction dict on the host out (evaluation.py:498-502)
    import time
    host = torch.randn(batch, 3, VIT_B16["image_size"], VIT_B16["image_size"]).pin_memory()
    runner = vitk.HostBatchRunner(det, batch, dev)
    for _ in runner.run([host] * 3):
        pass
    barrier()
    t0 = time.perf_counter()
    for res in runner.run([host] * steps):
        pass
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([e2e_s], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item())
    e2e = {"value": world * batch * steps / e2e_s, "unit": UNIT,
           "h2d_bytes_per_step": runner.h2d_bytes_per_step,
           "d2h_bytes_per_step": runner.d2h_bytes_per_step,
           "api": "HostBatchRunner.run over a ViTObjectDetector (pinned f32 NCHW host batches -> "
                  "host class_logits + bbox_coords)"}
    del runner
    P, D, Q, F, L = 196, 768, 100, 2048, 6
    head_flops = (2 * (P + 1) * D * L * 2 * D + L * (2 * Q * D * 3 * D + 4 * Q * Q * D + 4 * Q * D * D
                  + 2 * Q * D * D + 4 * Q * P * D + 4 * Q * D * F) + 2 * Q * D * (N_CLASSES + 5))
    assert bool(torch.isfinite(out["class_logits"]).all())
    del det
    torch.cuda.empty_cache()
    return {"metric": "vit_b16_224_detector_images_per_sec",
            "value": world * batch * steps / (ms * 1e-3), "unit": UNIT,
            "ms_per_step": ms / steps, "head_ms_per_step": ms_head / steps,
            "head_tflops": batch * head_flops / (ms_head / steps * 1e-3) / 1e12,
            "head_gflop_per_image": head_flops / 1e9, "batch_per_gpu": batch,
            "gpu_launches": int(launches), "steps": steps, "warmup": warmup, "e2e": e2e,
            "api": "ViTObjectDetector.forward (evaluation.py:203-241): vitk_forward + "
                   "vitk_detection_head_forward"}


def measure_detector_train(vitk, dev, world, barrier, batch: int = 64, steps: int = 4,
                           warmup: int = 2) -> dict:
    """SURVEY.md 8 rows f1 / f3 under training: train.py:1441-1455 for the detector -
    predictions = model(images) through the encoder bridge and the detection head, the device-side
    SetCriterion.loss_labels (weighted cross-entropy, background weight 0.1) + an L1 box term on
    synthetic targets (the Hungarian assignment is host-side control plane, out of scope), then
    loss.backward() through head and encoder.  No optimizer step: that is the caller's torch.optim."""
    import torch
    import torch.distributed as dist
    torch.manual_seed(0)
    det = vitk.ViTObjectDetector(num_classes=N_CLASSES, num_queries=100, dropout=0.0,
                                 **VIT_B16).to(dev).train()
    for m in det.modules():      # p = 0 everywhere: the configuration the parity tests pin
        if isinstance(m, torch.nn.Dropout):
            m.p = 0.0
        if isinstance(m, torch.nn.MultiheadAttention):
            m.dropout = 0.0
    x = torch.randn(batch, 3, VIT_B16["image_size"], VIT_B16["image_size"], device=dev)
    tgt = torch.randint(0, N_CLASSES + 1, (batch, 100), device=dev)
    box = torch.rand(batch, 100, 4, device=dev)
    w = torch.ones(N_CLASSES + 1, device=dev)
    w[-1] = 0.1

    def step():
        for p in det.parameters():
            p.grad = None
        out = det(x)
        loss = vitk.weighted_cross_entropy(out["class_logits"], tgt, w) + \
            (out["bbox_coords"] - box).abs().mean()
        loss.backward()
        return loss

    for _ in range(warmup):
        loss = step()
    barrier()
    n0 = vitk.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        loss = step()
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    launches = vitk.launch_count() - n0
    if world > 1:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    ok = bool(torch.isfinite(loss).item()) and all(p.grad is not None for p in det.parameters())
    del det
    torch.cuda.empty_cache()
    return {"metric": "vit_b16_224_detector_fwd_bwd_images_per_sec",
            "value": world * batch * steps / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms / steps,
            "batch_per_gpu": batch, "steps": steps, "warmup": warmup, "gpu_launches": int(launches),
            "finite_loss_and_all_grads": ok,
            "what": "ViTObjectDetector forward + weighted CE / L1 loss + backward through the "
                    "detection head (vitk_detection_head_backward) and the encoder "
                    "(vitk_backward_tokens); decoder dropout off (p = 0); no optimizer step"}


def _max_over_ranks(vals, dev, world):
    import torch
    import torch.distributed as dist
    if world == 1:
        return [float(v) for v in vals]
    t = torch.tensor([float(v) for v in vals], device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return [float(v) for v in t.tolist()]


def measure_inference_leg(vitk, O, dev, world, rank, barrier, label: str, kw: dict,
                          batch_per_gpu: int, scaling: str, steps: int = 8, warmup: int = 3) -> dict:
    """One more BASELINE.json configuration, measured exactly like the headline: random-init
    weights, device-resident synthetic images (a different shard per rank), CUDA events around
    `steps` forwards, max over ranks; then the per-kernel-class times of the same steps."""
    import torch
    torch.manual_seed(0)
    model = vitk.ViTClassifier(num_classes=N_CLASSES, dropout=0.0, **kw).to(dev).eval()
    x = O.synthetic_images(batch_per_gpu, kw["image_size"], seed=4321 + rank).to(dev)
    with torch.no_grad():
        for _ in range(warmup):
            logits = model(x)
        barrier()
        n0 = vitk.launch_count()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for _ in range(steps):
            logits = model(x)
        ev1.record()
        barrier()
        launches = vitk.launch_count() - n0
        (ms,) = _max_over_ranks([ev0.elapsed_time(ev1)], dev, world)
        vitk._lib.profile_enable(True)
        for _ in range(2):
            model(x)
        torch.cuda.synchronize()
        prof = vitk._lib.profile_collect()
        vitk._lib.profile_enable(False)
    assert bool(torch.isfinite(logits).all())
    flops = fwd_flops_per_image(kw)
    peaks, _ = measured_peaks()
    ips = world * batch_per_gpu * steps / (ms * 1e-3)
    tf = ips / world * flops / 1e12
    del model, x
    torch.cuda.empty_cache()
    P = (kw["image_size"] // kw["patch_size"]) ** 2
    return {"workload": label, "value": ips, "unit": UNIT, "ms_per_step": ms / steps,
            "batch_per_gpu": batch_per_gpu, "global_batch": batch_per_gpu * world,
            "scaling": scaling, "tokens_per_image": P + 1, "gflop_per_image": flops / 1e9,
            "tflops_per_gpu": tf, "frac_of_burst_peak": tf / float(peaks["bf16_tflops"]),
            "frac_of_sustained_peak": tf / float(peaks.get("bf16_tflops_sustained",
                                                           peaks["bf16_tflops"])),
            "steps": steps, "warmup": warmup, "gpu_launches": int(launches),
            "by_kind_ms_per_step": {k: v["ms"] / 2 for k, v in prof.items() if v["launches"]}}


def parity_check(model, x_dev, logits_dev, O, n: int = 8, tol: float = 2e-2) -> dict:
    """Logits of the first `n` images of the TIMED batch against the oracle (fp32, CPU, the same
    random-init weights): north_star's bar is 2e-2 absolute in bf16 and identical top-1.  Top-1 is
    compared where the oracle's own top-2 margin exceeds the tolerance (random-init ViT logits
    barely depend on the image, SURVEY.md 4)."""
    import torch
    sd = {k: v.detach().cpu() for k, v in model.state_dict().items()}
    heads = model.backbone.transformer_blocks[0].attention.num_heads
    with torch.no_grad():
        _, ref = O.classifier_forward(sd, x_dev[:n].cpu(), heads, dtype=torch.float32)
    got = logits_dev[:n].float().cpu()
    err = float((got - ref).abs().max())
    top2 = ref.topk(2, dim=-1).values
    decided = (top2[:, 0] - top2[:, 1]) > tol
    same = bool((got.argmax(-1) == ref.argmax(-1))[decided].all())
    ok = err < tol and same
    out = {"images": n, "max_abs_logit_diff": err, "tolerance": tol, "top1_identical": same,
           "top1_compared": int(decided.sum()), "ok": ok,
           "against": "oracle.classifier_forward fp32 on the host (pinned to the reference's classes "
                      "by tests/golden)"}
    if not ok:
        raise SystemExit(f"bench.py: parity check of the timed batch FAILED: {out}")
    return out


def gpu_eager_baseline(O, dev, batch: int, train_batch: int, steps: int = 10) -> dict:
    """The bar SURVEY.md 2.1 names: the reference's own modules run by PyTorch eager (cuBLASLt /
    ATen kernels) on THIS GPU under torch.autocast('cuda', bfloat16) - train.py:1441 with the
    dtype made explicit.  Inference at the headline batch and one fine-tune step (cross-entropy on
    the CLS head, torch.optim.AdamW per train.py:1598-1602).  Outside every timed region of the
    vitk arm; none of this repository's kernels run here."""
    import torch
    import torch.nn.functional as F
    bb, head, kind = reference_classifier(VIT_B16, dropout=0.1)
    x = O.synthetic_images(batch, VIT_B16["image_size"], seed=1234).to(dev)
    if bb is not None:
        bb, head = bb.to(dev), head.to(dev)

        def fwd(inp):
            return head(bb(inp)[:, 0])
        params = list(bb.parameters()) + list(head.parameters())
        set_train = lambda on: (bb.train(on), head.train(on))
        what = "the reference's VisionTransformer (oracle/_ref) + Linear head"
    else:
        import vitk
        torch.manual_seed(0)
        cont = vitk.ViTClassifier(num_classes=N_CLASSES, dropout=0.0, **VIT_B16)
        sd = {k: v.detach().to(dev).requires_grad_(True) for k, v in cont.state_dict().items()}

        def fwd(inp):
            return O.classifier_forward(sd, inp, VIT_B16["num_heads"])[1]
        params = list(sd.values())
        set_train = lambda on: None
        what = "oracle.classifier_forward (restatement; no dropout)"
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    set_train(False)
    with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16):
        for _ in range(3):
            fwd(x)
        torch.cuda.synchronize()
        ev0.record()
        for _ in range(steps):
            out = fwd(x)
        ev1.record()
        torch.cuda.synchronize()
    ms_inf = ev0.elapsed_time(ev1) / steps
    # one fine-tune step
    set_train(True)
    xt = x[:train_batch]
    y = O.synthetic_labels(train_batch, N_CLASSES, seed=5).to(dev)
    opt = torch.optim.AdamW(params, lr=1e-4, weight_decay=1e-4)
    tsteps = max(3, steps // 2)

    def step():
        opt.zero_grad()
        with torch.autocast("cuda", dtype=torch.bfloat16):
            loss = F.cross_entropy(fwd(xt).float(), y)
        loss.backward()
        opt.step()
        return loss
    for _ in range(2):
        step()
    torch.cuda.synchronize()
    ev0.record()
    for _ in range(tsteps):
        loss = step()
    ev1.record()
    torch.cuda.synchronize()
    ms_tr = ev0.elapsed_time(ev1) / tsteps
    flops = fwd_flops_per_image()
    del opt, params
    torch.cuda.empty_cache()
    return {"kind": f"{kind}, cuda eager, autocast bf16", "what": what,
            "inference": {"value": batch / (ms_inf * 1e-3), "unit": UNIT, "ms_per_step": ms_inf,
                          "batch": batch, "tflops": batch / (ms_inf * 1e-3) * flops / 1e12},
            "train_step": {"value": train_batch / (ms_tr * 1e-3), "unit": UNIT,
                           "ms_per_step": ms_tr, "batch": train_batch, "dropout": 0.1,
                           "tflops": train_batch / (ms_tr * 1e-3) * 3 * flops / 1e12,
                           "loss_after": float(loss.item())}}


DP_CHECK_KW = dict(VIT_B16, num_layers=2)   # ViT-B/16 width and token count, two blocks


def dp_check(vitk, O, dev, world, rank, steps: int = 3, batch: int = 8) -> dict:
    """Data-parallel equivalence on the hardware (SURVEY.md 4 tier 5): (1) one DP step - every rank
    on its own shard, NCCL gradient all-reduce - gives the gradients of a single-GPU step on the
    concatenated batch, within reduction-order tolerance; (2) after `steps` optimisation steps the
    parameters are bitwise identical on every rank."""
    import torch
    import torch.distributed as dist
    torch.manual_seed(0)
    model = vitk.ViTClassifier(num_classes=N_CLASSES, dropout=0.0, **DP_CHECK_KW).to(dev).train()
    sd0 = {k: v.clone() for k, v in model.state_dict().items()}
    tuner = vitk.FineTuner(model, lr=1e-4, weight_decay=1e-4)
    flat0 = tuner.state.flat.clone()
    x = O.synthetic_images(batch, DP_CHECK_KW["image_size"], seed=777 + rank).to(dev)
    y = O.synthetic_labels(batch, N_CLASSES, seed=55 + rank).to(dev)
    loss, _ = tuner.step(x, y)
    # summed over ranks, already scaled by 1/(B*world); with the peer-memory optimizer every rank
    # holds the sum of its own shard only
    pieces = tuner.reduced_grad_ranges()
    g_dp = torch.cat([tuner.state.grad[a:b] for a, b in pieces])
    lt = loss.clone()
    dist.all_reduce(lt)
    # the single-GPU step on the concatenated batch, from the same initial weights
    xs = [torch.empty_like(x) for _ in range(world)]
    ys = [torch.empty_like(y) for _ in range(world)]
    dist.all_gather(xs, x)
    dist.all_gather(ys, y)
    torch.manual_seed(0)
    solo = vitk.ViTClassifier(num_classes=N_CLASSES, dropout=0.0, **DP_CHECK_KW).to(dev).train()
    solo.load_state_dict(sd0)
    solo_tuner = vitk.FineTuner(solo, lr=1e-4, weight_decay=1e-4, data_parallel=False)
    loss1, _ = solo_tuner.step(torch.cat(xs), torch.cat(ys))
    g1 = torch.cat([solo_tuner.state.grad[a:b] for a, b in pieces])
    sq = torch.stack([(g_dp - g1).double().pow(2).sum(), g1.double().pow(2).sum()])
    dist.all_reduce(sq)
    rel = float((sq[0] / (sq[1] + 1e-60)).sqrt())
    loss_diff = abs(float(lt.item()) - float(loss1.item()))
    for _ in range(steps - 1):
        tuner.step(x, y)
    # the same steps with the gradient exchange over NCCL (all-reduce + replicated AdamW): the two
    # transports must agree up to the order of the cross-rank sum
    sync = tuner.grad_sync
    vs_nccl = None
    if sync == "peer":
        torch.manual_seed(0)
        other = vitk.ViTClassifier(num_classes=N_CLASSES, dropout=0.0, **DP_CHECK_KW).to(dev).train()
        other.load_state_dict(sd0)
        other_tuner = vitk.FineTuner(other, lr=1e-4, weight_decay=1e-4, grad_sync="nccl")
        for _ in range(steps):
            other_tuner.step(x, y)
        # relative L2 error of the parameter UPDATE (Adam turns a last-bit difference of a
        # near-zero gradient into a difference of the order of lr in that one element)
        du = (other_tuner.state.flat - tuner.state.flat).double().norm()
        dn = (other_tuner.state.flat - flat0).double().norm()
        vs_nccl = float(du / (dn + 1e-30))
        del other_tuner, other
    flat = tuner.state.flat
    lo, hi = flat.clone(), flat.clone()
    dist.all_reduce(lo, op=dist.ReduceOp.MIN)
    dist.all_reduce(hi, op=dist.ReduceOp.MAX)
    identical = bool(torch.equal(lo, hi))
    # (vs_nccl is reported, not gated: Adam turns a last-bit difference of a near-zero gradient into
    # an lr-sized difference of that element, so the two summation orders drift apart by design)
    ok = identical and rel < 2e-2 and loss_diff < 1e-3
    out = {"ok": ok, "grad_sync": sync, "params_bitwise_identical_across_ranks": identical,
           "peer_vs_nccl_relative_error_of_the_update": vs_nccl, "steps": steps,
           "grad_rel_l2_vs_single_gpu_concatenated_batch": rel, "grad_tolerance": 2e-2,
           "loss_abs_diff_vs_single_gpu": loss_diff,
           "config": f"ViT-B/16 width, 2 blocks, {batch} images per rank x {world} ranks, dropout 0"}
    del tuner, solo_tuner, model, solo
    torch.cuda.empty_cache()
    if not ok:
        raise SystemExit(f"bench.py: data-parallel check FAILED: {out}")
    return out


def gemm_traffic_per_launch(batch: int):
    """dram__bytes_read + dram__bytes_write per GEMM launch from the committed ncu capture
    (profiles/gemm_dram_traffic.json names the .csv it was read from); None off that geometry."""
    p = ROOT / "profiles" / "gemm_dram_traffic.json"
    if not p.exists():
        return None, None
    d = json.loads(p.read_text())
    if int(d.get("batch", -1)) != batch:
        return None, None
    return float(d["mean_bytes_per_launch"]), f"profiles/gemm_dram_traffic.json <- {d['source']}"


def run_vitk(args) -> None:
    import torch
    import torch.distributed as dist
    import vitk
    from oracle import vit_oracle as O

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device - the vitk path has no CPU fallback "
                         "(use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        opts = None
        if int(os.environ.get("VITK_NCCL_MAX_CTAS", "0")) > 0:
            opts = dist.ProcessGroupNCCL.Options()
            opts.config.max_ctas = int(os.environ["VITK_NCCL_MAX_CTAS"])
            opts.config.min_ctas = 1
        dist.init_process_group("nccl", device_id=dev, pg_options=opts)
    n_gpus = world

    B = args.batch
    global TRAIN_BATCH
    TRAIN_BATCH = args.train_batch
    torch.manual_seed(0)
    model = vitk.ViTClassifier(num_classes=N_CLASSES, dropout=0.0, **VIT_B16).to(dev).eval()
    # every rank owns a different shard of the global batch (weak scaling: B images per GPU)
    x_host = O.synthetic_images(B, VIT_B16["image_size"], seed=1234 + rank).pin_memory()
    x_dev = x_host.to(dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    with torch.no_grad():
        for _ in range(max(args.warmup, 3)):
            logits = model(x_dev)
        barrier()
        launches0 = vitk.launch_count()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with ClockSampler(local) as clk:
            ev0.record()
            for _ in range(args.steps):
                logits = model(x_dev)
            ev1.record()
            barrier()
        launches = vitk.launch_count() - launches0
        ms = ev0.elapsed_time(ev1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        value = n_gpus * B * args.steps / (ms * 1e-3)
        if args.dump_outputs:
            shards = [logits]
            if world > 1:
                shards = [torch.empty_like(logits) for _ in range(world)]
                dist.all_gather(shards, logits)
            if rank == 0:
                dump_outputs(args.dump_outputs, {"logits": torch.cat(shards)})

        # ---- per-kernel-class device times over the same steps (events around every launch)
        vitk._lib.profile_enable(True)
        for _ in range(args.steps):
            model(x_dev)
        torch.cuda.synchronize()
        prof = vitk._lib.profile_collect()
        vitk._lib.profile_enable(False)

        # ---- opt-in variant, reported NEXT TO the headline and never in it: the same logits with
        #      the last block evaluated for the CLS rows only (vitk_forward_cls - what the head does
        #      not read is not computed; the headline above evaluates every token, as the reference does)
        for _ in range(3):
            logits_p = model.classify_pruned(x_dev)
        barrier()
        evp0, evp1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        evp0.record()
        for _ in range(args.steps):
            logits_p = model.classify_pruned(x_dev)
        evp1.record()
        barrier()
        ms_p = evp0.elapsed_time(evp1)
        if world > 1:
            t = torch.tensor([ms_p], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms_p = float(t.item())
        pruned = {"value": n_gpus * B * args.steps / (ms_p * 1e-3), "unit": UNIT,
                  "ms_per_step": ms_p / args.steps,
                  "max_abs_logit_diff_vs_full": float((logits_p - logits).abs().max().item()),
                  "api": "ViTClassifier.classify_pruned (vitk_forward_cls): last encoder block "
                         "evaluated for the CLS rows only; not part of `value`"}

        # ---- end to end through the host-buffer API: H2D of the images + D2H of the logits per step
        runner = vitk.HostBatchRunner(model, B, dev)
        for _ in runner.run([x_host] * 3):
            pass
        barrier()
        t0 = time.perf_counter()
        n_out = 0
        for out in runner.run([x_host] * args.steps):
            n_out += out.shape[0]
        torch.cuda.synchronize()
        e2e_s = time.perf_counter() - t0
        if world > 1:
            t = torch.tensor([e2e_s], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            e2e_s = float(t.item())
        assert n_out == B * args.steps
        e2e_value = n_gpus * B * args.steps / e2e_s

        # ---- the same stream with raw 8-bit images as the host buffers (Normalize + ToTensorV2 of
        #      evaluation.py:362-364 fused into the patch gather on the device): reported next to
        #      `e2e`, which keeps the reference's own boundary (normalised f32 NCHW host tensors)
        g8 = torch.Generator().manual_seed(1234 + rank)
        u8_host = torch.randint(0, 256, (B, VIT_B16["image_size"], VIT_B16["image_size"], 3),
                                generator=g8, dtype=torch.uint8).pin_memory()
        runner8 = vitk.HostBatchRunner(model, B, dev, input_dtype=torch.uint8)
        for _ in runner8.run([u8_host] * 3):
            pass
        barrier()
        t0 = time.perf_counter()
        for out in runner8.run([u8_host] * args.steps):
            pass
        torch.cuda.synchronize()
        e2e8_s = time.perf_counter() - t0
        if world > 1:
            t = torch.tensor([e2e8_s], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            e2e8_s = float(t.item())
        e2e8_value = n_gpus * B * args.steps / e2e8_s

    # the reference trains with dropout 0.1 (train.py:519,559,639); the p = 0 step is the one the
    # parity tests pin, reported next to it
    train = None if args.no_train else measure_train_step(vitk, O, dev, world, rank, barrier)
    train0 = None if args.no_train else measure_train_step(vitk, O, dev, world, rank, barrier,
                                                           steps=5, dropout=0.0)

    detector = None if args.no_train else measure_detector(vitk, dev, world, barrier, B)
    detector_train = None if args.no_train else measure_detector_train(vitk, dev, world, barrier)

    # ---- the other BASELINE.json configurations, each under the same timing rules
    legs = []
    if not args.no_configs:
        st = min(args.steps, 8)
        legs.append(measure_inference_leg(
            vitk, O, dev, world, rank, barrier, "ViT-L/16 224px inference, 256 images per GPU "
            "(BASELINE.json configs[3], weak)", VIT_L16, 256, "weak", steps=st))
        if world > 1:
            legs.append(measure_inference_leg(
                vitk, O, dev, world, rank, barrier, f"ViT-L/16 224px inference, global batch 256 = "
                f"{256 // world} images per GPU (BASELINE.json configs[3], strong)", VIT_L16,
                256 // world, "strong", steps=st))
        legs.append(measure_inference_leg(
            vitk, O, dev, world, rank, barrier, "ViT-B/16 384px (577 tokens) inference, 64 images "
            "per GPU (BASELINE.json configs[4])", VIT_B16_384, 64, "weak", steps=st))
    dp = dp_check(vitk, O, dev, world, rank) if (world > 1 and not args.no_train) else None

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    parity = parity_check(model, x_dev, logits, O)
    eager = None
    if n_gpus == 1 and not args.no_eager_baseline:
        eager = gpu_eager_baseline(O, dev, B, TRAIN_BATCH)
    h2d, d2h = runner.h2d_bytes_per_step, runner.d2h_bytes_per_step
    h2d8, d2h8 = runner8.h2d_bytes_per_step, runner8.d2h_bytes_per_step
    peaks, peak_src = measured_peaks()
    flops_img = fwd_flops_per_image()
    gemm = prof["gemm"]
    gemm_tflops = gemm["work"] / (gemm["ms"] * 1e-3) / 1e12 if gemm["ms"] > 0 else 0.0
    # the GEMM launches are timed inside a multi-second loop under the power cap -> sustained peak
    peak_tf = float(peaks.get("bf16_tflops_sustained", peaks["bf16_tflops"]))
    total_prof_ms = sum(v["ms"] for v in prof.values()) or 1.0
    traffic, traffic_src = gemm_traffic_per_launch(B)
    roofline = {
        "bound": "tensor", "kernel": "gemm_tn_kernel (tcgen05, all Linear/Conv2d contractions)",
        "achieved": gemm_tflops, "peak": peak_tf, "unit": "TFLOP/s",
        "frac": gemm_tflops / peak_tf,
        "frac_of_burst_peak": gemm_tflops / float(peaks["bf16_tflops"]),
        # dram__bytes_read + dram__bytes_write per launch (ncu --set full), read from the
        # committed summary of the capture; algorithmic bytes beside it there
        "traffic": traffic, "traffic_source": traffic_src,
        "peak_source": f"{peak_src} MEASURED_PEAKS.json bf16_tflops_sustained (the GEMMs are timed "
                       f"inside a multi-second loop under the power cap); burst "
                       f"{peaks['bf16_tflops']} -> frac_of_burst_peak",
        "avg_launch_ms": gemm["ms"] / max(gemm["launches"], 1),
        "flops_per_launch": gemm["work"] / max(gemm["launches"], 1),
        "share_of_step": gemm["ms"] / total_prof_ms,
        "by_kind_ms_per_step": {k: v["ms"] / args.steps for k, v in prof.items() if v["launches"]},
        "hbm_kernels_gbs": {k: v["work"] / (v["ms"] * 1e-3) / 1e9
                            for k, v in prof.items() if k in ("layernorm", "patchify") and v["ms"] > 0},
        "whole_step_tflops": value / n_gpus * flops_img / 1e12,
        "whole_step_frac_of_burst_peak": value / n_gpus * flops_img / 1e12 / float(peaks["bf16_tflops"]),
    }
    cpu = cpu_forward_rate(32, budget_s=15.0) if n_gpus == 1 and not args.no_cpu_baseline else None
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": n_gpus, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": "ViT-B/16 224px 6-class inference (BASELINE.json configs[1])",
                   "batch_per_gpu": B, "global_batch": B * n_gpus, "tokens_per_image": 197,
                   "gflop_per_image": flops_img / 1e9, "parallelism": f"batch-sharded x{n_gpus}",
                   "l2_policy": "per-step working set ~1.0 GB (activations) + 154 MB images > 126 MB L2"},
        "clocks": clk.summary(),
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": d2h,
                "api": "HostBatchRunner.run (pinned f32 NCHW host batches, as evaluation.py:499 "
                       "copies them -> host logits)"},
        "e2e_uint8_input": {"value": e2e8_value, "unit": UNIT,
                            "h2d_bytes_per_step": h2d8,
                            "d2h_bytes_per_step": d2h8,
                            "api": "HostBatchRunner(input_dtype=uint8): raw u8 NHWC host batches, "
                                   "Normalize + ToTensorV2 on the device (vitk_forward_u8)"},
        "gpu_launches": int(launches),
        "roofline": roofline,
    }
    if train is not None:
        line["train_step"] = train
        line["train_step_no_dropout"] = {k: train0[k] for k in
                                         ("value", "unit", "ms_per_step", "tflops", "dropout")}
    line["cls_only_tail"] = pruned
    if detector is not None:
        line["detector"] = detector
    if detector_train is not None:
        line["detector_train"] = detector_train
    if legs:
        line["configs"] = legs
    line["parity_check"] = parity
    if dp is not None:
        line["dp_check"] = dp
    if eager is not None:
        line["gpu_eager_baseline"] = eager
        line["gpu_eager_baseline"]["vitk_over_eager_inference"] = value / eager["inference"]["value"]
        if train is not None:
            line["gpu_eager_baseline"]["vitk_over_eager_train_step"] = \
                train["value"] / eager["train_step"]["value"]
    if cpu is not None:
        line["cpu_baseline"] = cpu
    _emit(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def _emit(line: str) -> None:
    """The one JSON line goes to the process's original stdout; anything a library writes to fd 1
    meanwhile (e.g. NCCL's version banner) was diverted to stderr by main()."""
    os.write(_REAL_STDOUT, (line + "\n").encode())


_REAL_STDOUT = 1


def main():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--batch", type=int, default=256, help="images per GPU per step")
    ap.add_argument("--impl", choices=["vitk", "reference"], default="vitk")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-train", action="store_true", help="skip the fine-tune step measurement")
    ap.add_argument("--train-batch", type=int, default=128, help="images per GPU per train step")
    ap.add_argument("--no-configs", action="store_true",
                    help="skip the ViT-L/16 and 384 px legs (BASELINE.json configs[3], configs[4])")
    ap.add_argument("--no-eager-baseline", action="store_true",
                    help="skip the PyTorch-eager bf16 run of the reference's classes on this GPU")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the logits of the last timed step to DIR/logits.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_vitk(args)


if __name__ == "__main__":
    main()
