"""ctypes binding of libvitk.so — the C ABI declared in include/vitk.h.

There is deliberately no fallback: if the shared library is missing or a call fails, a
`VitkError` is raised.  PyTorch only supplies device buffers (`Tensor.data_ptr()`) and the current
CUDA stream.
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

import os

PKG_DIR = Path(__file__).resolve().parent
# VITK_LIB: another build of the same library (same ABI), for A/B timing of kernel variants on one box
LIB_PATH = Path(os.environ["VITK_LIB"]) if os.environ.get("VITK_LIB") else PKG_DIR / "libvitk.so"

ABI_VERSION = 6

EPI_BF16 = 0
EPI_GELU_BF16 = 1
EPI_RESID_F32 = 2
EPI_F32 = 3
EPI_DGELU_BF16 = 4
EPI_GELU_TANH_BF16 = 6
EPI_RELU_BF16 = 7


class VitkError(RuntimeError):
    pass


class VitkConfig(C.Structure):
    _fields_ = [
        ("image_size", C.c_int),
        ("patch_size", C.c_int),
        ("in_channels", C.c_int),
        ("embed_dim", C.c_int),
        ("num_layers", C.c_int),
        ("num_heads", C.c_int),
        ("mlp_dim", C.c_int),
        ("n_prefix_tokens", C.c_int),
        ("n_classes", C.c_int),
        ("precision", C.c_int),
        ("ln_eps", C.c_float),
        ("dropout_p", C.c_float),
        ("seed", C.c_uint64),
    ]


class VitkBlockWeights(C.Structure):
    _fields_ = [
        ("ln1_w", C.c_void_p), ("ln1_b", C.c_void_p),
        ("qkv_w", C.c_void_p), ("qkv_b", C.c_void_p),
        ("proj_w", C.c_void_p), ("proj_b", C.c_void_p),
        ("ln2_w", C.c_void_p), ("ln2_b", C.c_void_p),
        ("fc1_w", C.c_void_p), ("fc1_b", C.c_void_p),
        ("fc2_w", C.c_void_p), ("fc2_b", C.c_void_p),
        # optional: LayerNorm folded into qkv / linear1 (vitk_fold_layernorm); NULL = not folded
        ("qkv_w_ln", C.c_void_p), ("qkv_b_ln", C.c_void_p),
        ("fc1_w_ln", C.c_void_p), ("fc1_b_ln", C.c_void_p),
    ]


class VitkWeights(C.Structure):
    _fields_ = [
        ("patch_w", C.c_void_p), ("patch_b", C.c_void_p),
        ("cls_token", C.c_void_p), ("dist_token", C.c_void_p), ("pos_embed", C.c_void_p),
        ("blocks", C.POINTER(VitkBlockWeights)),
        ("ln_f_w", C.c_void_p), ("ln_f_b", C.c_void_p),
        ("head_w", C.c_void_p), ("head_b", C.c_void_p),
    ]


class VitkDetectionHeadConfig(C.Structure):
    _fields_ = [("embed_dim", C.c_int), ("num_heads", C.c_int), ("ffn_dim", C.c_int),
                ("num_layers", C.c_int), ("num_queries", C.c_int), ("num_outputs", C.c_int),
                ("ln_eps", C.c_float), ("dropout_p", C.c_float), ("seed", C.c_uint64)]


class VitkDecoderLayerWeights(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in (
        "sa_in_w", "sa_in_b", "sa_out_w", "sa_out_b", "ca_q_w", "ca_q_b", "ca_out_w", "ca_out_b",
        "ff1_w", "ff1_b", "ff2_w", "ff2_b", "norm1_w", "norm1_b", "norm2_w", "norm2_b", "norm3_w",
        "norm3_b")]


class VitkDetectionHeadWeights(C.Structure):
    _fields_ = [("object_queries", C.c_void_p), ("layers", C.POINTER(VitkDecoderLayerWeights)),
                ("ca_kv_w", C.c_void_p), ("ca_kv_b", C.c_void_p), ("class_w", C.c_void_p),
                ("class_b", C.c_void_p), ("bbox_w", C.c_void_p), ("bbox_b", C.c_void_p)]


class VitkDecoderLayerWeightsT(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("sa_in_wt", "sa_out_wt", "ca_q_wt", "ca_out_wt", "ff1_wt",
                                          "ff2_wt")]


class VitkDetectionHeadWeightsT(C.Structure):
    _fields_ = [("layers", C.POINTER(VitkDecoderLayerWeightsT)), ("ca_kv_wt", C.c_void_p)]


class VitkDecoderLayerGrads(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in (
        "sa_in_w", "sa_in_b", "sa_out_w", "sa_out_b", "ca_q_w", "ca_q_b", "ca_out_w", "ca_out_b",
        "ff1_w", "ff1_b", "ff2_w", "ff2_b", "norm1_w", "norm1_b", "norm2_w", "norm2_b", "norm3_w",
        "norm3_b")]


class VitkDetectionHeadGrads(C.Structure):
    _fields_ = [("object_queries", C.c_void_p), ("layers", C.POINTER(VitkDecoderLayerGrads)),
                ("ca_kv_w", C.c_void_p), ("ca_kv_b", C.c_void_p), ("class_w", C.c_void_p),
                ("class_b", C.c_void_p), ("bbox_w", C.c_void_p), ("bbox_b", C.c_void_p)]


MAX_PEERS = 16


class VitkPeerBuffers(C.Structure):
    _fields_ = [("world", C.c_int), ("rank", C.c_int),
                ("grad", C.c_void_p * MAX_PEERS), ("param", C.c_void_p * MAX_PEERS),
                ("shadow", C.c_void_p * MAX_PEERS), ("guard", C.c_void_p * MAX_PEERS),
                ("grad_mc", C.c_void_p), ("param_mc", C.c_void_p), ("shadow_mc", C.c_void_p)]


# name -> (restype, argtypes); must list every symbol include/vitk.h declares.
_SIGNATURES = {
    "vitk_abi_version": (C.c_int, []),
    "vitk_last_error": (C.c_char_p, []),
    "vitk_launch_count": (C.c_longlong, []),
    "vitk_gemm_set_cta_group": (C.c_int, [C.c_int]),
    "vitk_gemm_set_direct_epilogue": (C.c_int, [C.c_int]),
    "vitk_debug_gemm_trace": (C.c_int, [C.c_void_p, C.c_int]),
    "vitk_set_layernorm_folding": (C.c_int, [C.c_int]),
    "vitk_fold_layernorm": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                      C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "vitk_stats_parts": (C.c_int, [C.c_int]),
    "vitk_row_stats": (C.c_int, [C.c_void_p, C.c_longlong, C.c_void_p, C.c_longlong, C.c_void_p,
                                 C.c_int, C.c_int, C.c_void_p]),
    "vitk_gemm_resid_stats": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                        C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                        C.c_void_p]),
    "vitk_gemm_layernorm_folded": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int,
                                             C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                             C.c_int, C.c_float, C.c_void_p, C.c_int, C.c_void_p]),
    "vitk_attention_set_impl": (C.c_int, [C.c_int]),
    "vitk_reserve_sms": (C.c_int, [C.c_int]),
    "vitk_postprocess_scores": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                          C.c_void_p, C.c_void_p, C.c_void_p]),
    "vitk_postprocess_detections": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                              C.c_float, C.c_void_p, C.c_void_p, C.c_void_p,
                                              C.c_void_p, C.c_void_p]),
    "vitk_linear_rows": (C.c_int, [C.c_void_p, C.c_longlong, C.c_void_p, C.c_void_p, C.c_void_p,
                                   C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "vitk_linear_rows_backward": (C.c_int, [C.c_void_p, C.c_longlong, C.c_void_p, C.c_void_p,
                                            C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int,
                                            C.c_int, C.c_void_p]),
    "vitk_dropout_keep_mask": (C.c_int, [C.c_float, C.c_uint, C.c_int, C.c_int, C.c_longlong,
                                         C.c_void_p, C.c_void_p]),
    "vitk_profile_enable": (C.c_int, [C.c_int]),
    "vitk_profile_collect": (C.c_int, [C.POINTER(C.c_double), C.POINTER(C.c_double),
                                       C.POINTER(C.c_longlong), C.c_int]),
    "vitk_workspace_bytes": (C.c_int, [C.POINTER(VitkConfig), C.c_int, C.POINTER(C.c_size_t)]),
    "vitk_forward": (C.c_int, [C.POINTER(VitkConfig), C.POINTER(VitkWeights), C.c_void_p, C.c_int,
                               C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "vitk_forward_cls": (C.c_int, [C.POINTER(VitkConfig), C.POINTER(VitkWeights), C.c_void_p, C.c_int,
                                   C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "vitk_gemm": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int,
                            C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p,
                            C.c_void_p, C.c_int, C.c_float, C.c_float, C.c_void_p]),
    "vitk_gemm_resid_layernorm": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                            C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                            C.c_float, C.c_void_p, C.c_void_p, C.c_void_p,
                                            C.c_void_p]),
    "vitk_gemm_wgrad": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int,
                                  C.c_void_p, C.c_int, C.c_float, C.c_float, C.c_int, C.c_void_p]),
    "vitk_layernorm": (C.c_int, [C.c_void_p, C.c_longlong, C.c_void_p, C.c_void_p, C.c_void_p,
                                 C.c_int, C.c_longlong, C.c_void_p, C.c_void_p, C.c_int, C.c_int,
                                 C.c_float, C.c_void_p]),
    "vitk_attention": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                 C.c_int, C.c_void_p]),
    "vitk_patchify": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int,
                                C.c_void_p]),
    "vitk_cast_f32_to_bf16": (C.c_int, [C.c_void_p, C.c_void_p, C.c_longlong, C.c_void_p]),
    "vitk_split3": (C.c_int, [C.c_void_p, C.c_longlong, C.c_void_p, C.c_longlong, C.c_int, C.c_int,
                              C.c_void_p]),
    # ---- training step
    "vitk_train_workspace_bytes": (C.c_int, [C.POINTER(VitkConfig), C.c_int, C.POINTER(C.c_size_t),
                                             C.POINTER(C.c_size_t)]),
    "vitk_forward_u8": (C.c_int, [C.POINTER(VitkConfig), C.POINTER(VitkWeights), C.c_void_p,
                                  C.POINTER(C.c_float), C.POINTER(C.c_float), C.c_int, C.c_void_p,
                                  C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "vitk_forward_train": (C.c_int, [C.POINTER(VitkConfig), C.POINTER(VitkWeights), C.c_void_p,
                                     C.c_int, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p,
                                     C.c_size_t, C.c_void_p]),
    "vitk_classifier_loss_backward": (C.c_int, [C.POINTER(VitkConfig), C.POINTER(VitkWeights),
                                                C.c_void_p, C.c_void_p, C.c_void_p, C.c_int,
                                                C.c_float, C.c_void_p, C.c_void_p, C.c_void_p,
                                                C.c_void_p, C.c_void_p]),
    "vitk_classifier_loss_backward_ev": (C.c_int, [C.POINTER(VitkConfig), C.POINTER(VitkWeights),
                                                   C.c_void_p, C.c_void_p, C.c_void_p, C.c_int,
                                                   C.c_float, C.c_void_p, C.c_void_p, C.c_void_p,
                                                   C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "vitk_backward_tokens": (C.c_int, [C.POINTER(VitkConfig), C.POINTER(VitkWeights), C.c_void_p,
                                       C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p,
                                       C.c_void_p]),
    "vitk_adamw_step": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                  C.c_longlong, C.c_double, C.c_double, C.c_double, C.c_double,
                                  C.c_double, C.c_int, C.c_float, C.c_void_p]),
    "vitk_adamw_step_guarded": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                          C.c_longlong, C.c_double, C.c_double, C.c_double,
                                          C.c_double, C.c_double, C.c_int, C.c_float, C.c_void_p,
                                          C.c_void_p]),
    "vitk_grad_guard_scan": (C.c_int, [C.c_void_p, C.c_longlong, C.c_void_p, C.c_int, C.c_void_p]),
    "vitk_grad_guard_finish": (C.c_int, [C.c_void_p, C.c_void_p]),
    "vitk_transpose_bf16_batched": (C.c_int, [C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p),
                                              C.POINTER(C.c_int), C.POINTER(C.c_int), C.c_void_p]),
    "vitk_layernorm_bwd": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                     C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p,
                                     C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "vitk_attention_bwd": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                     C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "vitk_colsum_bf16": (C.c_int, [C.c_void_p, C.c_longlong, C.c_int, C.c_int, C.c_void_p,
                                   C.c_void_p]),
    # ---- detection head
    "vitk_detection_head_workspace_bytes": (C.c_int, [C.POINTER(VitkDetectionHeadConfig), C.c_int,
                                                      C.c_int, C.c_int, C.POINTER(C.c_size_t)]),
    "vitk_detection_head_forward": (C.c_int, [C.POINTER(VitkDetectionHeadConfig),
                                              C.POINTER(VitkDetectionHeadWeights), C.c_void_p,
                                              C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                              C.c_void_p, C.c_size_t, C.c_void_p]),
    "vitk_detection_head_train_bytes": (C.c_int, [C.POINTER(VitkDetectionHeadConfig), C.c_int,
                                                  C.c_int, C.c_int, C.POINTER(C.c_size_t),
                                                  C.POINTER(C.c_size_t)]),
    "vitk_detection_head_forward_train": (C.c_int, [C.POINTER(VitkDetectionHeadConfig),
                                                    C.POINTER(VitkDetectionHeadWeights), C.c_void_p,
                                                    C.c_int, C.c_int, C.c_int, C.c_void_p,
                                                    C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p,
                                                    C.c_size_t, C.c_void_p]),
    "vitk_detection_head_backward": (C.c_int, [C.POINTER(VitkDetectionHeadConfig),
                                               C.POINTER(VitkDetectionHeadWeights),
                                               C.POINTER(VitkDetectionHeadWeightsT),
                                               C.POINTER(VitkDetectionHeadGrads), C.c_void_p,
                                               C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                               C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "vitk_peer_reduce_scan": (C.c_int, [C.POINTER(VitkPeerBuffers), C.c_longlong, C.c_longlong,
                                        C.c_void_p]),
    "vitk_peer_adamw_broadcast": (C.c_int, [C.POINTER(VitkPeerBuffers), C.c_void_p, C.c_void_p,
                                            C.c_longlong, C.c_longlong, C.c_double, C.c_double,
                                            C.c_double, C.c_double, C.c_double, C.c_int, C.c_float,
                                            C.c_void_p]),
    "vitk_weighted_cross_entropy": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int,
                                              C.c_void_p, C.c_void_p, C.c_void_p, C.c_float,
                                              C.c_void_p]),
}


class VitkBlockWeightsT(C.Structure):
    _fields_ = [("qkv_wt", C.c_void_p), ("proj_wt", C.c_void_p), ("fc1_wt", C.c_void_p),
                ("fc2_wt", C.c_void_p)]


class VitkWeightsT(C.Structure):
    _fields_ = [("blocks", C.POINTER(VitkBlockWeightsT))]


class VitkBlockGrads(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("ln1_w", "ln1_b", "qkv_w", "qkv_b", "proj_w", "proj_b",
                                          "ln2_w", "ln2_b", "fc1_w", "fc1_b", "fc2_w", "fc2_b")]


class VitkGrads(C.Structure):
    _fields_ = [("patch_w", C.c_void_p), ("patch_b", C.c_void_p), ("cls_token", C.c_void_p),
                ("dist_token", C.c_void_p), ("pos_embed", C.c_void_p),
                ("blocks", C.POINTER(VitkBlockGrads)), ("ln_f_w", C.c_void_p),
                ("ln_f_b", C.c_void_p), ("head_w", C.c_void_p), ("head_b", C.c_void_p)]

_lib = None


def exported_symbols() -> list[str]:
    return sorted(_SIGNATURES)


def lib() -> C.CDLL:
    """Loads libvitk.so (once). Raises VitkError when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise VitkError(
            f"{LIB_PATH} not found - build it with `python {PKG_DIR.name}/build.py` "
            "(there is no CPU or PyTorch fallback)")
    if os.environ.get("VITK_LIB"):
        import sys
        print(f"vitk: loading the library named by VITK_LIB: {LIB_PATH}", file=sys.stderr)
    l = C.CDLL(str(LIB_PATH))
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(l, name)
        fn.restype = res
        fn.argtypes = args
    got = l.vitk_abi_version()
    if got != ABI_VERSION:
        raise VitkError(f"libvitk ABI version {got}, binding expects {ABI_VERSION}")
    _lib = l
    return l


def check(rc: int) -> None:
    if rc != 0:
        msg = lib().vitk_last_error()
        raise VitkError(f"vitk error {rc}: {msg.decode() if msg else '?'}")


def set_gemm_cta_group(ctas: int) -> None:
    """0 = auto, 1 = single-CTA tiles, 2 = CTA-pair (cta_group::2) tiles."""
    check(lib().vitk_gemm_set_cta_group(ctas))


def set_gemm_direct_epilogue(on: bool) -> None:
    check(lib().vitk_gemm_set_direct_epilogue(1 if on else 0))


def set_layernorm_folding(on: bool) -> None:
    """vitk_forward: True (default) = LayerNorm folded into the GEMMs around it when the packed
    weights carry the folded matrices; False = separate LayerNorm launches (A/B, tests)."""
    check(lib().vitk_set_layernorm_folding(1 if on else 0))


def set_attention_impl(impl: int) -> None:
    """0 = auto, 1 = flash (mma.sync), 2 = tcgen05 single-key-block kernel."""
    check(lib().vitk_attention_set_impl(impl))


def launch_count() -> int:
    return int(lib().vitk_launch_count())


PROF_KINDS = ("gemm", "attention", "layernorm", "patchify", "other", "optimizer")


def profile_enable(on: bool) -> None:
    check(lib().vitk_profile_enable(1 if on else 0))


def profile_collect() -> dict:
    """{kind: {"ms": total device ms, "work": FLOPs or bytes, "launches": n}} since the last call."""
    n = len(PROF_KINDS)
    ms = (C.c_double * n)()
    work = (C.c_double * n)()
    cnt = (C.c_longlong * n)()
    check(lib().vitk_profile_collect(ms, work, cnt, n))
    return {k: {"ms": ms[i], "work": work[i], "launches": cnt[i]} for i, k in enumerate(PROF_KINDS)}
