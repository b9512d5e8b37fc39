// The attention core as the encoder, training and detection-head drivers see it: softmax(q k^T /
// sqrt(hd)) v per (image, head), forward and backward.  attention.cu chooses the kernel for each
// call; the per-kernel launchers behind it (attention_kernels.cuh) are private to the attention
// sources.
#pragma once
#include <cuda_runtime.h>

#include "dropout.cuh"

namespace vitk {

// Separate query and key / value sources: query row r of image b at q + b*q_img + r*ldq + h*hd,
// keys / values at k|v + b*kv_img + r*ldkv + h*hd (bf16, strides in elements).
struct AttnXSrc {
  const void* q; long long q_img; int ldq;
  const void* k; const void* v; long long kv_img; int ldkv;
};

// qkv bf16 [B*N, 3*D] packed as the reference packs it (column = which*D + h*hd + d); ctx bf16
// [B*N, D]; optional lse fp32 [B, H, N].  `drop` (training only): dropout on the attention
// probabilities (train.py:545).
int attention_fwd(const void* qkv, void* ctx, float* lse, int B, int N, int H, int hd,
                  cudaStream_t stream, const DropParams* drop = nullptr);

// dqkv = backward of attention_fwd given d_ctx, using the saved log-sum-exp.
// dbias (optional, [3 H hd]) += column sums of dqkv: the bias gradient of the qkv Linear.
int attention_bwd(const void* qkv, const void* ctx, const void* dctx, const float* lse, void* dqkv,
                  int B, int N, int H, int hd, cudaStream_t stream,
                  const DropParams* drop = nullptr, float* dbias = nullptr);

// Separate-source forward: output row r of image b at ctx + b*ctx_img + r*ldc + h*hd.  Without
// `lse` this is inference (`drop` is ignored); with it, the training forward.
int attention_src_fwd(const AttnXSrc& s, void* ctx, long long ctx_img, int ldc, float* lse, int B,
                      int Nq, int Nk, int H, int hd, cudaStream_t stream,
                      const DropParams* drop = nullptr);

// Separate-source backward: dq rows at dq + b*dq_img + r*lddq + h*hd, dk / dv rows at
// dk|dv + b*dkv_img + r*lddkv + h*hd (overwritten).
int attention_src_bwd(const AttnXSrc& s, const void* ctx, const void* dctx, long long ctx_img,
                      int ldc, const float* lse, void* dq, long long dq_img, int lddq, void* dk,
                      void* dv, long long dkv_img, int lddkv, int B, int Nq, int Nk, int H, int hd,
                      cudaStream_t stream, const DropParams* drop = nullptr);

// Whether the separate-source entry points take (Nq, Nk) at any head_dim hd, not only 32 / 64 /
// 96 / 128, in every mode (inference, log-sum-exp, dropout, backward): 16 <= hd <= 128, at most
// 128 queries and at most 256 keys.  A shape-only check, usable before anything is launched.
bool attention_src_supported(int Nq, int Nk, int hd);

// Whether attention_bwd covers N tokens of head_dim hd.
bool attention_trainable(int N, int hd);

// vitk_attention_set_impl (include/vitk.h).
void attention_force_impl(int impl);

}  // namespace vitk
