// Host launchers of the training-step kernels (train_ops.cu).
#pragma once
#include <cuda_runtime.h>

#include "dropout.cuh"

namespace vitk {

// dx_io (+)= LN backward; optional bf16 copy; dgamma/dbeta accumulate (atomics).  dx_colsum
// (optional, [D]) += column sums of the bf16 copy: the bias gradient of the Linear layer whose
// output gradient dx is, produced here instead of by a separate pass over dx_bf16.
int layernorm_bwd(const void* dy, int dy_is_f32, long long dy_stride, const float* x,
                  long long x_stride, const float* mean, const float* rstd, const float* gamma,
                  float* dx_io, long long dx_stride, int add_resid, void* dx_bf16,
                  long long dxb_stride, float* dgamma, float* dbeta, int rows, int D,
                  cudaStream_t stream, float* dx_colsum = nullptr,
                  const DropParams* drop = nullptr);  // mask of the branch dx_bf16 enters (dropout.cuh)

// out[n] += sum_m y[m, n]   (y bf16)
int colsum_bf16(const void* y, long long ld, int M, int N, float* out, cudaStream_t stream);

// CLS-row LayerNorm + head + mean cross-entropy, forward and backward. `scale` = 1 / global batch.
// dx (fp32 [B*N, D]) must be zero-filled by the caller; only the CLS rows are written.
int cls_loss_bwd(const float* x, long long row_stride, const float* gamma, const float* beta,
                 const float* head_w, const float* head_b, const long long* labels, float scale,
                 float eps, int B, int D, int C, float* logits_out, float* loss_out, float* feat_ws,
                 float* dlogits_ws, float* dx, void* dx_bf16, float* dgamma, float* dbeta,
                 float* dhead_w, float* dhead_b, cudaStream_t stream);

// F.cross_entropy(logits, targets, weight) - the weighted mean of SetCriterion.loss_labels
// (train.py:1220-1239) - and grad_scale * its gradient.  sums_ws: 2 floats of scratch.
int weighted_cross_entropy(const float* logits, const long long* targets, const float* weight,
                           int rows, int C, float* loss_out, float* sums_ws, float* dlogits,
                           float grad_scale, cudaStream_t stream);

// dpos[t,:] += sum_b dx[b,t,:]; dxp = bf16 copy of the patch rows of dx.
int token_grads(const float* dx, int B, int Ntok, int D, int prefix, float* dpos, float* dcls,
                float* ddist, void* dxp_bf16, cudaStream_t stream);

// nn.Dropout as stand-alone passes (dropout.cuh): x <- dropout(x) in place (the embedding dropout and
// its backward), out_bf16 = bf16(dropout(x)) (the gradient entering a branch whose output was
// dropped), and the keep mask itself (0/1 bytes) for the oracle tests.  n must be even.
int dropout_f32_inplace(float* x, long long n, const DropParams& d, cudaStream_t stream);
int dropout_cast_bf16(const float* x, void* out_bf16, long long n, const DropParams& d,
                      cudaStream_t stream);
int dropout_keep_mask(unsigned char* out, long long n, const DropParams& d, cudaStream_t stream);

constexpr int kMaxTransposeJobs = 64;
struct TransposeBatch {
  const void* src[kMaxTransposeJobs];
  void* dst[kMaxTransposeJobs];
  int rows[kMaxTransposeJobs];
  int cols[kMaxTransposeJobs];
  int tiles[kMaxTransposeJobs];
  int n;
};
int transpose_batched(const TransposeBatch& tb, cudaStream_t stream);

int adamw_flat(float* p, const float* g, float* m, float* v, void* shadow_bf16, long long n,
               double lr, double beta1, double beta2, double eps, double weight_decay, int step,
               float grad_scale, cudaStream_t stream, const int* guard = nullptr);
// Skip-on-non-finite guard of the optimizer step (train.py:1456: scaler.step): guard = device
// int[2] {flag, steps skipped}.  scan: flag |= any(!isfinite(g[0..n))) (reset clears it first);
// finish: folds the flag into the skipped count once the step's AdamW launches are queued.
int grad_guard_scan(const float* g, long long n, int* guard, int reset, cudaStream_t stream);
int grad_guard_finish(int* guard, cudaStream_t stream);

}  // namespace vitk
