// HBM-bound row kernels (rowops.cu): host launchers.
#pragma once
#include <cuda_runtime.h>

namespace vitk {

// y[r,:] = LN(x[r,:]) * gamma + beta ; x fp32 rows at `in_stride` elements, y bf16 or fp32 rows at
// `out_stride`; optional per-row mean / rstd outputs (saved for backward).
int layernorm_fwd(const float* x, long long in_stride, const float* gamma, const float* beta,
                  void* y, int y_is_f32, long long out_stride, float* mean_out, float* rstd_out,
                  int rows, int D, float eps, cudaStream_t stream, float* x_copy = nullptr);

// LayerNorm folded into the neighbouring GEMMs (gemm_sm100.cuh, GemmEpilogue::ln_part):
// row_stats: y = bf16(x) and part[r] = (sum, sum of squares) of row r - the entry of the chain;
// ln_fold: w_out = bf16(W * gamma - row mean) (zero-sum rows), colsum[n] = what rounding leaves of
// the row sum (optional), bias_out = b + W beta.
int row_stats(const float* x, long long in_stride, void* y_bf16, long long out_stride, float2* part,
              int rows, int D, cudaStream_t stream);
int ln_fold(const float* W, const float* gamma, const float* beta, const float* b, void* w_out_bf16,
            float* colsum, float* bias_out, int N, int K, cudaStream_t stream);

// f32 NCHW images -> bf16 patch rows [B*P, C*p*p] in conv-weight column order.
int patchify(const float* img, void* out_bf16, int B, int C, int S, int p, cudaStream_t stream);

// u8 HWC images [B, S, S, 3] -> (u / 255 - mean) / std -> bf16 patch rows (the input edge of
// evaluation.py:362-364 fused into the gather); mean / stddev: 3 host floats.
int patchify_u8(const unsigned char* img_hwc, void* out_bf16, int B, int S, int p, const float* mean,
                const float* stddev, cudaStream_t stream);

// Rows of the learned prefix tokens (+ their position embeddings) of the residual stream.
int prefix_tokens(float* x, const float* cls, const float* dist, const float* pos, int B, int Ntok,
                  int D, int n_prefix, cudaStream_t stream);

// Final LayerNorm on row 0 of every image + Linear(D, n_classes).
int cls_head(const float* x, long long row_stride, const float* gamma, const float* beta,
             const float* head_w, const float* head_b, float* feat_out, float* logits, int B, int D,
             int n_classes, float eps, cudaStream_t stream);

// softmax over the last dim, then max / argmax over the classes (optionally without the last,
// "background", class) - evaluation.py:403-404; scores f32 [rows], labels i64 [rows], probs
// f32 [rows, C], each optional.
int postprocess_scores(const float* logits, int rows, int C, int exclude_last, float* scores,
                       long long* labels, float* probs, cudaStream_t stream);

// out[r, :] = x[r, :] W^T + b (fp32, W [n_out, D]), optionally divided by max(||.||_2, 1e-12):
// `triplet_projection` + F.normalize on the CLS rows (train.py:833-838).
int linear_rows(const float* x, long long row_stride, const float* w, const float* b, float* out,
                int rows, int D, int n_out, int l2_normalize, cudaStream_t stream);

// Backward of linear_rows without the normalisation: dx [rows, D], dw [n_out, D], db [n_out]
// (each optional, overwritten).
int linear_rows_bwd(const float* x, long long row_stride, const float* w, const float* dy,
                    float* dx, float* dw, float* db, int rows, int D, int n_out,
                    cudaStream_t stream);

// Batched post_process_predictions (evaluation.py:393-426): scores / labels as above without the
// background class, `score > threshold`, kept queries compacted to the front of each image's row
// of boxes_out [B,Q,4] / labels_out [B,Q] / scores_out [B,Q]; counts [B].
int postprocess_detections(const float* logits, const float* boxes, int batch, int Q, int C,
                           float threshold, int* counts, float* boxes_out, long long* labels_out,
                           float* scores_out, cudaStream_t stream);

int cast_f32_to_bf16(const float* in, void* out, long long n, cudaStream_t stream);

}  // namespace vitk
