/* vitk — C ABI of the B200-native ViT/DeiT encoder hot path.
 *
 * The reference (akavkl/Automated-Recycling-Sorter-with-Vision-Transformers) has no FFI of its
 * own: the only seam on this path is the nn.Module protocol,
 *     features = self.backbone(images)            evaluation.py:231, train.py:831
 *     losses.backward(); optimizer.step()         train.py:1455-1460
 * with `backbone = VisionTransformer(...)` (evaluation.py:120-157) or
 * `DataEfficientImageTransformer(...)` (train.py:637-688).  This header is what a Python (ctypes)
 * or C++ host binds to replace that call; INTEGRATION.md shows the reference-side stub.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the comment says "host"
 *   - the caller owns all memory (inputs, outputs, workspace, saved activations); the library
 *     never allocates on the hot path and keeps no references after a call returns
 *   - all work is enqueued on the caller's stream; nothing synchronises
 *   - every function returns 0 on success, otherwise a VITK_ERR_* code whose text is available
 *     from vitk_last_error() (thread-local); no C++ exception crosses this boundary
 *   - there is no CPU fallback: without an sm_100 device every compute entry point fails
 */
#ifndef VITK_H_
#define VITK_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VITK_ABI_VERSION 8

#define VITK_OK 0
#define VITK_ERR_INVALID 1
#define VITK_ERR_CUDA 2
#define VITK_ERR_WORKSPACE 3
#define VITK_ERR_NO_DEVICE 4

typedef void* vitk_stream_t; /* cudaStream_t */

/* Constructor arguments of VisionTransformer / DataEfficientImageTransformer
 * (evaluation.py:121-122, train.py:638-639) plus what the wrapper adds. */
typedef struct VitkConfig {
  int image_size;      /* S */
  int patch_size;      /* p (16) */
  int in_channels;     /* 3 */
  int embed_dim;       /* D */
  int num_layers;      /* L */
  int num_heads;       /* H */
  int mlp_dim;         /* M */
  int n_prefix_tokens; /* 1 = ViT (CLS), 2 = DeiT (CLS + DIST) */
  int n_classes;       /* classifier head on the CLS row; 0 = no head */
  int precision;       /* 0 = bf16 operands / fp32 accumulate; 1 = fp32-parity (split-bf16) */
  float ln_eps;        /* nn.LayerNorm default 1e-5 */
  float dropout_p;     /* applied only when training != 0 */
  uint64_t seed;
} VitkConfig;

/* One pre-LN encoder block (train.py:576-593); names follow the state_dict keys
 * transformer_blocks.{i}.{layer_norm1,attention.qkv,attention.projection,layer_norm2,
 * mlp.linear1,mlp.linear2}.{weight,bias}.  Matrix weights are bf16 row-major [out, in]
 * (nn.Linear layout); everything else fp32. */
typedef struct VitkBlockWeights {
  const float* ln1_w;
  const float* ln1_b;
  const void* qkv_w; /* bf16 [3D, D] */
  const float* qkv_b;
  const void* proj_w; /* bf16 [D, D] */
  const float* proj_b;
  const float* ln2_w;
  const float* ln2_b;
  const void* fc1_w; /* bf16 [M, D] */
  const float* fc1_b;
  const void* fc2_w; /* bf16 [D, M] */
  const float* fc2_b;
  /* Optional (inference, bf16 mode): layer_norm1 folded into qkv and layer_norm2 into linear1 by
   * vitk_fold_layernorm - *_w_ln bf16 [out, D], *_b_ln f32 [out].
   * When all four are set for every block, vitk_forward runs no LayerNorm pass between the
   * blocks: the projection / linear2 GEMMs leave the row statistics and a bf16 copy of the
   * residual stream, the qkv / linear1 GEMMs normalise in their epilogue.  NULL: separate
   * LayerNorm launches (the training entry points never read these). */
  const void* qkv_w_ln;
  const float* qkv_b_ln;
  const void* fc1_w_ln;
  const float* fc1_b_ln;
} VitkBlockWeights;

typedef struct VitkWeights {
  const void* patch_w;  /* bf16 [D, C*p*p] == patch_embedding.projection.weight.reshape(D,-1) */
  const float* patch_b; /* [D] */
  const float* cls_token;  /* [D] */
  const float* dist_token; /* [D] or NULL (ViT) */
  const float* pos_embed;  /* [N, D] */
  const VitkBlockWeights* blocks; /* HOST array of num_layers entries */
  const float* ln_f_w; /* layer_norm.weight */
  const float* ln_f_b;
  const float* head_w; /* fp32 [n_classes, D] or NULL */
  const float* head_b;
} VitkWeights;

int vitk_abi_version(void);
const char* vitk_last_error(void);
/* Kernels launched by this library since process start (bench.py's gpu_launches). */
long long vitk_launch_count(void);

/* Per-kernel-class device timing for the roofline report: while enabled, every launcher brackets
 * its kernel with CUDA events on the launching stream. Kinds: 0 GEMM (work = FLOPs), 1 attention
 * (FLOPs), 2 LayerNorm (bytes), 3 patchify (bytes), 4 other, 5 optimizer (bytes). */
#define VITK_PROF_NKINDS 6
int vitk_profile_enable(int on);
int vitk_profile_collect(double* ms_by_kind, double* work_by_kind, long long* launches_by_kind,
                         int nkinds);

/* GEMM tile mode: 0 = automatic (CTA pairs / tcgen05 cta_group::2 whenever M > 128), 1 = single
 * CTA 128-row tiles, 2 = CTA-pair 256-row tiles.  Process-wide; meant for tests and A/B timing. */
int vitk_gemm_set_cta_group(int ctas);
/* 1 = write GEMM outputs with per-thread global stores instead of the smem-staged TMA
 * store / reduce-add epilogue (tests, A/B timing). */
int vitk_gemm_set_direct_epilogue(int on);
/* Debug aid: in a library built with -DVITK_GEMM_TRACE the MMA-issuing warp of every CTA pair counts
 * the SM clocks it waits for operands / for a free accumulator stage; copies
 * [pair][{total, wait operands, wait accumulator, tiles}] of the last GEMM launch to HOST memory
 * (n entries).  Returns the entries written; 0 in a normal build. */
int vitk_debug_gemm_trace(long long* out_host, int n);
/* vitk_forward with VitkBlockWeights::*_ln set: 1 (default) = LayerNorm folded into the GEMMs
 * around it, 0 = separate LayerNorm launches (A/B timing, tests).  Initial value from the
 * environment variable VITK_LN_FOLD. */
int vitk_set_layernorm_folding(int on);

/* Device side of post_process_predictions (evaluation.py:393-407, lines 403-404): softmax over the
 * class logits f32 [rows, n_classes], then the maximum probability and its class per row,
 * optionally ignoring the last ("background") class as the detector does.  scores_out f32 [rows],
 * labels_out i64 [rows], probs_out f32 [rows, n_classes]; each may be null.  Replaces the
 * per-image Python loop and its host synchronisations. */
int vitk_postprocess_scores(const float* logits, int rows, int n_classes, int exclude_last,
                            float* scores_out, long long* labels_out, float* probs_out,
                            vitk_stream_t stream);

/* post_process_predictions (evaluation.py:393-426) for a whole batch in one launch and without a
 * host synchronisation per image: class_logits f32 [batch, Q, num_outputs] (last output =
 * background), bbox_coords f32 [batch, Q, 4].  Per query: softmax, best non-background class and
 * its probability; a query is kept when that probability > confidence_threshold.  The kept queries
 * of image b are written, in query order (what boolean-mask indexing yields), to the front of row b
 * of boxes_out [batch, Q, 4], labels_out i64 [batch, Q], scores_out [batch, Q]; counts_out i32
 * [batch] holds how many.  Q <= 1024. */
int vitk_postprocess_detections(const float* class_logits, const float* bbox_coords, int batch,
                                int num_queries, int num_outputs, float confidence_threshold,
                                int* counts_out, float* boxes_out, long long* labels_out,
                                float* scores_out, vitk_stream_t stream);

/* The CLS-row consumers of the reference (SURVEY row a9; DeiTObjectDetector.forward,
 * train.py:833-838): out[r, :] = x[r, :] W^T + b in fp32 for a few rows (x rows `row_stride`
 * elements apart, e.g. the CLS row of every image of backbone(images): stride N*D), optionally
 * followed by F.normalize(p=2, dim=1).  weight fp32 [out_features, in_features]; bias may be null. */
int vitk_linear_rows(const float* x, long long row_stride, const float* weight, const float* bias,
                     float* out, int rows, int in_features, int out_features, int l2_normalize,
                     vitk_stream_t stream);

/* Backward of vitk_linear_rows (l2_normalize = 0): given dy f32 [rows, out_features] writes
 * dx f32 [rows, in_features] = dy W, dweight f32 [out, in] = dy^T x and dbias f32 [out] = column
 * sums of dy (each optional).  The 6-class head on the CLS rows under the autograd bridge
 * (loss.backward() of train.py:1455 with a user-supplied loss). */
int vitk_linear_rows_backward(const float* x, long long row_stride, const float* weight,
                              const float* dy, float* dx, float* dweight, float* dbias, int rows,
                              int in_features, int out_features, vitk_stream_t stream);

/* Persistent kernels (GEMM, attention) launch one CTA per SM; keep `n` SMs out of their grids, e.g.
 * for the NCCL kernels of a gradient all-reduce that overlaps the backward pass. 0 restores all. */
int vitk_reserve_sms(int n);

/* Attention kernel choice, for tests and A/B timing (the table in csrc/attention.cu):
 *   0 = automatic: by shape and device.
 *   1 = no tcgen05 kernel where another one covers the call: the head_dim-64 mma.sync flash
 *       kernels, the mma.sync generic-source inference kernel, and the CUDA-core training kernels
 *       of the separate-source (detection head) and head_dim != 64 paths.  Dropout in the
 *       head_dim-64 encoder still uses the tcgen05 kernels.
 *   2-4 change the head_dim-64 inference / log-sum-exp forward only (elsewhere they act as 0):
 *   2 = tcgen05 forwards chosen by N as 0 does (item-pipelined up to 208 tokens, single key block
 *       up to 256, key blocks up to 640), also off sm_100;
 *   3 = the single-key-block kernel up to 256 tokens, key blocks above (never the pipelined one);
 *   4 = the key-block kernel for every N (up to 640). */
int vitk_attention_set_impl(int impl);

/* Scratch bytes vitk_forward needs for `batch` images. */
int vitk_workspace_bytes(const VitkConfig* cfg, int batch, size_t* out_bytes);

/* The model call.  images: f32 NCHW [batch, C, S, S] (the tensor evaluation.py:499-502 feeds).
 * tokens_out: f32 [batch, N, D] = backbone(images) (all tokens after the final LayerNorm), or NULL.
 * logits_out: f32 [batch, n_classes] = head(LN(x)[:,0]), or NULL.  At least one must be given. */
int vitk_forward(const VitkConfig* cfg, const VitkWeights* w, const float* images, int batch,
                 float* tokens_out, float* logits_out, void* workspace, size_t workspace_bytes,
                 vitk_stream_t stream);

/* The classifier call with the last block evaluated for the CLS rows only: logits_out is what
 * vitk_forward(tokens_out = NULL) returns, but since head(LN(x)[:, 0]) reads a single row per
 * image, the last block's attention is run for that one query (against the keys / values of all
 * tokens) and its projection, LayerNorm and MLP on `batch` rows instead of batch * N - 71 % of the
 * last block's contraction work feeds nothing the classifier returns.  bf16 mode; head_dim 32,
 * 64, 96 or 128, or any other head_dim from 16 to 128 up to 256 tokens (train.py's Config: 16). */
int vitk_forward_cls(const VitkConfig* cfg, const VitkWeights* w, const float* images, int batch,
                     float* logits_out, void* workspace, size_t workspace_bytes,
                     vitk_stream_t stream);

/* vitk_forward for 8-bit images straight from the decoder (HWC, u8 [batch, S, S, 3], 8-byte
 * aligned): A.Normalize(mean, std) + ToTensorV2 of the reference's data pipeline
 * (evaluation.py:362-364, 369-372; train.py:442-443) are fused into the patch gather, evaluated
 * exactly as the reference does in fp32, (u / 255 - mean) / std, so the result is bit-identical
 * to vitk_forward on the normalised float image while the host sends a quarter of the bytes.
 * mean / stddev: 3 HOST floats each.  bf16 mode only. */
int vitk_forward_u8(const VitkConfig* cfg, const VitkWeights* w, const unsigned char* images_hwc,
                    const float* mean, const float* stddev, int batch, float* tokens_out,
                    float* logits_out, void* workspace, size_t workspace_bytes,
                    vitk_stream_t stream);

/* ---- per-operator entry points (unit-tested individually; same kernels vitk_forward uses) ---- */

/* epilogue ids for vitk_gemm */
#define VITK_EPI_BF16 0      /* out bf16 = A B^T + bias */
/* The GELUs approximate x * Phi(x), Phi the normal CDF; the bounds are per element against the
 * exact erf form, before the bf16 rounding of the output (tests/test_gemm_epilogues_gpu.py). */
#define VITK_EPI_BF16 0      /* out bf16 = A B^T + bias */
/* out bf16 = x Phi(x), x = A B^T + bias, with Phi an erf-fitted logistic of an odd polynomial:
 * |error| <= 9e-5 [, out2 bf16 = x] */
#define VITK_EPI_GELU_BF16 1
#define VITK_EPI_RESID_F32 2 /* out f32  = A B^T + bias + resid f32 */
#define VITK_EPI_F32 3       /* out f32  = alpha * A B^T + bias + beta * out */
/* out bf16 = g * gelu'(x), g = A B^T + bias, x = aux bf16: exact erf derivative (|error| <= 1e-5 |g|)
 * where the epilogue writes directly, tanh form (|error| <= |g| (1.3e-4 + 2^-11 (0.5 + 2|x|)))
 * where it is TMA-staged */
#define VITK_EPI_DGELU_BF16 4
#define VITK_EPI_RELU_BF16 7  /* out bf16 = max(A B^T + bias, 0) (decoder feed-forward) */
/* As VITK_EPI_GELU_BF16 with Phi = 0.5 + 0.5 tanh.approx(odd polynomial): |error| <= 3.3e-5 +
 * 2.5e-4 |x|.  The fc1 epilogue of the encoder forward and training. */
#define VITK_EPI_GELU_TANH_BF16 6

/* C[M,N] = A[M,K] * B[N,K]^T (bf16 operands, fp32 accumulate on tcgen05) + fused epilogue.
 * Replaces nn.Linear / F.linear at train.py:527,529,561,564 and the Conv2d at train.py:505. */
int vitk_gemm(const void* A, int lda, const void* B, int ldb, int M, int N, int K, int epilogue,
              const float* bias, const float* resid, int ldr, const void* aux, void* out, void* out2,
              int ldo, float alpha, float beta, vitk_stream_t stream);

/* Residual update and the LayerNorm that follows it (train.py:586-591: x = x + f(..), then
 * layer_norm(x) feeds the next Linear): x[M,N] f32 += A[M,K] W[N,K]^T + bias (TMA reduce-add
 * epilogue) and ln_out bf16 [M,N] = LN(x) * gamma + beta (optionally mean / rstd f32 [M]), N <= 1024.
 * Two launches: vitk_gemm(VITK_EPI_RESID_F32) followed by vitk_layernorm, with the same bits. */
int vitk_gemm_resid_layernorm(const void* A, int lda, const void* W, int ldb, int M, int N, int K,
                              const float* bias, float* x_inout, const float* gamma,
                              const float* beta, float eps, void* ln_out, float* mean_out,
                              float* rstd_out, vitk_stream_t stream);

/* ---- LayerNorm folded into the two GEMMs around it (train.py:584-591: x = x + f(..);
 * Linear(layer_norm(x))).  Instead of a LayerNorm pass over the fp32 residual stream between two
 * GEMMs, the residual GEMM's epilogue (thread == row) leaves per-row partial sums and a bf16 copy
 * of x, and the next GEMM contracts that copy against the ROW-CENTRED matrix
 * V[n,k] = gamma_k W[n,k] - mean_k(gamma_k W[n,k]) and scales in its epilogue.  A zero-sum row
 * drops the mean of x inside the contraction (sum_k mu V[n,k] = 0), so
 *   Linear(LN(x))[m,n] = rstd_m * sum_k x[m,k] V[n,k] + b[n] + sum_k beta_k W[n,k]. */

/* Weights of the folded form.  weight f32 [out, in], gamma / beta f32 [in], bias f32 [out] or NULL
 * -> w_ln bf16 [out, in] = V (above), b_ln f32 [out] = bias + weight beta; rowsum_or_null f32
 * [out]: what bf16 rounding leaves of the row sums of w_ln (the mean of x leaks into the output
 * as mu * rstd * rowsum[n]; ~1e-3 for ViT weights, below the bf16 output resolution). */
int vitk_fold_layernorm(const float* weight, const float* gamma, const float* beta,
                        const float* bias, void* w_ln_bf16, float* b_ln, float* rowsum_or_null,
                        int out_features, int in_features, vitk_stream_t stream);

/* Partial sums per row that vitk_gemm_resid_stats writes for an N-column output. */
int vitk_stats_parts(int n_features);

/* Entry of the chain: x_bf16[rows, D] = bf16(x) and stats[r] = (sum, sum of squares) of row r
 * (one partial).  stats: f32 pairs [rows]. */
int vitk_row_stats(const float* x, long long in_stride, void* x_bf16, long long out_stride,
                   float* stats, int rows, int D, vitk_stream_t stream);

/* x[M,N] f32 += A[M,K] W[N,K]^T + bias in place (the x tile is TMA-loaded into the epilogue's
 * staging slab, updated there and TMA-stored), x_bf16[M,N] = bf16(x), stats f32 pairs
 * [vitk_stats_parts(N)][M]: (sum, sum of squares) of the updated row over each column group. */
int vitk_gemm_resid_stats(const void* A, int lda, const void* W, int ldb, int M, int N, int K,
                          const float* bias, float* x_inout, void* x_bf16, float* stats,
                          vitk_stream_t stream);

/* out bf16 [M,N] = epilogue(Linear(LayerNorm(x))) from x_bf16 [M,K], the folded weights and the
 * row statistics (n_parts partials of M pairs; K features per row).  epilogue: VITK_EPI_BF16,
 * VITK_EPI_GELU_BF16, VITK_EPI_GELU_TANH_BF16 or VITK_EPI_RELU_BF16. */
int vitk_gemm_layernorm_folded(const void* x_bf16, int lda, const void* w_ln, int ldb, int M, int N,
                               int K, int epilogue, const float* b_ln, const float* stats,
                               int n_parts, float eps, void* out, int ldo, vitk_stream_t stream);

/* Weight-gradient contraction C[M,N] (+)= A^T B with A stored [K, lda] (M contiguous) and B stored
 * [K, ldb] (N contiguous): dW[out,in] = sum over tokens of dY[token,out] * X[token,in] - the
 * backward of nn.Linear w.r.t. its weight (autograd of train.py:1455).  fp32 output,
 * out = alpha * A^T B + beta * out with beta in {0, 1}; split_k > 1 spreads the token range over
 * several CTAs that accumulate with TMA reduce-add (then beta must be 1 and out pre-initialised). */
int vitk_gemm_wgrad(const void* A, int lda, const void* B, int ldb, int M, int N, int K, float* out,
                    int ldo, float alpha, float beta, int split_k, vitk_stream_t stream);

/* nn.LayerNorm(D) over `rows` rows (train.py:581-582). y is bf16 (y_is_f32 = 0) or f32.  D % 4 == 0,
 * D <= 1024; strides multiples of 4; x, gamma, beta 16-byte aligned, y 16-byte (f32) or 8-byte
 * (bf16) aligned. */
int vitk_layernorm(const float* x, long long in_stride, const float* gamma, const float* beta,
                   void* y, int y_is_f32, long long out_stride, float* mean_out, float* rstd_out,
                   int rows, int D, float eps, vitk_stream_t stream);

/* MultiHeadSelfAttention core (train.py:537-549) on the packed qkv activation. */
int vitk_attention(const void* qkv_bf16, void* ctx_bf16, float* lse_or_null, int batch, int n_tokens,
                   int num_heads, int head_dim, vitk_stream_t stream);

/* Attention with separate query and key / value sources (the detection head's decoder attentions,
 * unit tests): per (image, head) ctx = softmax(q k^T / sqrt(head_dim)) v, bf16.  Query row r of
 * image b at q + b*q_img + r*ldq + h*head_dim, key / value rows at k|v + b*kv_img + r*ldkv +
 * h*head_dim, output rows at ctx + b*ctx_img + r*ldc + h*head_dim (strides in elements; q, k, v
 * 16-byte aligned with pitches that are multiples of 8).  head_dim 32 / 64 / 96 / 128, or any
 * other head_dim from 16 to 128 with n_q <= 128 and n_k <= 256.  lse_or_null (fp32
 * [batch, num_heads, n_q]) selects the training forward; only then is dropout_p applied to the
 * probabilities, with the masks of vitk_dropout_keep_mask(dropout_p, seed, site, layer) at index
 * ((b*num_heads + h)*n_q + i)*Nk + j, Nk = n_k rounded up to 16. */
int vitk_attention_src(const void* q, long long q_img, int ldq, const void* k, const void* v,
                       long long kv_img, int ldkv, void* ctx, long long ctx_img, int ldc,
                       float* lse_or_null, int batch, int n_q, int n_k, int num_heads,
                       int head_dim, float dropout_p, unsigned int seed, int site, int layer,
                       vitk_stream_t stream);

/* Conv2d(k=p, s=p) input gather: f32 NCHW -> bf16 [B*P, C*p*p] (train.py:505-515). */
int vitk_patchify(const float* images, void* patches_bf16, int batch, int channels, int image_size,
                  int patch_size, vitk_stream_t stream);

int vitk_cast_f32_to_bf16(const float* in, void* out_bf16, long long n, vitk_stream_t stream);

/* fp32-parity mode (VitkConfig.precision = 1, logits within 1e-4 of the fp32 reference): fp32
 * operands are split into three bf16 terms and contracted by the same tcgen05 kernel with
 * K' = 6K.  The matrix members of VitkWeights / VitkBlockWeights must then point at split
 * weights made with this function (is_weight = 1): in f32 [rows, K] (row pitch ld_in elements)
 * -> out bf16 [rows, 6K].  Forward only. */
int vitk_split3(const float* in, long long ld_in, void* out_bf16, long long rows, int K,
                int is_weight, vitk_stream_t stream);

/* =========================== training step (train.py:1441-1460) ===========================
 * forward (saving activations) -> loss -> backward -> AdamW, replacing
 *     outputs = model(images) ; losses.backward() ; optimizer.step()
 * The loss of north_star's fine-tune is the mean cross-entropy of the 6-class CLS head; the
 * generic vitk_backward_tokens serves any loss computed by the caller on backbone(images).
 * Dropout: config.dropout_p > 0 applies nn.Dropout at the reference's five sites (see
 * vitk_dropout_keep_mask below); forward and backward of a step must be given the same seed. */

/* W^T copies ([in, out], bf16) of the four nn.Linear weights of a block: the input-gradient GEMMs
 * read the weight with its two dimensions swapped. Kept current by the caller after every
 * optimizer step (vitk_transpose_bf16_batched). */
typedef struct VitkBlockWeightsT {
  const void* qkv_wt;  /* [D, 3D] */
  const void* proj_wt; /* [D, D]  */
  const void* fc1_wt;  /* [D, M]  */
  const void* fc2_wt;  /* [M, D]  */
} VitkBlockWeightsT;

typedef struct VitkWeightsT {
  const VitkBlockWeightsT* blocks; /* HOST array of num_layers entries */
} VitkWeightsT;

/* fp32 gradient buffers, one per parameter, same shapes as the parameters (state_dict order).
 * Every backward entry point ACCUMULATES into them; the caller zeroes them once per step. */
typedef struct VitkBlockGrads {
  float* ln1_w;
  float* ln1_b;
  float* qkv_w;
  float* qkv_b;
  float* proj_w;
  float* proj_b;
  float* ln2_w;
  float* ln2_b;
  float* fc1_w;
  float* fc1_b;
  float* fc2_w;
  float* fc2_b;
} VitkBlockGrads;

typedef struct VitkGrads {
  float* patch_w;
  float* patch_b;
  float* cls_token;
  float* dist_token; /* NULL for ViT */
  float* pos_embed;
  const VitkBlockGrads* blocks; /* HOST array */
  float* ln_f_w;
  float* ln_f_b;
  float* head_w; /* NULL when there is no classifier head */
  float* head_b;
} VitkGrads;

/* Bytes of the saved-activation arena and of the scratch workspace for `batch` images. */
int vitk_train_workspace_bytes(const VitkConfig* cfg, int batch, size_t* saved_bytes,
                               size_t* workspace_bytes);

/* Dropout (cfg->dropout_p > 0, training entry points only; reference train.py:528-530,545,553,
 * 563-572,650,681).  Masks are a pure function of (cfg->seed, site, layer, element index) and are
 * regenerated by the backward kernels, so forward and backward of one step must be given the same
 * seed; change the seed every step.  Sites: 0 tokens+position embedding (index = flat [B*N, D]),
 * 1 attention probabilities (index = ((b*H + h)*N + i)*Nk + j with Nk = N rounded up to 16),
 * 2 projection output, 3 MLP hidden activation, 4 MLP output (index = row * width + column).
 * Detection head (VitkDetectionHeadConfig.dropout_p; layer = decoder layer): 8 self-attention
 * probabilities, 10 cross-attention probabilities (index = ((b*8 + h)*Q + i)*Nk + j, Nk = keys
 * rounded up to 16), 9 / 11 / 13 the self-attention / cross-attention / linear2 outputs before
 * their residual adds, 12 the ReLU output of linear1 (index = row * width + column).
 * vitk_dropout_keep_mask writes the 0/1 keep decisions of elements [0, n) of one site (n even) -
 * what the parity tests inject into the oracle.  p is quantised to 1/65536. */
int vitk_dropout_keep_mask(float p, unsigned int seed, int site, int layer, long long n,
                           unsigned char* out, vitk_stream_t stream);

/* Forward in training mode: same arithmetic as vitk_forward, every activation the backward needs
 * is written into `saved`; the residual stream stays in `workspace`. tokens_out (f32 [B,N,D],
 * optional) = backbone(images). */
int vitk_forward_train(const VitkConfig* cfg, const VitkWeights* w, const float* images, int batch,
                       float* tokens_out, void* saved, size_t saved_bytes, void* workspace,
                       size_t workspace_bytes, vitk_stream_t stream);

/* After vitk_forward_train: logits = head(LN(x)[:,0]); loss_out += loss_scale * sum_b CE(logits_b,
 * labels_b) (loss_scale = 1 / global batch gives F.cross_entropy's mean); then the full backward.
 * labels: int64 [batch]. logits_out f32 [batch, n_classes] and loss_out (f32 scalar, pre-zeroed)
 * are optional. */
int vitk_classifier_loss_backward(const VitkConfig* cfg, const VitkWeights* w,
                                  const VitkWeightsT* wt, const VitkGrads* g,
                                  const long long* labels, int batch, float loss_scale,
                                  float* logits_out, float* loss_out, void* saved, void* workspace,
                                  vitk_stream_t stream);

/* Same, for data-parallel training: bucket_events[k] (a cudaEvent_t each, n_events = num_layers + 2)
 * is recorded on `stream` as soon as gradient bucket k is final, so that the caller can start that
 * bucket's all-reduce on another stream while the rest of the backward runs (north_star: "gradient
 * allreduce over NCCL/NVLink overlapped with backward").  Bucket 0 = final LayerNorm + head,
 * bucket 1 + i = encoder block (num_layers - 1 - i), last bucket = tokens, position and patch
 * embedding.  bucket_events may be null (then identical to vitk_classifier_loss_backward). */
typedef void* vitk_event_t;
int vitk_classifier_loss_backward_ev(const VitkConfig* cfg, const VitkWeights* w,
                                     const VitkWeightsT* wt, const VitkGrads* g,
                                     const long long* labels, int batch, float loss_scale,
                                     float* logits_out, float* loss_out, void* saved,
                                     void* workspace, const vitk_event_t* bucket_events,
                                     int n_events, vitk_stream_t stream);

/* After vitk_forward_train with tokens_out: backward from d_tokens = dLoss/d backbone(images)
 * (f32 [B,N,D]) - what autograd hands to the backbone at train.py:1455. */
int vitk_backward_tokens(const VitkConfig* cfg, const VitkWeights* w, const VitkWeightsT* wt,
                         const VitkGrads* g, const float* d_tokens, int batch, void* saved,
                         void* workspace, vitk_stream_t stream);

/* torch.optim.AdamW (train.py:1598-1602: one group, decay on every parameter) over a flat fp32
 * arena of n parameters in ONE launch; grads are multiplied by grad_scale first; refreshes the
 * bf16 shadow arena (same element order) when shadow_bf16 != NULL. step is 1-based. */
int vitk_adamw_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq,
                    void* shadow_bf16, long long n, double lr, double beta1, double beta2,
                    double eps, double weight_decay, int step, float grad_scale,
                    vitk_stream_t stream);

/* Skip-on-non-finite guard of the optimizer step: the reference's `scaler.step(optimizer)`
 * (train.py:1456 with the GradScaler of train.py:1615) leaves the parameters alone when any
 * gradient is inf / nan.  guard: device int[2] {flag, steps skipped so far}, zero-initialised by
 * the caller once.  Per step: vitk_grad_guard_scan over the (reduced) gradients - reset = 1 on
 * the first call of the step clears the flag, several calls may cover the arena slice by slice;
 * vitk_adamw_step_guarded does nothing while the flag is set and evaluates Adam's bias
 * corrections for step - skipped (a skipped step does not advance the step counter);
 * vitk_grad_guard_finish, queued after the step's last AdamW launch, adds the flag to the count.
 * No host synchronisation anywhere. */
int vitk_grad_guard_scan(const float* grads, long long n, int* guard, int reset,
                         vitk_stream_t stream);
int vitk_adamw_step_guarded(float* params, const float* grads, float* exp_avg, float* exp_avg_sq,
                            void* shadow_bf16, long long n, double lr, double beta1, double beta2,
                            double eps, double weight_decay, int step, float grad_scale,
                            const int* guard, vitk_stream_t stream);
int vitk_grad_guard_finish(int* guard, vitk_stream_t stream);

/* dst_i [cols_i, rows_i] = src_i [rows_i, cols_i]^T for n bf16 matrices (host pointer arrays). */
int vitk_transpose_bf16_batched(int n, const void* const* src, void* const* dst, const int* rows,
                                const int* cols, vitk_stream_t stream);

/* Per-operator backward entry points (unit tests; the same kernels the step uses). */
/* LayerNorm backward over dense [rows, D] rows (D % 4 == 0, D <= 1024): dx_io = dLN (+ dx_io when
 * add_resid); dx_bf16 (optional) its bf16 copy; dgamma / dbeta (optional, together) accumulate.
 * dx_colsum (optional, needs dx_bf16) accumulates the column sums of the bf16 copy; outside the
 * fused kernel (dgamma given and D <= 768) it needs D % 8 == 0.  dropout_p > 0 (fused kernel and
 * dx_bf16 only) applies the keep mask of vitk_dropout_keep_mask(dropout_p, seed, site, layer) at
 * index row * D + column to the bf16 copy, which is then scaled by 1 / (1 - p); dx_io stays
 * unmasked.  dy may be dx_io (f32, add_resid = 0).  Every argument is checked before the first
 * launch, so a rejected call changes nothing. */
int vitk_layernorm_bwd(const void* dy, int dy_is_f32, const float* x, const float* mean,
                       const float* rstd, const float* gamma, float* dx_io, int add_resid,
                       void* dx_bf16, float* dgamma, float* dbeta, int rows, int D,
                       float* dx_colsum, float dropout_p, unsigned int seed, int site, int layer,
                       vitk_stream_t stream);
/* The classifier tail of vitk_classifier_loss_backward on its own: for each image b, with the
 * CLS row x + b*row_stride (D floats), feat = LayerNorm(x_b; gamma, beta, eps), logits = feat
 * head_w^T + head_b (head_w [n_classes, D]), loss_out += scale * CE(logits, labels[b]) and the
 * backward of that loss: dlogits_ws [batch, n_classes] and feat_ws [batch, D] (both required),
 * dx (required) and dx_bf16 (optional) at the CLS rows (same row_stride; nothing else is
 * written), dgamma /
 * dbeta (optional, together) and dhead_w / dhead_b (optional, together) accumulate.
 * logits_out [batch, n_classes] and loss_out are optional; n_classes <= 1024. */
int vitk_classifier_head_loss_backward(const float* x, long long row_stride, const float* gamma,
                                       const float* beta, const float* head_w, const float* head_b,
                                       const long long* labels, float scale, float eps, int batch,
                                       int D, int n_classes, float* logits_out, float* loss_out,
                                       float* feat_ws, float* dlogits_ws, float* dx,
                                       void* dx_bf16, float* dgamma, float* dbeta, float* dhead_w,
                                       float* dhead_b, vitk_stream_t stream);
int vitk_attention_bwd(const void* qkv_bf16, const void* ctx_bf16, const void* dctx_bf16,
                       const float* lse, void* dqkv_bf16, int batch, int n_tokens, int num_heads,
                       int head_dim, vitk_stream_t stream);
/* Backward of vitk_attention_src with its saved log-sum-exp and the same dropout arguments: dq
 * rows at dq + b*dq_img + r*lddq + h*head_dim, dk / dv rows at dk|dv + b*dkv_img + r*lddkv +
 * h*head_dim (exactly head_dim columns of each row are written). */
int vitk_attention_src_bwd(const void* q, long long q_img, int ldq, const void* k, const void* v,
                           long long kv_img, int ldkv, const void* ctx, const void* dctx,
                           long long ctx_img, int ldc, const float* lse, void* dq, long long dq_img,
                           int lddq, void* dk, void* dv, long long dkv_img, int lddkv, int batch,
                           int n_q, int n_k, int num_heads, int head_dim, float dropout_p,
                           unsigned int seed, int site, int layer, vitk_stream_t stream);
/* out[n] += sum_m y[m, n] over a bf16 [M, N] matrix of row pitch ld (N and ld multiples of 8, y
 * 16-byte aligned). */
int vitk_colsum_bf16(const void* y, long long ld, int M, int N, float* out, vitk_stream_t stream);

/* ============ detection head (ObjectDetectionHead, evaluation.py:160-200 == train.py:691-731) ====
 * The consumer of the backbone's tokens in both reference scripts:
 *     decoder_output = self.decoder(object_queries, encoder_features)     evaluation.py:189
 *     class_logits = self.class_head(decoder_output)                      evaluation.py:192
 *     bbox_coords  = sigmoid(self.bbox_head(decoder_output))              evaluation.py:193-194
 * with decoder = nn.TransformerDecoder(nn.TransformerDecoderLayer(d_model = D, nhead = 8,
 * dim_feedforward = 2048, dropout = 0.1, batch_first = True), num_layers = 6): post-LN layers,
 * ReLU, no final norm.  Eval-mode (inference) forward.  Matrix weights bf16 row-major [out, in],
 * everything else fp32; member names follow the state_dict keys
 * detection_head.decoder.layers.{i}.{self_attn.in_proj_weight, self_attn.out_proj, multihead_attn.*,
 * linear1, linear2, norm1, norm2, norm3}. */
typedef struct VitkDetectionHeadConfig {
  int embed_dim;   /* D (768) */
  int num_heads;   /* 8: head_dim = D / 8 of 32, 64, 96 or 128, or any other head_dim from 16 to
                    * 128 with num_queries <= 128 and at most 256 memory tokens (D = 400: 50) */
  int ffn_dim;     /* 2048 */
  int num_layers;  /* 6 */
  int num_queries; /* 100 */
  int num_outputs; /* num_classes + 1 (background) */
  float ln_eps;    /* 1e-5 */
  /* nn.TransformerDecoderLayer(dropout=0.1) (train.py:701-707), applied by the *_train / backward
   * entry points only: attention probabilities of both attentions, the three branch outputs before
   * their residual adds, the ReLU output of the feed-forward.  Masks are a hash of (seed, site,
   * layer, element): forward and backward must be given the same seed.  0 = off. */
  float dropout_p;
  uint64_t seed;
} VitkDetectionHeadConfig;

typedef struct VitkDecoderLayerWeights {
  const void* sa_in_w; /* bf16 [3D, D]  self_attn.in_proj_weight */
  const float* sa_in_b;
  const void* sa_out_w; /* bf16 [D, D]  self_attn.out_proj.weight */
  const float* sa_out_b;
  const void* ca_q_w; /* bf16 [D, D]    multihead_attn.in_proj_weight[:D] */
  const float* ca_q_b; /*               multihead_attn.in_proj_bias[:D] */
  const void* ca_out_w; /* bf16 [D, D]  multihead_attn.out_proj.weight */
  const float* ca_out_b;
  const void* ff1_w; /* bf16 [F, D]     linear1.weight */
  const float* ff1_b;
  const void* ff2_w; /* bf16 [D, F]     linear2.weight */
  const float* ff2_b;
  const float* norm1_w;
  const float* norm1_b;
  const float* norm2_w;
  const float* norm2_b;
  const float* norm3_w;
  const float* norm3_b;
} VitkDecoderLayerWeights;

typedef struct VitkDetectionHeadWeights {
  const float* object_queries;           /* f32 [Q, D] */
  const VitkDecoderLayerWeights* layers; /* HOST array of num_layers entries */
  /* K and V projections of the memory for every layer, concatenated so that ONE GEMM projects the
   * encoder tokens for all layers: rows [l*2D, (l+1)*2D) = layer l's
   * multihead_attn.in_proj_weight[D:3D] (K rows, then V rows); bias likewise. */
  const void* ca_kv_w;  /* bf16 [L*2D, D] */
  const float* ca_kv_b; /* f32 [L*2D] */
  const float* class_w; /* f32 [num_outputs, D]  class_head.weight */
  const float* class_b;
  const float* bbox_w; /* f32 [4, D]  bbox_head.weight */
  const float* bbox_b;
} VitkDetectionHeadWeights;

int vitk_detection_head_workspace_bytes(const VitkDetectionHeadConfig* cfg, int batch, int n_tokens,
                                        int skip_tokens, size_t* out_bytes);

/* tokens: f32 [batch, n_tokens, D] = backbone(images) (vitk_forward's tokens_out); the first
 * skip_tokens rows of every image (the CLS token, evaluation.py:235 `features[:, 1:, :]`; 2 for
 * DeiT) are not part of the memory.  class_logits_out f32 [batch, Q, num_outputs];
 * bbox_out f32 [batch, Q, 4] in (0, 1). */
int vitk_detection_head_forward(const VitkDetectionHeadConfig* cfg,
                                const VitkDetectionHeadWeights* w, const float* tokens, int batch,
                                int n_tokens, int skip_tokens, float* class_logits_out,
                                float* bbox_out, void* workspace, size_t workspace_bytes,
                                vitk_stream_t stream);

/* ---- training through the head (train.py:842-845 under losses.backward(), train.py:1455) ----
 * The forward below keeps every activation the backward needs in `saved`; with
 * VitkDetectionHeadConfig.dropout_p > 0 the decoder layers' dropout is applied (same seed for the
 * forward and the backward of a step). */

/* W^T copies (bf16 [in, out]) for the input-gradient GEMMs. */
typedef struct VitkDecoderLayerWeightsT {
  const void* sa_in_wt;  /* [D, 3D] */
  const void* sa_out_wt; /* [D, D]  */
  const void* ca_q_wt;   /* [D, D]  */
  const void* ca_out_wt; /* [D, D]  */
  const void* ff1_wt;    /* [D, F]  */
  const void* ff2_wt;    /* [F, D]  */
} VitkDecoderLayerWeightsT;

typedef struct VitkDetectionHeadWeightsT {
  const VitkDecoderLayerWeightsT* layers; /* HOST array of num_layers entries */
  const void* ca_kv_wt;                   /* [D, L*2D] */
} VitkDetectionHeadWeightsT;

/* fp32 gradient buffers with the shapes of VitkDecoderLayerWeights / VitkDetectionHeadWeights;
 * the backward ACCUMULATES into them, the caller zeroes them once per step. */
typedef struct VitkDecoderLayerGrads {
  float* sa_in_w;
  float* sa_in_b;
  float* sa_out_w;
  float* sa_out_b;
  float* ca_q_w;
  float* ca_q_b;
  float* ca_out_w;
  float* ca_out_b;
  float* ff1_w;
  float* ff1_b;
  float* ff2_w;
  float* ff2_b;
  float* norm1_w;
  float* norm1_b;
  float* norm2_w;
  float* norm2_b;
  float* norm3_w;
  float* norm3_b;
} VitkDecoderLayerGrads;

typedef struct VitkDetectionHeadGrads {
  float* object_queries;               /* [Q, D] */
  const VitkDecoderLayerGrads* layers; /* HOST array of num_layers entries */
  float* ca_kv_w;                      /* [L*2D, D] */
  float* ca_kv_b;                      /* [L*2D] */
  float* class_w;
  float* class_b;
  float* bbox_w;
  float* bbox_b;
} VitkDetectionHeadGrads;

/* Bytes of the saved-activation buffer and of the scratch shared by forward and backward. */
int vitk_detection_head_train_bytes(const VitkDetectionHeadConfig* cfg, int batch, int n_tokens,
                                    int skip_tokens, size_t* saved_bytes, size_t* workspace_bytes);

/* vitk_detection_head_forward keeping the activations (both buffers 1024-byte aligned). */
int vitk_detection_head_forward_train(const VitkDetectionHeadConfig* cfg,
                                      const VitkDetectionHeadWeights* w, const float* tokens,
                                      int batch, int n_tokens, int skip_tokens,
                                      float* class_logits_out, float* bbox_out, void* saved,
                                      size_t saved_bytes, void* workspace, size_t workspace_bytes,
                                      vitk_stream_t stream);

/* Backward of the above: d_class_logits f32 [batch, Q, num_outputs] and d_bbox f32 [batch, Q, 4]
 * (gradient w.r.t. the SIGMOID output; bbox = what the forward returned) ->
 * every parameter gradient (accumulated) and d_tokens_out f32 [batch, n_tokens, D] (overwritten;
 * rows of the skipped prefix tokens are zero; may be NULL).  All hand-written kernels: tcgen05
 * GEMMs for the input and weight gradients, CUDA-core attention backward with separate query and
 * key / value sources, fused LayerNorm backward. */
int vitk_detection_head_backward(const VitkDetectionHeadConfig* cfg,
                                 const VitkDetectionHeadWeights* w,
                                 const VitkDetectionHeadWeightsT* wt,
                                 const VitkDetectionHeadGrads* grads, const float* d_class_logits,
                                 const float* d_bbox, const float* bbox, int batch, int n_tokens,
                                 int skip_tokens, float* d_tokens_out, void* saved, void* workspace,
                                 vitk_stream_t stream);

/* ---- data-parallel optimizer step over peer memory (NVLink / NVSwitch) ----
 * Replaces "all-reduce the gradients, then every rank runs the same AdamW" (the data-parallel
 * form of train.py:1455-1460) by a sharded reduce + update + broadcast through symmetric memory:
 * rank r owns the elements [lo_r, hi_r) of the flat arenas.  The caller provides every rank's
 * arenas as peer-mapped device pointers (e.g. torch.distributed._symmetric_memory) and, when the
 * fabric supports it, their multicast addresses; it also enqueues a cross-rank barrier before
 * vitk_peer_reduce_scan, between the two calls and after vitk_peer_adamw_broadcast. */
#define VITK_MAX_PEERS 16
typedef struct VitkPeerBuffers {
  int world;
  int rank;
  const float* grad[VITK_MAX_PEERS]; /* fp32 gradient arena of every rank ([rank] = local) */
  float* param[VITK_MAX_PEERS];      /* fp32 parameter arena of every rank */
  void* shadow[VITK_MAX_PEERS];      /* bf16 shadow arena of every rank */
  int* guard[VITK_MAX_PEERS];        /* int[2] {non-finite flag, steps skipped} of every rank, or all NULL */
  const float* grad_mc;              /* multicast address of the gradient arenas, or NULL */
  float* param_mc;                   /* multicast addresses of the parameter / shadow arenas, or NULL */
  void* shadow_mc;
} VitkPeerBuffers;

/* grad[rank][lo, hi) = sum over ranks of grad[r][lo, hi) (multimem.ld_reduce through the switch
 * when grad_mc is given, else peer loads in rank order); with guard buffers, a non-finite sum sets
 * the flag of EVERY rank.  lo, hi: element offsets, multiples of 4. */
int vitk_peer_reduce_scan(const VitkPeerBuffers* pb, long long lo, long long hi,
                          vitk_stream_t stream);

/* AdamW (the arithmetic of vitk_adamw_step_guarded) on the elements [lo, hi) of the LOCAL arenas
 * with the local exp_avg / exp_avg_sq (full-size arrays indexed by the same offsets: only the owned
 * shard is ever touched), the updated fp32 parameters and bf16 shadows stored to every rank
 * (multimem.st when param_mc / shadow_mc are given).  Skipped when guard[rank][0] != 0. */
int vitk_peer_adamw_broadcast(const VitkPeerBuffers* pb, float* exp_avg, float* exp_avg_sq,
                              long long lo, long long hi, double lr, double beta1, double beta2,
                              double eps, double weight_decay, int step, float grad_scale,
                              vitk_stream_t stream);

/* SetCriterion.loss_labels (train.py:1220-1239): F.cross_entropy(logits, targets, class_weight) -
 * the weighted mean  sum_i w[t_i] * (-log softmax(logits_i)[t_i]) / sum_i w[t_i]  over `rows`
 * predictions (every query of every image; background weight 0.1, train.py:1215-1217).
 * logits f32 [rows, n_classes], targets i64 [rows], class_weight f32 [n_classes] or NULL (ones).
 * loss_out: 1 float; sums_ws: 2 floats of scratch; dlogits_out (optional) f32 [rows, n_classes] =
 * grad_scale * dLoss/dlogits. */
int vitk_weighted_cross_entropy(const float* logits, const long long* targets,
                                const float* class_weight, int rows, int n_classes, float* loss_out,
                                float* sums_ws, float* dlogits_out, float grad_scale,
                                vitk_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* VITK_H_ */
