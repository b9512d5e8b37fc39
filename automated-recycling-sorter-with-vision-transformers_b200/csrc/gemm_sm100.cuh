// Host-visible declarations for the tcgen05 GEMM (gemm_sm100.cu).
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "dropout.cuh"

namespace vitk {

// Epilogue selector (compile-time variants of one kernel).
enum GemmEpi : int {
  // Per-element bounds of the approximations against the exact erf forms, x = acc + bias (enforced
  // by tests/test_gemm_epilogues_gpu.py):
  EPI_BF16 = 0,        // out_bf16 = acc + bias
  // out_bf16 = x Phi(x) with an erf-fitted logistic Phi (gelu_fast): |error| <= 9e-5;
  // optional out2_bf16 = x
  EPI_GELU_BF16 = 1,
  EPI_RESID_F32 = 2,   // out_f32 = acc + bias + resid_f32   (optional row remap: patch embed)
  EPI_F32 = 3,         // out_f32 = alpha * acc + bias (+ beta * out_f32)
  // out_bf16 = g * gelu'(aux_bf16), g = acc + bias (fc2 dgrad): the exact erf derivative on the
  // direct path (|error| <= 1e-5 |g|), dgelu_tanh_pair on the TMA path (|error| <= |g| (1.3e-4 +
  // 2^-11 (0.5 + 2 |x|)))
  EPI_DGELU_BF16 = 4,
  // the fc1 epilogue of the encoder forward and training: as EPI_GELU_BF16 with the tanh.approx
  // form of the normal CDF, |error| <= 3.3e-5 + 2.5e-4 |x|
  EPI_GELU_TANH_BF16 = 6,
  EPI_RELU_BF16 = 7,   // out_bf16 = max(acc + bias, 0)   (decoder feed-forward, evaluation.py:170-176)
  // x = x + acc + bias in place (out == resid; the tile of x is TMA-loaded into the staging slab,
  // updated there and TMA-stored back), out2_bf16 = bf16(x) and per-row partial sums (sum x,
  // sum x^2) of the updated values -> ln_part_out: what the LayerNorm that follows needs, without
  // a pass of its own over x (train.py:586-591).  TMA epilogue only.
  EPI_RESID_STATS_F32 = 8,
};

struct GemmEpilogue {
  const float* bias = nullptr;   // [N] or null
  const float* resid = nullptr;  // EPI_RESID_F32: fp32 [*, ldr]
  const void* aux = nullptr;     // EPI_DGELU_BF16: bf16 [M, ldo] pre-activation
  void* out = nullptr;           // [M(out rows), ldo]
  void* out2 = nullptr;          // EPI_GELU_BF16 optional pre-activation copy (bf16, ldo)
  int ldo = 0;                   // elements
  int ldr = 0;                   // elements
  // Row remap (token assembly, reference evaluation.py:145-148 / train.py:673-678):
  //   out_row   = (m / rows_per_group) * group_stride + group_offset + m % rows_per_group
  //   resid_row = group_offset + m % rows_per_group        (position-embedding row)
  // rows_per_group == 0 disables the remap (out_row = resid_row = m).
  int rows_per_group = 0;
  int group_stride = 0;
  int group_offset = 0;
  float alpha = 1.f;
  float beta = 0.f;
  // nn.Dropout on the epilogue's result, element index = row * N + column (dropout.cuh):
  //   EPI_RESID_F32: out += dropout(acc + bias)          (projection / linear2 output dropout)
  //   EPI_GELU_*   : out = dropout(gelu(acc + bias))     (out2 keeps the undropped pre-activation)
  //   EPI_DGELU    : out = dropout_mask(acc) * gelu'(aux) (the backward of the above)
  DropParams drop;
  // ---- LayerNorm folded into the two GEMMs around it (inference; DESIGN.md 3.9).
  // Producer (EPI_RESID_STATS_F32): every epilogue thread owns a row and 128 (BLOCK_N / 2) of its
  // columns, so the partial sums need no exchange: ln_part_out[(column group) * M + row] =
  // (sum x, sum x^2) over that group; gemm_stats_parts(N) groups per row, summed by the consumer
  // in a fixed order (deterministic, no atomics).
  float2* ln_part_out = nullptr;
  // Consumer (EPI_BF16 / EPI_GELU_*): A holds bf16(x) (NOT normalised), B holds the row-centred
  // bf16(W * gamma - mean_k(W * gamma)): a zero-sum weight row makes the contraction itself drop
  // the row mean of x, so with rstd of the row from ln_part[0 .. ln_nparts) (M entries each;
  // ln_dim features) out = rstd * acc + bias[n], bias[n] = b[n] + sum_k W[n,k] beta[k]
  // (ln_fold, rowops.cuh) == Linear(LayerNorm(x)).
  const float2* ln_part = nullptr;
  int ln_nparts = 0;
  int ln_dim = 0;
  float ln_eps = 1e-5f;
};

struct GemmProblem {
  const void* A = nullptr;  // bf16 [M, lda], K contiguous
  const void* B = nullptr;  // bf16 [N, ldb], K contiguous  (C = A * B^T)
  int M = 0, N = 0, K = 0;
  int lda = 0, ldb = 0;     // elements
  // mn_major: A is stored [K, lda] with M contiguous and B [K, ldb] with N contiguous
  // (C = A^T B, the weight-gradient contraction over tokens).  EPI_F32 only.
  bool mn_major = false;
  int split_k = 1;          // K range split across work items; needs EPI_F32 with beta == 1
  GemmEpi epi = EPI_BF16;
  GemmEpilogue e;
};

// Returns 0 on success, else a vitk error code (message via vitk_last_error()).
int gemm_bf16_tn(const GemmProblem& p, cudaStream_t stream);

// 0 = choose automatically (CTA pairs whenever M > 128), 1 / 2 = force the cta_group (tests, A/B).
void gemm_force_cta_group(int ctas);
// 1 = always use the register->global epilogue instead of the smem-staged TMA store/reduce.
void gemm_force_direct_epilogue(int on);
// Trace builds (-DVITK_GEMM_TRACE): copies [pair][{total, wait operands, wait accumulator stage,
// tiles}] SM-clock counts of the last GEMM launch into out (n entries); returns the entries
// written, 0 when the library is not a trace build.
int gemm_debug_trace(long long* out, int n);
// Column groups per row of EPI_RESID_STATS_F32's partial sums for an N-column output.
int gemm_stats_parts(int N);

// ---- The GEMM calls of the encoder, training and detection-head drivers (gemm_sm100.cu).  W is
// bf16 [N, K] with K contiguous; leading dimensions are in elements.

// out = epilogue(A W^T + bias): EPI_RESID_F32 adds resid (rows of ldr elements; out == resid
// updates in place), the GELU epilogues keep the pre-activation in out2.
int linear_fwd(const void* A, int lda, const void* W, int M, int N, int K, GemmEpi epi,
               const float* bias, const float* resid, int ldr, void* out, void* out2, int ldo,
               cudaStream_t stream, const DropParams& drop = DropParams());
// dX[M, in_f] = dY[M, out_f] W[out_f, in_f] with Wt = W^T [in_f, out_f] as the K-major operand:
// a bf16 epilogue (aux: EPI_DGELU_BF16's pre-activation), or EPI_F32 with dX = acc + beta * dX.
int linear_dgrad(const void* dY, int out_f, const void* Wt, int M, int in_f, GemmEpi epi,
                 const void* aux, void* dX, float beta, cudaStream_t stream,
                 const DropParams& drop = DropParams());
// dW[out_f, in_f] += dY[rows, out_f]^T X[rows, in_f], split over the rows so that every CTA pair
// gets about two work items; db[out_f] += column sums of dY unless db is null.
int linear_wgrad(const void* dY, int out_f, const void* X, int in_f, int rows, float* dW,
                 float* db, cudaStream_t stream);
// out[M, N] = alpha * A^T B + beta * out with A [K, lda] (M contiguous) and B [K, ldb] (N
// contiguous): the MN-major form linear_wgrad runs, with the caller's split_k.
int gemm_wgrad(const void* A, int lda, const void* B, int ldb, int M, int N, int K, float* out,
               int ldo, float alpha, float beta, int split_k, cudaStream_t stream);
// Patch embedding: x[token row] = patches W^T + bias + pos_embed[token], patches [B * P, K], for
// the P patch rows of every image; they land after the `prefix` learned tokens of its N-row block
// of the residual stream x [B * N, D].
int patch_embed(const void* patches, const void* W, int B, int P, int K, int D, int N, int prefix,
                const float* bias, const float* pos_embed, float* x, cudaStream_t stream);
// x[M, N] += A W^T + bias in place, then ln_out bf16 = LN(x) * gamma + beta with optional mean /
// rstd: the residual GEMM and a layernorm_fwd launch.
int linear_resid_ln(const void* A, int lda, const void* W, int ldb, int M, int N, int K,
                    const float* bias, float* x, const float* gamma, const float* beta, float eps,
                    void* ln_out, float* mean_out, float* rstd_out, cudaStream_t stream);
// x[M, N] += A W^T + bias in place; xb = bf16(x); partial row statistics of the updated x
// (EPI_RESID_STATS_F32).
int linear_resid_stats(const void* A, int lda, const void* W, int ldb, int M, int N, int K,
                       const float* bias, float* x, void* xb, float2* stats, cudaStream_t stream);
// out = epilogue(Linear(LayerNorm(x))) from xb = bf16(x) [M, K], the folded weights w_ln / b_ln
// and nparts partial row statistics (the consumer side of GemmEpilogue::ln_part).
int linear_ln(const void* xb, int lda, const void* w_ln, int ldb, int M, int N, int K, GemmEpi epi,
              const float* b_ln, const float2* stats, int nparts, float eps, void* out, int ldo,
              cudaStream_t stream);
}  // namespace vitk
