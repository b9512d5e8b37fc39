// extern "C" surface of libvitk (include/vitk.h) and the forward orchestration: the kernel
// sequence that replaces `self.backbone(images)` (reference evaluation.py:231 / train.py:831).
#include "../../include/vitk.h"

#include <cuda_bf16.h>

#include <cstdlib>

#include "attention.cuh"
#include "common.h"
#include "encoder.cuh"
#include "fp32_mode.cuh"
#include "gemm_sm100.cuh"
#include "rowops.cuh"

namespace vitk {
namespace {

struct Workspace {
  float* x;     // residual stream f32 [M, D]
  void* xn;     // LN output bf16 [M, D]
  void* qkv;    // bf16 [M, 3D]
  void* ctx;    // bf16 [M, D]
  void* h;      // bf16 [M, Mlp]
  void* patch;  // bf16 [Mp, Kp]
  // CLS-only tail of the last block (vitk_forward_cls): one row per image
  float* c_x;   // f32 [B, D]
  void* c_b;    // bf16 [B, D]  (attention context, then the LayerNorm output)
  void* c_h;    // bf16 [B, Mlp]
  float2* stats;         // folded LayerNorm: [gemm_stats_parts(D)][M] partial (sum, sum of squares)
  size_t bytes;
};

Workspace carve(const Dims& d, void* base) {
  Carver c(base);
  Workspace w;
  w.x = static_cast<float*>(c.take(d.M * d.D * 4));
  w.xn = c.take(d.M * d.D * 2);
  w.qkv = c.take(d.M * 3 * d.D * 2);
  w.ctx = c.take(d.M * d.D * 2);
  w.h = c.take(d.M * d.Mlp * 2);
  w.patch = c.take(d.Mp * d.Kp * 2);
  w.c_x = static_cast<float*>(c.take(static_cast<size_t>(d.B) * d.D * 4));
  w.c_b = c.take(static_cast<size_t>(d.B) * d.D * 2);
  w.c_h = c.take(static_cast<size_t>(d.B) * d.Mlp * 2);
  w.stats = static_cast<float2*>(c.take(static_cast<size_t>(gemm_stats_parts(d.D)) * d.M * 8));
  w.bytes = c.off;
  return w;
}

// LayerNorm folding in vitk_forward: on when every block carries folded weights, unless
// VITK_LN_FOLD=0 / vitk_set_layernorm_folding(0) (A/B timing, tests).
int g_ln_fold = [] {
  const char* v = getenv("VITK_LN_FOLD");
  return (v != nullptr && v[0] == '0') ? 0 : 1;
}();

bool folded_weights_present(const VitkWeights* w, int L) {
  for (int l = 0; l < L; ++l) {
    const VitkBlockWeights& b = w->blocks[l];
    if (!b.qkv_w_ln || !b.qkv_b_ln || !b.fc1_w_ln || !b.fc1_b_ln) return false;
  }
  return true;
}

// The classifier reads only row 0 of the last block's output: its attention needs the keys and
// values of every token (ws.qkv, already computed) but a single query per image, and everything
// after it - projection, LayerNorm, MLP - is row-wise, so it runs on B rows instead of B*N.
// Same logits as the full evaluation (nothing that is skipped feeds them).
int cls_tail(const VitkConfig* cfg, const VitkWeights* w, const Dims& d, const Workspace& ws,
             float* logits_out, cudaStream_t stream) {
  const int D = d.D;
  const VitkBlockWeights& bw = w->blocks[d.L - 1];
  const __nv_bfloat16* qkv = static_cast<const __nv_bfloat16*>(ws.qkv);
  const long long img = static_cast<long long>(d.N) * 3 * D;
  const AttnXSrc src{qkv, img, 3 * D, qkv + D, qkv + 2 * D, img, 3 * D};
  VITK_TRY(attention_src_fwd(src, ws.c_b, D, D, nullptr, d.B, 1, d.N, d.H, d.hd, stream));
  VITK_TRY(linear_fwd(ws.c_b, D, bw.proj_w, d.B, D, D, EPI_RESID_F32, bw.proj_b, ws.x, d.N * D,
                      ws.c_x, nullptr, D, stream));
  VITK_TRY(layernorm_fwd(ws.c_x, D, bw.ln2_w, bw.ln2_b, ws.c_b, 0, D, nullptr, nullptr, d.B, D,
                         cfg->ln_eps, stream));
  VITK_TRY(linear_fwd(ws.c_b, D, bw.fc1_w, d.B, d.Mlp, D, EPI_GELU_TANH_BF16, bw.fc1_b, nullptr, 0,
                      ws.c_h, nullptr, d.Mlp, stream));
  VITK_TRY(linear_fwd(ws.c_h, d.Mlp, bw.fc2_w, d.B, D, d.Mlp, EPI_RESID_F32, bw.fc2_b, ws.c_x, D,
                      ws.c_x, nullptr, D, stream));
  return cls_head(ws.c_x, D, w->ln_f_w, w->ln_f_b, w->head_w, w->head_b, nullptr, logits_out, d.B,
                  D, cfg->n_classes, cfg->ln_eps, stream);
}

// Final LayerNorm of the residual stream x: over every token into tokens_out (the backbone
// contract), and on the CLS rows with the classifier into logits_out; either may be null.
int encoder_tail(const VitkConfig* cfg, const VitkWeights* w, const Dims& d, const float* x,
                 float* tokens_out, float* logits_out, cudaStream_t stream) {
  const int D = d.D;
  if (tokens_out)
    VITK_TRY(layernorm_fwd(x, D, w->ln_f_w, w->ln_f_b, tokens_out, 1, D, nullptr, nullptr,
                           static_cast<int>(d.M), D, cfg->ln_eps, stream));
  if (logits_out)
    VITK_TRY(cls_head(x, static_cast<long long>(d.N) * D, w->ln_f_w, w->ln_f_b, w->head_w,
                      w->head_b, nullptr, logits_out, d.B, D, cfg->n_classes, cfg->ln_eps, stream));
  return VITK_OK;
}

struct U8Input {
  const unsigned char* images_hwc;  // [B, S, S, 3]
  const float* mean;                // 3 host floats
  const float* stddev;
};

int forward_bf16(const VitkConfig* cfg, const VitkWeights* w, const float* images, const Dims& d,
                 float* tokens_out, float* logits_out, const Workspace& ws, cudaStream_t stream,
                 const U8Input* u8 = nullptr, bool cls_only_tail = false) {
  const int M = static_cast<int>(d.M), D = d.D;
  SweepAlternation sweep;  // consecutive row-ordered kernels run in opposite directions (L2 reuse)
  // -- patch embedding as a GEMM; epilogue adds bias + position embedding and writes each patch
  //    row at its token slot (evaluation.py:142-149)
  if (u8 != nullptr)
    VITK_TRY(patchify_u8(u8->images_hwc, ws.patch, d.B, d.S, d.p, u8->mean, u8->stddev, stream));
  else
    VITK_TRY(patchify(images, ws.patch, d.B, d.C, d.S, d.p, stream));
  VITK_TRY(prefix_tokens(ws.x, w->cls_token, w->dist_token, w->pos_embed, d.B, d.N, D, d.prefix,
                         stream));
  VITK_TRY(patch_embed(ws.patch, w->patch_w, d.B, d.P, d.Kp, D, d.N, d.prefix, w->patch_b,
                       w->pos_embed, ws.x, stream));
  if (g_ln_fold && folded_weights_present(w, d.L)) {
    // -- encoder blocks with every LayerNorm folded into the GEMMs around it: 5 launches per
    //    block, no pass over the fp32 residual stream other than the residual GEMMs' own update
    const int parts = gemm_stats_parts(D);
    VITK_TRY(row_stats(ws.x, D, ws.xn, D, ws.stats, M, D, stream));
    int nparts = 1;
    for (int l = 0; l < d.L; ++l) {
      const VitkBlockWeights& bw = w->blocks[l];
      const bool last = (l == d.L - 1);
      VITK_TRY(linear_ln(ws.xn, D, bw.qkv_w_ln, D, M, 3 * D, D, EPI_BF16, bw.qkv_b_ln, ws.stats,
                         nparts, cfg->ln_eps, ws.qkv, 3 * D, stream));
      if (cls_only_tail && last) break;  // cls_tail finishes the block
      VITK_TRY(attention_fwd(ws.qkv, ws.ctx, nullptr, d.B, d.N, d.H, d.hd, stream));
      VITK_TRY(linear_resid_stats(ws.ctx, D, bw.proj_w, D, M, D, D, bw.proj_b, ws.x, ws.xn,
                                  ws.stats, stream));
      nparts = parts;
      VITK_TRY(linear_ln(ws.xn, D, bw.fc1_w_ln, D, M, d.Mlp, D, EPI_GELU_TANH_BF16, bw.fc1_b_ln,
                         ws.stats, nparts, cfg->ln_eps, ws.h, d.Mlp, stream));
      if (!last)
        VITK_TRY(linear_resid_stats(ws.h, d.Mlp, bw.fc2_w, d.Mlp, M, D, d.Mlp, bw.fc2_b, ws.x,
                                    ws.xn, ws.stats, stream));
      else
        VITK_TRY(linear_fwd(ws.h, d.Mlp, bw.fc2_w, M, D, d.Mlp, EPI_RESID_F32, bw.fc2_b, ws.x, D,
                            ws.x, nullptr, D, stream));
    }
  } else {
    // -- encoder blocks (train.py:584-593)
    // LayerNorm 1 of block 0 runs on its own; every later one follows the residual GEMM that
    // produces its input in linear_resid_ln (projection -> LN2, linear2 -> LN1 of the next
    // block)
    VITK_TRY(layernorm_fwd(ws.x, D, w->blocks[0].ln1_w, w->blocks[0].ln1_b, ws.xn, 0, D, nullptr,
                           nullptr, M, D, cfg->ln_eps, stream));
    for (int l = 0; l < d.L; ++l) {
      const VitkBlockWeights& bw = w->blocks[l];
      VITK_TRY(linear_fwd(ws.xn, D, bw.qkv_w, M, 3 * D, D, EPI_BF16, bw.qkv_b, nullptr, 0, ws.qkv,
                          nullptr, 3 * D, stream));
      if (cls_only_tail && l == d.L - 1) break;  // cls_tail finishes the block
      VITK_TRY(attention_fwd(ws.qkv, ws.ctx, nullptr, d.B, d.N, d.H, d.hd, stream));
      VITK_TRY(linear_resid_ln(ws.ctx, D, bw.proj_w, D, M, D, D, bw.proj_b, ws.x, bw.ln2_w,
                               bw.ln2_b, cfg->ln_eps, ws.xn, nullptr, nullptr, stream));
      VITK_TRY(linear_fwd(ws.xn, D, bw.fc1_w, M, d.Mlp, D, EPI_GELU_TANH_BF16, bw.fc1_b, nullptr, 0,
                          ws.h, nullptr, d.Mlp, stream));
      if (l + 1 < d.L) {
        const VitkBlockWeights& nx = w->blocks[l + 1];
        VITK_TRY(linear_resid_ln(ws.h, d.Mlp, bw.fc2_w, d.Mlp, M, D, d.Mlp, bw.fc2_b, ws.x,
                                 nx.ln1_w, nx.ln1_b, cfg->ln_eps, ws.xn, nullptr, nullptr, stream));
      } else {
        VITK_TRY(linear_fwd(ws.h, d.Mlp, bw.fc2_w, M, D, d.Mlp, EPI_RESID_F32, bw.fc2_b, ws.x, D,
                            ws.x, nullptr, D, stream));
      }
    }
  }
  if (cls_only_tail) return cls_tail(cfg, w, d, ws, logits_out, stream);
  return encoder_tail(cfg, w, d, ws.x, tokens_out, logits_out, stream);
}

// ---------------------------------------------------------------------------------------------
// fp32-parity mode (precision = 1): fp32 activations everywhere, every contraction evaluated by
// the tcgen05 kernel on three-term bf16 splits (K' = 6K), attention in fp32 FMAs, exact erf-GELU.
// Weight pointers of VitkWeights then address bf16 [out, 6*in] split matrices (vitk_split3).
// ---------------------------------------------------------------------------------------------
struct WorkspaceF32 {
  float* x;      // residual stream [M, D]
  float* xn;     // LayerNorm output [M, D]
  float* qkv;    // [M, 3D]
  float* ctx;    // [M, D]
  float* h;      // fc1 pre-activation [M, Mlp]
  float* patch;  // [Mp, Kp]
  void* a6;      // split activation operand bf16 [M, 6 * max(D, Mlp, Kp)]
  size_t bytes;
};

WorkspaceF32 carve_f32(const Dims& d, void* base) {
  Carver c(base);
  WorkspaceF32 w;
  int kmax = d.D > d.Mlp ? d.D : d.Mlp;
  if (d.Kp > kmax) kmax = d.Kp;
  w.x = static_cast<float*>(c.take(d.M * d.D * 4));
  w.xn = static_cast<float*>(c.take(d.M * d.D * 4));
  w.qkv = static_cast<float*>(c.take(d.M * 3 * d.D * 4));
  w.ctx = static_cast<float*>(c.take(d.M * d.D * 4));
  w.h = static_cast<float*>(c.take(d.M * d.Mlp * 4));
  w.patch = static_cast<float*>(c.take(d.Mp * d.Kp * 4));
  w.a6 = c.take(d.M * 6 * static_cast<size_t>(kmax) * 2);
  w.bytes = c.off;
  return w;
}

// out(f32) = epilogue(split(A) * W6^T); A f32 [M, K]; W6 bf16 [N, 6K]
int linear_f32(const float* A, int K, const void* W6, int M, int N, GemmEpi epi, const float* bias,
               float* resid_out, float* out, int apply_gelu_to_a, void* a6, cudaStream_t stream) {
  VITK_TRY(split3(A, K, a6, M, K, 0, apply_gelu_to_a, stream));
  return linear_fwd(a6, 6 * K, W6, M, N, 6 * K, epi, bias, resid_out, N,
                    (epi == EPI_RESID_F32) ? resid_out : out, nullptr, N, stream);
}

int forward_f32(const VitkConfig* cfg, const VitkWeights* w, const float* images, const Dims& d,
                float* tokens_out, float* logits_out, const WorkspaceF32& ws, cudaStream_t stream) {
  const int M = static_cast<int>(d.M), D = d.D;
  VITK_TRY(patchify_f32(images, ws.patch, d.B, d.C, d.S, d.p, stream));
  VITK_TRY(prefix_tokens(ws.x, w->cls_token, w->dist_token, w->pos_embed, d.B, d.N, D, d.prefix,
                         stream));
  VITK_TRY(split3(ws.patch, d.Kp, ws.a6, d.Mp, d.Kp, 0, 0, stream));
  VITK_TRY(patch_embed(ws.a6, w->patch_w, d.B, d.P, 6 * d.Kp, D, d.N, d.prefix, w->patch_b,
                       w->pos_embed, ws.x, stream));
  for (int l = 0; l < d.L; ++l) {
    const VitkBlockWeights& bw = w->blocks[l];
    VITK_TRY(layernorm_fwd(ws.x, D, bw.ln1_w, bw.ln1_b, ws.xn, 1, D, nullptr, nullptr, M, D,
                           cfg->ln_eps, stream));
    VITK_TRY(linear_f32(ws.xn, D, bw.qkv_w, M, 3 * D, EPI_F32, bw.qkv_b, nullptr, ws.qkv, 0, ws.a6,
                        stream));
    VITK_TRY(attention_f32(ws.qkv, ws.ctx, d.B, d.N, d.H, d.hd, stream));
    VITK_TRY(linear_f32(ws.ctx, D, bw.proj_w, M, D, EPI_RESID_F32, bw.proj_b, ws.x, nullptr, 0,
                        ws.a6, stream));
    VITK_TRY(layernorm_fwd(ws.x, D, bw.ln2_w, bw.ln2_b, ws.xn, 1, D, nullptr, nullptr, M, D,
                           cfg->ln_eps, stream));
    VITK_TRY(linear_f32(ws.xn, D, bw.fc1_w, M, d.Mlp, EPI_F32, bw.fc1_b, nullptr, ws.h, 0, ws.a6,
                        stream));
    // exact erf-GELU is applied while splitting the fc2 operand
    VITK_TRY(linear_f32(ws.h, d.Mlp, bw.fc2_w, M, D, EPI_RESID_F32, bw.fc2_b, ws.x, nullptr, 1,
                        ws.a6, stream));
  }
  return encoder_tail(cfg, w, d, ws.x, tokens_out, logits_out, stream);
}

size_t workspace_size(const VitkConfig* cfg, const Dims& d) {
  return (cfg->precision == 1) ? carve_f32(d, nullptr).bytes : carve(d, nullptr).bytes;
}

// Argument checks shared by the inference entry points, run after each one's own: the weights,
// the classifier head when logits are requested, and the workspace.
int check_forward_args(const VitkConfig* cfg, const VitkWeights* w, const Dims& d,
                       const float* tokens_out, const float* logits_out, const void* workspace,
                       size_t workspace_bytes) {
  VITK_REQUIRE(w != nullptr && workspace != nullptr, "null argument");
  VITK_REQUIRE(tokens_out != nullptr || logits_out != nullptr,
               "at least one of tokens_out / logits_out must be non-null");
  VITK_REQUIRE(w->blocks != nullptr && w->patch_w && w->patch_b && w->cls_token && w->pos_embed &&
                   w->ln_f_w && w->ln_f_b,
               "weights struct has null members");
  VITK_REQUIRE(d.prefix == 1 || w->dist_token != nullptr, "DeiT needs dist_token");
  if (logits_out)
    VITK_REQUIRE(cfg->n_classes > 0 && w->head_w && w->head_b,
                 "logits requested but no classifier head configured");
  VITK_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 1023) == 0,
               "workspace must be 1024-byte aligned");
  const size_t need = workspace_size(cfg, d);
  if (need > workspace_bytes)
    return set_error(VITK_ERR_WORKSPACE, "workspace too small: need %zu bytes, got %zu", need,
                     workspace_bytes);
  return VITK_OK;
}

}  // namespace
}  // namespace vitk

using namespace vitk;

extern "C" {

int vitk_abi_version(void) { return VITK_ABI_VERSION; }
const char* vitk_last_error(void) { return last_error(); }
long long vitk_launch_count(void) { return launch_count(); }
int vitk_gemm_set_cta_group(int ctas) {
  VITK_REQUIRE(ctas >= 0 && ctas <= 2, "cta_group must be 0 (auto), 1 or 2");
  gemm_force_cta_group(ctas);
  return VITK_OK;
}
int vitk_gemm_set_direct_epilogue(int on) {
  gemm_force_direct_epilogue(on != 0);
  return VITK_OK;
}
int vitk_debug_gemm_trace(long long* out_host, int n) { return gemm_debug_trace(out_host, n); }
int vitk_set_layernorm_folding(int on) {
  g_ln_fold = on != 0;
  return VITK_OK;
}
int vitk_fold_layernorm(const float* weight, const float* gamma, const float* beta,
                        const float* bias, void* w_ln_bf16, float* b_ln, float* rowsum_or_null,
                        int out_features, int in_features, vitk_stream_t stream) {
  return ln_fold(weight, gamma, beta, bias, w_ln_bf16, rowsum_or_null, b_ln, out_features,
                 in_features,
                 static_cast<cudaStream_t>(stream));
}
int vitk_stats_parts(int n_features) { return gemm_stats_parts(n_features); }
int vitk_row_stats(const float* x, long long in_stride, void* x_bf16, long long out_stride,
                   float* stats, int rows, int D, vitk_stream_t stream) {
  return row_stats(x, in_stride, x_bf16, out_stride, reinterpret_cast<float2*>(stats), rows, D,
                   static_cast<cudaStream_t>(stream));
}
int vitk_gemm_resid_stats(const void* A, int lda, const void* W, int ldb, int M, int N, int K,
                          const float* bias, float* x_inout, void* x_bf16, float* stats,
                          vitk_stream_t stream) {
  VITK_REQUIRE(x_inout && x_bf16 && stats, "gemm_resid_stats: null output");
  return linear_resid_stats(A, lda, W, ldb, M, N, K, bias, x_inout, x_bf16,
                            reinterpret_cast<float2*>(stats), static_cast<cudaStream_t>(stream));
}
int vitk_gemm_layernorm_folded(const void* x_bf16, int lda, const void* w_ln, int ldb, int M, int N,
                               int K, int epilogue, const float* b_ln, const float* stats,
                               int n_parts, float eps, void* out, int ldo, vitk_stream_t stream) {
  VITK_REQUIRE(stats != nullptr, "gemm_layernorm_folded: null statistics");
  return linear_ln(x_bf16, lda, w_ln, ldb, M, N, K, static_cast<GemmEpi>(epilogue), b_ln,
                   reinterpret_cast<const float2*>(stats), n_parts, eps, out, ldo,
                   static_cast<cudaStream_t>(stream));
}
int vitk_postprocess_scores(const float* logits, int rows, int n_classes, int exclude_last,
                            float* scores_out, long long* labels_out, float* probs_out,
                            vitk_stream_t stream) {
  return postprocess_scores(logits, rows, n_classes, exclude_last, scores_out, labels_out, probs_out,
                            static_cast<cudaStream_t>(stream));
}
int vitk_postprocess_detections(const float* class_logits, const float* bbox_coords, int batch,
                                int num_queries, int num_outputs, float confidence_threshold,
                                int* counts_out, float* boxes_out, long long* labels_out,
                                float* scores_out, vitk_stream_t stream) {
  return postprocess_detections(class_logits, bbox_coords, batch, num_queries, num_outputs,
                                confidence_threshold, counts_out, boxes_out, labels_out, scores_out,
                                static_cast<cudaStream_t>(stream));
}
int vitk_linear_rows(const float* x, long long row_stride, const float* weight, const float* bias,
                     float* out, int rows, int in_features, int out_features, int l2_normalize,
                     vitk_stream_t stream) {
  return linear_rows(x, row_stride, weight, bias, out, rows, in_features, out_features, l2_normalize,
                     static_cast<cudaStream_t>(stream));
}
int vitk_linear_rows_backward(const float* x, long long row_stride, const float* weight,
                              const float* dy, float* dx, float* dweight, float* dbias, int rows,
                              int in_features, int out_features, vitk_stream_t stream) {
  return linear_rows_bwd(x, row_stride, weight, dy, dx, dweight, dbias, rows, in_features,
                         out_features, static_cast<cudaStream_t>(stream));
}
int vitk_reserve_sms(int n) {
  VITK_REQUIRE(n >= 0 && n <= 64, "reserve_sms: 0 <= n <= 64");
  reserve_sms(n);
  return VITK_OK;
}
int vitk_attention_set_impl(int impl) {
  VITK_REQUIRE(impl >= 0 && impl <= 4,
               "attention impl must be 0 (auto), 1 (flash), 2 (tcgen05), 3 (unpipelined tcgen05) or "
               "4 (long-sequence tcgen05)");
  attention_force_impl(impl);
  return VITK_OK;
}
int vitk_profile_enable(int on) {
  profile_enable(on != 0);
  return VITK_OK;
}
int vitk_profile_collect(double* ms, double* work, long long* launches, int nkinds) {
  VITK_REQUIRE(ms && work && launches && nkinds > 0 && nkinds <= PROF_NKINDS, "bad profile buffers");
  return profile_collect(ms, work, launches, nkinds);
}

int vitk_workspace_bytes(const VitkConfig* cfg, int batch, size_t* out_bytes) {
  Dims d;
  VITK_TRY(check_config(cfg, batch, &d));
  VITK_REQUIRE(out_bytes != nullptr, "out_bytes is null");
  *out_bytes = workspace_size(cfg, d);
  return VITK_OK;
}

int vitk_forward(const VitkConfig* cfg, const VitkWeights* w, const float* images, int batch,
                 float* tokens_out, float* logits_out, void* workspace, size_t workspace_bytes,
                 vitk_stream_t stream) {
  Dims d;
  VITK_TRY(check_config(cfg, batch, &d));
  VITK_REQUIRE(images != nullptr, "null argument");
  VITK_REQUIRE(cfg->precision == 0 || cfg->precision == 1, "unknown precision mode %d",
               cfg->precision);
  VITK_REQUIRE(d.hd == 64 || (cfg->precision == 0 && d.hd >= 8 && d.hd <= 128 && d.hd % 8 == 0),
               "head_dim %d unsupported (bf16: 8..128 in steps of 8; fp32-parity mode: 64)", d.hd);
  VITK_TRY(check_forward_args(cfg, w, d, tokens_out, logits_out, workspace, workspace_bytes));
  if (cfg->precision == 1)
    return forward_f32(cfg, w, images, d, tokens_out, logits_out, carve_f32(d, workspace),
                       static_cast<cudaStream_t>(stream));
  return forward_bf16(cfg, w, images, d, tokens_out, logits_out, carve(d, workspace),
                      static_cast<cudaStream_t>(stream));
}

int vitk_forward_cls(const VitkConfig* cfg, const VitkWeights* w, const float* images, int batch,
                     float* logits_out, void* workspace, size_t workspace_bytes,
                     vitk_stream_t stream) {
  Dims d;
  VITK_TRY(check_config(cfg, batch, &d));
  VITK_REQUIRE(images != nullptr && logits_out != nullptr, "null argument");
  VITK_REQUIRE(cfg->precision == 0, "the CLS-only tail is implemented for the bf16 path");
  VITK_REQUIRE(d.hd == 32 || d.hd == 64 || d.hd == 96 || d.hd == 128 ||
                   attention_src_supported(1, d.N, d.hd),
               "head_dim %d unsupported (32, 64, 96 or 128; any other head_dim from 16 to 128 up to "
               "256 tokens)", d.hd);
  VITK_TRY(check_forward_args(cfg, w, d, nullptr, logits_out, workspace, workspace_bytes));
  return forward_bf16(cfg, w, images, d, nullptr, logits_out, carve(d, workspace),
                      static_cast<cudaStream_t>(stream), nullptr, true);
}

int vitk_forward_u8(const VitkConfig* cfg, const VitkWeights* w, const unsigned char* images_hwc,
                    const float* mean, const float* stddev, int batch, float* tokens_out,
                    float* logits_out, void* workspace, size_t workspace_bytes,
                    vitk_stream_t stream) {
  Dims d;
  VITK_TRY(check_config(cfg, batch, &d));
  VITK_REQUIRE(images_hwc != nullptr && mean != nullptr && stddev != nullptr, "null argument");
  VITK_REQUIRE(cfg->precision == 0, "the 8-bit input edge feeds the bf16 path only");
  VITK_REQUIRE(d.C == 3, "the 8-bit input edge needs RGB images");
  VITK_REQUIRE(d.hd >= 8 && d.hd <= 128 && d.hd % 8 == 0,
               "head_dim %d unsupported (8..128 in steps of 8)", d.hd);
  VITK_TRY(check_forward_args(cfg, w, d, tokens_out, logits_out, workspace, workspace_bytes));
  const U8Input u8{images_hwc, mean, stddev};
  return forward_bf16(cfg, w, nullptr, d, tokens_out, logits_out, carve(d, workspace),
                      static_cast<cudaStream_t>(stream), &u8);
}

int vitk_split3(const float* in, long long ld_in, void* out_bf16, long long rows, int K,
                int is_weight, vitk_stream_t stream) {
  return split3(in, ld_in, out_bf16, rows, K, is_weight, 0, static_cast<cudaStream_t>(stream));
}

int vitk_gemm(const void* A, int lda, const void* B, int ldb, int M, int N, int K, int epilogue,
              const float* bias, const float* resid, int ldr, const void* aux, void* out, void* out2,
              int ldo, float alpha, float beta, vitk_stream_t stream) {
  GemmProblem p;
  p.A = A;
  p.lda = lda;
  p.B = B;
  p.ldb = ldb;
  p.M = M;
  p.N = N;
  p.K = K;
  p.epi = static_cast<GemmEpi>(epilogue);
  p.e.bias = bias;
  p.e.resid = resid;
  p.e.ldr = ldr;
  p.e.aux = aux;
  p.e.out = out;
  p.e.out2 = out2;
  p.e.ldo = ldo;
  p.e.alpha = alpha;
  p.e.beta = beta;
  return gemm_bf16_tn(p, static_cast<cudaStream_t>(stream));
}

int vitk_gemm_resid_layernorm(const void* A, int lda, const void* W, int ldb, int M, int N, int K,
                              const float* bias, float* x_inout, const float* gamma,
                              const float* beta, float eps, void* ln_out, float* mean_out,
                              float* rstd_out, vitk_stream_t stream) {
  // checked before the GEMM updates x: layernorm_fwd takes rows of at most 1024 features
  VITK_REQUIRE(ln_out && x_inout && gamma && beta && N <= 1024,
               "gemm_resid_layernorm: null operand or N > 1024");
  return linear_resid_ln(A, lda, W, ldb, M, N, K, bias, x_inout, gamma, beta, eps, ln_out, mean_out,
                         rstd_out, static_cast<cudaStream_t>(stream));
}

int vitk_gemm_wgrad(const void* A, int lda, const void* B, int ldb, int M, int N, int K, float* out,
                    int ldo, float alpha, float beta, int split_k, vitk_stream_t stream) {
  return gemm_wgrad(A, lda, B, ldb, M, N, K, out, ldo, alpha, beta, split_k,
                    static_cast<cudaStream_t>(stream));
}

int vitk_layernorm(const float* x, long long in_stride, const float* gamma, const float* beta,
                   void* y, int y_is_f32, long long out_stride, float* mean_out, float* rstd_out,
                   int rows, int D, float eps, vitk_stream_t stream) {
  return layernorm_fwd(x, in_stride, gamma, beta, y, y_is_f32, out_stride, mean_out, rstd_out, rows,
                       D, eps, static_cast<cudaStream_t>(stream));
}

int vitk_attention(const void* qkv_bf16, void* ctx_bf16, float* lse_or_null, int batch, int n_tokens,
                   int num_heads, int head_dim, vitk_stream_t stream) {
  return attention_fwd(qkv_bf16, ctx_bf16, lse_or_null, batch, n_tokens, num_heads, head_dim,
                       static_cast<cudaStream_t>(stream));
}

int vitk_attention_src(const void* q, long long q_img, int ldq, const void* k, const void* v,
                       long long kv_img, int ldkv, void* ctx, long long ctx_img, int ldc,
                       float* lse_or_null, int batch, int n_q, int n_k, int num_heads,
                       int head_dim, float dropout_p, unsigned int seed, int site, int layer,
                       vitk_stream_t stream) {
  VITK_REQUIRE(((site >= 0 && site <= 4) || (site >= 8 && site <= 13)) && layer >= 0,
               "bad dropout site / layer (encoder sites 0..4, decoder-layer sites 8..13)");
  const AttnXSrc src{q, q_img, ldq, k, v, kv_img, ldkv};
  const DropParams drop = make_drop_params(dropout_p, seed, site, layer);
  return attention_src_fwd(src, ctx, ctx_img, ldc, lse_or_null, batch, n_q, n_k, num_heads,
                           head_dim, static_cast<cudaStream_t>(stream), &drop);
}

int vitk_attention_src_bwd(const void* q, long long q_img, int ldq, const void* k, const void* v,
                           long long kv_img, int ldkv, const void* ctx, const void* dctx,
                           long long ctx_img, int ldc, const float* lse, void* dq, long long dq_img,
                           int lddq, void* dk, void* dv, long long dkv_img, int lddkv, int batch,
                           int n_q, int n_k, int num_heads, int head_dim, float dropout_p,
                           unsigned int seed, int site, int layer, vitk_stream_t stream) {
  VITK_REQUIRE(((site >= 0 && site <= 4) || (site >= 8 && site <= 13)) && layer >= 0,
               "bad dropout site / layer (encoder sites 0..4, decoder-layer sites 8..13)");
  const AttnXSrc src{q, q_img, ldq, k, v, kv_img, ldkv};
  const DropParams drop = make_drop_params(dropout_p, seed, site, layer);
  return attention_src_bwd(src, ctx, dctx, ctx_img, ldc, lse, dq, dq_img, lddq, dk, dv, dkv_img,
                           lddkv, batch, n_q, n_k, num_heads, head_dim,
                           static_cast<cudaStream_t>(stream), &drop);
}

int vitk_patchify(const float* images, void* patches_bf16, int batch, int channels, int image_size,
                  int patch_size, vitk_stream_t stream) {
  return patchify(images, patches_bf16, batch, channels, image_size, patch_size,
                  static_cast<cudaStream_t>(stream));
}

int vitk_cast_f32_to_bf16(const float* in, void* out_bf16, long long n, vitk_stream_t stream) {
  return cast_f32_to_bf16(in, out_bf16, n, static_cast<cudaStream_t>(stream));
}

}  // extern "C"
