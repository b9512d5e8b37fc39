// Training-step orchestration behind the C ABI: forward that saves activations, cross-entropy on
// the CLS head, hand-written backward through every encoder block and the patch embedding, fused
// AdamW.  Replaces the autograd part of the reference step (train.py:1441-1460):
//     outputs = model(images) ; loss.backward() ; optimizer.step()
#include "../../include/vitk.h"

#include "attention.cuh"
#include "common.h"
#include "encoder.cuh"
#include "gemm_sm100.cuh"
#include "rowops.cuh"
#include "train_ops.cuh"

namespace vitk {
namespace {

// The shared encoder checks, then what training adds to them.
int check_train_config(const VitkConfig* cfg, int batch, Dims* d) {
  VITK_TRY(check_config(cfg, batch, d));
  VITK_REQUIRE(cfg->precision == 0, "training runs in the bf16 mode only");
  VITK_REQUIRE(cfg->dropout_p >= 0.f && cfg->dropout_p < 1.f, "dropout_p must be in [0, 1)");
  VITK_REQUIRE(attention_trainable(d->N, d->hd),
               "training: head_dim %d with %d tokens is not covered (head_dim 8..128 in steps of 8, "
               "and tokens * head_dim within shared memory)", d->hd, d->N);
  VITK_REQUIRE(cfg->dropout_p == 0.f || d->M * d->Mlp < (1ll << 32),
               "dropout_p > 0 needs batch * tokens * mlp_dim < 2^32");
  return VITK_OK;
}

// Dropout site parameters of one layer (all off when dropout_p == 0).
struct DropSet {
  float p;
  uint32_t seed;
  DropParams at(int site, int layer) const { return make_drop_params(p, seed, site, layer); }
};

// Activations kept from the forward pass for one encoder block.
struct SavedBlock {
  float* x1;     // LN1 input (residual stream before the attention branch) f32 [M, D]
  float* mean1;  // [M]
  float* rstd1;
  void* xn1;     // LN1 output bf16 [M, D]
  void* qkv;     // bf16 [M, 3D]
  float* lse;    // [B, H, N]
  void* ctx;     // bf16 [M, D]
  float* x2;     // LN2 input f32 [M, D]
  float* mean2;
  float* rstd2;
  void* xn2;     // bf16 [M, D]
  void* hpre;    // fc1 pre-activation bf16 [M, Mlp]
  void* hact;    // gelu(hpre) bf16 [M, Mlp]
};

struct Saved {
  void* patches;  // bf16 [Mp, Kp]
  float* mean_f;  // final LayerNorm statistics [M] (token path)
  float* rstd_f;
  size_t block_bytes;
  char* blocks;   // L consecutive block regions
  size_t bytes;
};

SavedBlock carve_block(const Dims& d, void* base, size_t* bytes) {
  Carver c(base);
  SavedBlock s;
  s.x1 = static_cast<float*>(c.take(d.M * d.D * 4));
  s.mean1 = static_cast<float*>(c.take(d.M * 4));
  s.rstd1 = static_cast<float*>(c.take(d.M * 4));
  s.xn1 = c.take(d.M * d.D * 2);
  s.qkv = c.take(d.M * 3 * d.D * 2);
  s.lse = static_cast<float*>(c.take(static_cast<size_t>(d.B) * d.H * d.N * 4));
  s.ctx = c.take(d.M * d.D * 2);
  s.x2 = static_cast<float*>(c.take(d.M * d.D * 4));
  s.mean2 = static_cast<float*>(c.take(d.M * 4));
  s.rstd2 = static_cast<float*>(c.take(d.M * 4));
  s.xn2 = c.take(d.M * d.D * 2);
  s.hpre = c.take(d.M * d.Mlp * 2);
  s.hact = c.take(d.M * d.Mlp * 2);
  if (bytes) *bytes = c.off;
  return s;
}

Saved carve_saved(const Dims& d, void* base) {
  Carver c(base);
  Saved s;
  s.patches = c.take(d.Mp * d.Kp * 2);
  s.mean_f = static_cast<float*>(c.take(d.M * 4));
  s.rstd_f = static_cast<float*>(c.take(d.M * 4));
  carve_block(d, nullptr, &s.block_bytes);
  s.blocks = static_cast<char*>(c.take(s.block_bytes * d.L));
  s.bytes = c.off;
  return s;
}

struct TrainWs {
  float* x;      // residual stream f32 [M, D] (forward) - kept for the loss / final LN backward
  float* dx;     // gradient of the residual stream f32 [M, D]
  void* dxb;     // bf16 copy of dx
  void* dxn;     // gradient w.r.t. a LayerNorm output bf16 [M, D]
  void* dh;      // gradient w.r.t. the fc1 pre-activation bf16 [M, Mlp]
  void* dctx;    // bf16 [M, D]
  void* dqkv;    // bf16 [M, 3D]
  void* dxp;     // bf16 [Mp, D]
  float* feat;   // [B, D]
  float* dlogits;  // [B, C]
  size_t bytes;
};

TrainWs carve_ws(const Dims& d, void* base) {
  Carver c(base);
  TrainWs w;
  w.x = static_cast<float*>(c.take(d.M * d.D * 4));
  w.dx = static_cast<float*>(c.take(d.M * d.D * 4));
  w.dxb = c.take(d.M * d.D * 2);
  w.dxn = c.take(d.M * d.D * 2);
  w.dh = c.take(d.M * d.Mlp * 2);
  w.dctx = c.take(d.M * d.D * 2);
  w.dqkv = c.take(d.M * 3 * d.D * 2);
  w.dxp = c.take(d.Mp * d.D * 2);
  w.feat = static_cast<float*>(c.take(static_cast<size_t>(d.B) * d.D * 4));
  w.dlogits = static_cast<float*>(c.take(static_cast<size_t>(d.B) * (d.ncls > 0 ? d.ncls : 1) * 4));
  w.bytes = c.off;
  return w;
}

int forward_train(const VitkConfig* cfg, const VitkWeights* w, const float* images, const Dims& d,
                  float* tokens_out, const Saved& sv, const TrainWs& ws, cudaStream_t stream) {
  const int M = static_cast<int>(d.M), D = d.D;
  VITK_TRY(patchify(images, sv.patches, d.B, d.C, d.S, d.p, stream));
  VITK_TRY(prefix_tokens(ws.x, w->cls_token, w->dist_token, w->pos_embed, d.B, d.N, D, d.prefix,
                         stream));
  VITK_TRY(patch_embed(sv.patches, w->patch_w, d.B, d.P, d.Kp, D, d.N, d.prefix, w->patch_b,
                       w->pos_embed, ws.x, stream));
  const DropSet drop{cfg->dropout_p, static_cast<uint32_t>(cfg->seed)};
  if (drop.p > 0.f)   // nn.Dropout on tokens + position embedding (train.py:681)
    VITK_TRY(dropout_f32_inplace(ws.x, d.M * D, drop.at(DROP_EMBED, 0), stream));
  for (int l = 0; l < d.L; ++l) {
    const VitkBlockWeights& bw = w->blocks[l];
    const SavedBlock sb = carve_block(d, sv.blocks + l * sv.block_bytes, nullptr);
    const DropParams drop_a = drop.at(DROP_ATTN, l);
    VITK_TRY(layernorm_fwd(ws.x, D, bw.ln1_w, bw.ln1_b, sb.xn1, 0, D, sb.mean1, sb.rstd1, M, D,
                           cfg->ln_eps, stream, sb.x1));
    VITK_TRY(linear_fwd(sb.xn1, D, bw.qkv_w, M, 3 * D, D, EPI_BF16, bw.qkv_b, nullptr, 0, sb.qkv,
                        nullptr, 3 * D, stream));
    VITK_TRY(attention_fwd(sb.qkv, sb.ctx, sb.lse, d.B, d.N, d.H, d.hd, stream, &drop_a));
    VITK_TRY(linear_fwd(sb.ctx, D, bw.proj_w, M, D, D, EPI_RESID_F32, bw.proj_b, ws.x, D, ws.x,
                        nullptr, D, stream, drop.at(DROP_PROJ, l)));
    VITK_TRY(layernorm_fwd(ws.x, D, bw.ln2_w, bw.ln2_b, sb.xn2, 0, D, sb.mean2, sb.rstd2, M, D,
                           cfg->ln_eps, stream, sb.x2));
    VITK_TRY(linear_fwd(sb.xn2, D, bw.fc1_w, M, d.Mlp, D, EPI_GELU_TANH_BF16, bw.fc1_b, nullptr, 0,
                        sb.hact, sb.hpre, d.Mlp, stream, drop.at(DROP_GELU, l)));
    VITK_TRY(linear_fwd(sb.hact, d.Mlp, bw.fc2_w, M, D, d.Mlp, EPI_RESID_F32, bw.fc2_b, ws.x, D,
                        ws.x, nullptr, D, stream, drop.at(DROP_FC2, l)));
  }
  if (tokens_out)
    VITK_TRY(layernorm_fwd(ws.x, D, w->ln_f_w, w->ln_f_b, tokens_out, 1, D, sv.mean_f, sv.rstd_f, M,
                           D, cfg->ln_eps, stream));
  return VITK_OK;
}

// Backward through the blocks and the patch embedding. On entry ws.dx (f32) / ws.dxb (bf16) hold
// the gradient w.r.t. the residual stream after the last block.
int backward_blocks(const VitkConfig* cfg, const VitkWeights* w, const VitkWeightsT* wt,
                    const VitkGrads* g, const Dims& d, const Saved& sv, const TrainWs& ws,
                    cudaStream_t stream, const vitk_event_t* bucket_events = nullptr) {
  const int M = static_cast<int>(d.M), D = d.D, Mlp = d.Mlp;
  const DropSet drop{cfg->dropout_p, static_cast<uint32_t>(cfg->seed)};
  auto bucket_done = [&](int k) -> int {
    if (bucket_events != nullptr && bucket_events[k] != nullptr)
      VITK_CHECK_CUDA(cudaEventRecord(static_cast<cudaEvent_t>(bucket_events[k]), stream));
    return VITK_OK;
  };
  VITK_TRY(bucket_done(0));  // final LayerNorm + head gradients were produced by the caller
  for (int l = d.L - 1; l >= 0; --l) {
    const VitkBlockWeights& bw = w->blocks[l];
    const VitkBlockWeightsT& bt = wt->blocks[l];
    const VitkBlockGrads& bg = g->blocks[l];
    const SavedBlock sb = carve_block(d, sv.blocks + l * sv.block_bytes, nullptr);
    // ---- MLP branch: x_out = x2 + drop(fc2(drop(gelu(fc1(LN2(x2))))))   (train.py:567-573,590-591)
    // with dropout, ws.dxb already carries the linear2-output mask: applied by the LayerNorm backward
    // of the block above (below), or here for the top block whose dxb came from the loss
    if (drop.p > 0.f && l == d.L - 1)
      VITK_TRY(dropout_cast_bf16(ws.dx, ws.dxb, d.M * D, drop.at(DROP_FC2, l), stream));
    VITK_TRY(linear_dgrad(ws.dxb, D, bt.fc2_wt, M, Mlp, EPI_DGELU_BF16, sb.hpre, ws.dh, 0.f, stream,
                          drop.at(DROP_GELU, l)));
    // the bias gradient (column sums of ws.dxb) was produced together with ws.dxb by the
    // LayerNorm backward of the block above, unless dropout re-masked it or this is the top block
    VITK_TRY(linear_wgrad(ws.dxb, D, sb.hact, Mlp, M, bg.fc2_w, l == d.L - 1 ? bg.fc2_b : nullptr,
                          stream));
    VITK_TRY(linear_dgrad(ws.dh, Mlp, bt.fc1_wt, M, D, EPI_BF16, nullptr, ws.dxn, 0.f, stream));
    VITK_TRY(linear_wgrad(ws.dh, Mlp, sb.xn2, D, M, bg.fc1_w, bg.fc1_b, stream));
    const DropParams drop_p = drop.at(DROP_PROJ, l);   // ws.dxb enters the dropped projection output
    VITK_TRY(layernorm_bwd(ws.dxn, 0, D, sb.x2, D, sb.mean2, sb.rstd2, bw.ln2_w, ws.dx, D, 1, ws.dxb,
                           D, bg.ln2_w, bg.ln2_b, M, D, stream, bg.proj_b, &drop_p));
    // ---- attention branch: x2 = x1 + drop(proj(attn(qkv(LN1(x1)))))      (train.py:552-553,586-587)
    VITK_TRY(linear_dgrad(ws.dxb, D, bt.proj_wt, M, D, EPI_BF16, nullptr, ws.dctx, 0.f, stream));
    VITK_TRY(linear_wgrad(ws.dxb, D, sb.ctx, D, M, bg.proj_w, nullptr, stream));
    const DropParams drop_a = drop.at(DROP_ATTN, l);
    VITK_TRY(attention_bwd(sb.qkv, sb.ctx, ws.dctx, sb.lse, ws.dqkv, d.B, d.N, d.H, d.hd, stream,
                           &drop_a, bg.qkv_b));   // also accumulates the qkv bias gradient
    VITK_TRY(linear_dgrad(ws.dqkv, 3 * D, bt.qkv_wt, M, D, EPI_BF16, nullptr, ws.dxn, 0.f, stream));
    VITK_TRY(linear_wgrad(ws.dqkv, 3 * D, sb.xn1, D, M, bg.qkv_w, nullptr, stream));
    // ws.dxb next enters the (dropped) linear2 output of the block below
    const DropParams drop_f = l > 0 ? drop.at(DROP_FC2, l - 1) : DropParams();
    VITK_TRY(layernorm_bwd(ws.dxn, 0, D, sb.x1, D, sb.mean1, sb.rstd1, bw.ln1_w, ws.dx, D, 1, ws.dxb,
                           D, bg.ln1_w, bg.ln1_b, M, D, stream,
                           l == 0 ? nullptr : g->blocks[l - 1].fc2_b, &drop_f));
    VITK_TRY(bucket_done(d.L - l));
  }
  // ---- token assembly + patch embedding                             (evaluation.py:142-149)
  if (drop.p > 0.f)
    VITK_TRY(dropout_f32_inplace(ws.dx, d.M * D, drop.at(DROP_EMBED, 0), stream));
  VITK_TRY(token_grads(ws.dx, d.B, d.N, D, d.prefix, g->pos_embed, g->cls_token, g->dist_token,
                       ws.dxp, stream));
  VITK_TRY(linear_wgrad(ws.dxp, D, sv.patches, d.Kp, static_cast<int>(d.Mp), g->patch_w, g->patch_b,
                        stream));
  return bucket_done(d.L + 1);
}

int check_train_ptrs(const VitkWeights* w, const VitkWeightsT* wt, const VitkGrads* g,
                     const Dims& d) {
  VITK_REQUIRE(w && wt && g, "null weights / grads");
  VITK_REQUIRE(w->blocks && wt->blocks && g->blocks, "null block arrays");
  VITK_REQUIRE(g->patch_w && g->patch_b && g->cls_token && g->pos_embed && g->ln_f_w && g->ln_f_b,
               "grads struct has null members");
  VITK_REQUIRE(d.prefix == 1 || g->dist_token, "DeiT needs a dist_token gradient buffer");
  return VITK_OK;
}

}  // namespace
}  // namespace vitk

using namespace vitk;

extern "C" {

int vitk_dropout_keep_mask(float p, unsigned int seed, int site, int layer, long long n,
                           unsigned char* out, vitk_stream_t stream) {
  VITK_REQUIRE(((site >= 0 && site <= 4) || (site >= 8 && site <= 13)) && layer >= 0,
               "bad dropout site / layer (encoder sites 0..4, decoder-layer sites 8..13)");
  return dropout_keep_mask(out, n, make_drop_params(p, seed, site, layer),
                           static_cast<cudaStream_t>(stream));
}

int vitk_train_workspace_bytes(const VitkConfig* cfg, int batch, size_t* saved_bytes,
                               size_t* workspace_bytes) {
  Dims d;
  VITK_TRY(check_train_config(cfg, batch, &d));
  VITK_REQUIRE(saved_bytes && workspace_bytes, "null output");
  *saved_bytes = carve_saved(d, nullptr).bytes;
  *workspace_bytes = carve_ws(d, nullptr).bytes;
  return VITK_OK;
}

int vitk_forward_train(const VitkConfig* cfg, const VitkWeights* w, const float* images, int batch,
                       float* tokens_out, void* saved, size_t saved_bytes, void* workspace,
                       size_t workspace_bytes, vitk_stream_t stream) {
  Dims d;
  VITK_TRY(check_train_config(cfg, batch, &d));
  VITK_REQUIRE(w && images && saved && workspace && w->blocks, "null argument");
  VITK_REQUIRE((reinterpret_cast<uintptr_t>(saved) & 1023) == 0 &&
                   (reinterpret_cast<uintptr_t>(workspace) & 1023) == 0,
               "saved / workspace must be 1024-byte aligned");
  const Saved sv = carve_saved(d, saved);
  const TrainWs ws = carve_ws(d, workspace);
  if (sv.bytes > saved_bytes || ws.bytes > workspace_bytes)
    return set_error(VITK_ERR_WORKSPACE, "buffers too small: need %zu / %zu bytes", sv.bytes,
                     ws.bytes);
  return forward_train(cfg, w, images, d, tokens_out, sv, ws, static_cast<cudaStream_t>(stream));
}

int vitk_classifier_loss_backward(const VitkConfig* cfg, const VitkWeights* w,
                                  const VitkWeightsT* wt, const VitkGrads* g,
                                  const long long* labels, int batch, float loss_scale,
                                  float* logits_out, float* loss_out, void* saved, void* workspace,
                                  vitk_stream_t stream_) {
  return vitk_classifier_loss_backward_ev(cfg, w, wt, g, labels, batch, loss_scale, logits_out,
                                          loss_out, saved, workspace, nullptr, 0, stream_);
}

int vitk_classifier_loss_backward_ev(const VitkConfig* cfg, const VitkWeights* w,
                                     const VitkWeightsT* wt, const VitkGrads* g,
                                     const long long* labels, int batch, float loss_scale,
                                     float* logits_out, float* loss_out, void* saved,
                                     void* workspace, const vitk_event_t* bucket_events,
                                     int n_events, vitk_stream_t stream_) {
  Dims d;
  VITK_TRY(check_train_config(cfg, batch, &d));
  VITK_REQUIRE(bucket_events == nullptr || n_events == d.L + 2,
               "bucket_events needs num_layers + 2 = %d entries (got %d)", d.L + 2, n_events);
  VITK_TRY(check_train_ptrs(w, wt, g, d));
  VITK_REQUIRE(labels && saved && workspace, "null argument");
  VITK_REQUIRE(d.ncls > 0 && w->head_w && w->head_b && g->head_w && g->head_b,
               "classifier head / head gradients missing");
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  const Saved sv = carve_saved(d, saved);
  const TrainWs ws = carve_ws(d, workspace);
  const int D = d.D;
  VITK_CHECK_CUDA(cudaMemsetAsync(ws.dx, 0, d.M * D * 4, stream));
  VITK_CHECK_CUDA(cudaMemsetAsync(ws.dxb, 0, d.M * D * 2, stream));
  VITK_TRY(cls_loss_bwd(ws.x, static_cast<long long>(d.N) * D, w->ln_f_w, w->ln_f_b, w->head_w,
                        w->head_b, labels, loss_scale, cfg->ln_eps, d.B, D, d.ncls, logits_out,
                        loss_out, ws.feat, ws.dlogits, ws.dx, ws.dxb, g->ln_f_w, g->ln_f_b,
                        g->head_w, g->head_b, stream));
  return backward_blocks(cfg, w, wt, g, d, sv, ws, stream, bucket_events);
}

int vitk_backward_tokens(const VitkConfig* cfg, const VitkWeights* w, const VitkWeightsT* wt,
                         const VitkGrads* g, const float* d_tokens, int batch, void* saved,
                         void* workspace, vitk_stream_t stream_) {
  Dims d;
  VITK_TRY(check_train_config(cfg, batch, &d));
  VITK_TRY(check_train_ptrs(w, wt, g, d));
  VITK_REQUIRE(d_tokens && saved && workspace, "null argument");
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  const Saved sv = carve_saved(d, saved);
  const TrainWs ws = carve_ws(d, workspace);
  const int M = static_cast<int>(d.M), D = d.D;
  // final LayerNorm backward over every token (evaluation.py:156); ws.x still holds its input
  VITK_TRY(layernorm_bwd(d_tokens, 1, D, ws.x, D, sv.mean_f, sv.rstd_f, w->ln_f_w, ws.dx, D, 0,
                         ws.dxb, D, g->ln_f_w, g->ln_f_b, M, D, stream));
  return backward_blocks(cfg, w, wt, g, d, sv, ws, stream);
}

int vitk_adamw_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq,
                    void* shadow_bf16, long long n, double lr, double beta1, double beta2,
                    double eps, double weight_decay, int step, float grad_scale,
                    vitk_stream_t stream) {
  return adamw_flat(params, grads, exp_avg, exp_avg_sq, shadow_bf16, n, lr, beta1, beta2, eps,
                    weight_decay, step, grad_scale, static_cast<cudaStream_t>(stream));
}

int vitk_adamw_step_guarded(float* params, const float* grads, float* exp_avg, float* exp_avg_sq,
                            void* shadow_bf16, long long n, double lr, double beta1, double beta2,
                            double eps, double weight_decay, int step, float grad_scale,
                            const int* guard, vitk_stream_t stream) {
  return adamw_flat(params, grads, exp_avg, exp_avg_sq, shadow_bf16, n, lr, beta1, beta2, eps,
                    weight_decay, step, grad_scale, static_cast<cudaStream_t>(stream), guard);
}

int vitk_grad_guard_scan(const float* grads, long long n, int* guard, int reset,
                         vitk_stream_t stream) {
  return grad_guard_scan(grads, n, guard, reset, static_cast<cudaStream_t>(stream));
}

int vitk_grad_guard_finish(int* guard, vitk_stream_t stream) {
  return grad_guard_finish(guard, static_cast<cudaStream_t>(stream));
}

int vitk_transpose_bf16_batched(int n, const void* const* src, void* const* dst, const int* rows,
                                const int* cols, vitk_stream_t stream) {
  VITK_REQUIRE(n > 0 && src && dst && rows && cols, "transpose: bad argument");
  for (int i0 = 0; i0 < n; i0 += kMaxTransposeJobs) {
    TransposeBatch tb;
    tb.n = (n - i0 < kMaxTransposeJobs) ? n - i0 : kMaxTransposeJobs;
    for (int i = 0; i < tb.n; ++i) {
      tb.src[i] = src[i0 + i];
      tb.dst[i] = dst[i0 + i];
      tb.rows[i] = rows[i0 + i];
      tb.cols[i] = cols[i0 + i];
      VITK_REQUIRE(tb.src[i] && tb.dst[i] && tb.rows[i] > 0 && tb.cols[i] > 0, "transpose: bad job");
      tb.tiles[i] = ((tb.rows[i] + 63) / 64) * ((tb.cols[i] + 63) / 64);
    }
    VITK_TRY(transpose_batched(tb, static_cast<cudaStream_t>(stream)));
  }
  return VITK_OK;
}

int vitk_layernorm_bwd(const void* dy, int dy_is_f32, const float* x, const float* mean,
                       const float* rstd, const float* gamma, float* dx_io, int add_resid,
                       void* dx_bf16, float* dgamma, float* dbeta, int rows, int D,
                       vitk_stream_t stream) {
  return layernorm_bwd(dy, dy_is_f32, D, x, D, mean, rstd, gamma, dx_io, D, add_resid, dx_bf16, D,
                       dgamma, dbeta, rows, D, static_cast<cudaStream_t>(stream));
}

int vitk_attention_bwd(const void* qkv_bf16, const void* ctx_bf16, const void* dctx_bf16,
                       const float* lse, void* dqkv_bf16, int batch, int n_tokens, int num_heads,
                       int head_dim, vitk_stream_t stream) {
  return attention_bwd(qkv_bf16, ctx_bf16, dctx_bf16, lse, dqkv_bf16, batch, n_tokens, num_heads,
                       head_dim, static_cast<cudaStream_t>(stream));
}

int vitk_weighted_cross_entropy(const float* logits, const long long* targets,
                                const float* class_weight, int rows, int n_classes, float* loss_out,
                                float* sums_ws, float* dlogits_out, float grad_scale,
                                vitk_stream_t stream) {
  return weighted_cross_entropy(logits, targets, class_weight, rows, n_classes, loss_out, sums_ws,
                                dlogits_out, grad_scale, static_cast<cudaStream_t>(stream));
}

int vitk_colsum_bf16(const void* y, long long ld, int M, int N, float* out, vitk_stream_t stream) {
  return colsum_bf16(y, ld, M, N, out, static_cast<cudaStream_t>(stream));
}

}  // extern "C"
