// Detection head (SURVEY.md 8 row f1): ObjectDetectionHead.forward, evaluation.py:160-200 ==
// train.py:691-731 - `nn.TransformerDecoder` of 6 post-LN `nn.TransformerDecoderLayer`s
// (d_model = D, nhead = 8, dim_feedforward = 2048, ReLU, batch_first) decoding `num_queries`
// learned object queries against the encoder's patch tokens, then `class_head` and
// `sigmoid(bbox_head)`.  Inference (eval-mode) forward.
//
// Per layer (torch's TransformerDecoderLayer with norm_first = False):
//     x = norm1(x + self_attn(x, x, x))
//     x = norm2(x + multihead_attn(x, memory, memory))
//     x = norm3(x + linear2(relu(linear1(x))))
//
// What is done differently from the reference's op-by-op execution:
//   * the K/V projections of the encoder tokens for ALL layers are one tcgen05 GEMM
//     ([B*N, D] x [D, L*2D]): the memory does not change between layers;
//   * layer 0's self-attention sees the same queries for every image, so it is evaluated once
//     (Q rows) and broadcast by the LayerNorm that follows;
//   * residual adds are the GEMMs' fp32 reduce-add epilogue, ReLU is fc1's epilogue, every
//     LayerNorm writes the fp32 stream and its bf16 GEMM operand in one pass;
//   * attention (head_dim = D / 8 = 96 for ViT-B) never materialises [B, 8, Q, keys] scores.
#include <cuda_bf16.h>

#include "attention.cuh"
#include "common.h"
#include "gemm_sm100.cuh"
#include "ptx.cuh"
#include "rowops.cuh"
#include "train_ops.cuh"

namespace vitk {
using namespace ptx;

namespace {

// ---------------------------------------------------------------------------------------------
// Post-norm LayerNorm: y = LN(in[r % in_rows]) written twice, fp32 (the residual stream the next
// GEMM reduce-adds into; may alias `in`) and bf16 (the next GEMM's operand).  in_rows < rows
// broadcasts (layer 0: the same queries for every image).  One warp per row.
// ---------------------------------------------------------------------------------------------
constexpr int kLnVec = 8;  // D <= 1024

// Training: the pre-norm row (in_copy), its mean and rstd (rows < in_rows) are kept for the backward.
__global__ void __launch_bounds__(256)
ln_post_kernel(const float* in, int in_rows, const float* __restrict__ gamma,
               const float* __restrict__ beta, float* out_f32, __nv_bfloat16* __restrict__ out_bf16,
               int rows, int D, float eps, float* __restrict__ in_copy,
               float* __restrict__ mean_out, float* __restrict__ rstd_out) {
  const int row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  const float* xr = in + static_cast<size_t>(row % in_rows) * D;
  const int nvec = D >> 2;
  float4 v[kLnVec];
  float s = 0.f;
#pragma unroll
  for (int j = 0; j < kLnVec; ++j) {
    const int i = lane + 32 * j;
    if (i < nvec) {
      v[j] = *reinterpret_cast<const float4*>(xr + 4 * i);
      s += (v[j].x + v[j].y) + (v[j].z + v[j].w);
      if (in_copy != nullptr && row < in_rows)
        *reinterpret_cast<float4*>(in_copy + static_cast<size_t>(row) * D + 4 * i) = v[j];
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  const float mean = s / static_cast<float>(D);
  float sq = 0.f;
#pragma unroll
  for (int j = 0; j < kLnVec; ++j) {
    const int i = lane + 32 * j;
    if (i < nvec) {
      const float a = v[j].x - mean, b = v[j].y - mean, c = v[j].z - mean, d = v[j].w - mean;
      sq += (a * a + b * b) + (c * c + d * d);
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, o);
  const float rstd = rsqrtf(sq / static_cast<float>(D) + eps);
  if (lane == 0 && mean_out != nullptr && row < in_rows) {
    mean_out[row] = mean;
    rstd_out[row] = rstd;
  }
  float* yf = out_f32 + static_cast<size_t>(row) * D;
  __nv_bfloat16* yb = out_bf16 + static_cast<size_t>(row) * D;
#pragma unroll
  for (int j = 0; j < kLnVec; ++j) {
    const int i = lane + 32 * j;
    if (i < nvec) {
      const float4 gm = __ldg(reinterpret_cast<const float4*>(gamma) + i);
      const float4 bt = __ldg(reinterpret_cast<const float4*>(beta) + i);
      float4 y;
      y.x = (v[j].x - mean) * rstd * gm.x + bt.x;
      y.y = (v[j].y - mean) * rstd * gm.y + bt.y;
      y.z = (v[j].z - mean) * rstd * gm.z + bt.z;
      y.w = (v[j].w - mean) * rstd * gm.w + bt.w;
      *reinterpret_cast<float4*>(yf + 4 * i) = y;
      uint2 pk;
      pk.x = pack_bf16x2(y.x, y.y);
      pk.y = pack_bf16x2(y.z, y.w);
      *reinterpret_cast<uint2*>(yb + 4 * i) = pk;
    }
  }
}

int ln_post(const float* in, int in_rows, const float* gamma, const float* beta, float* out_f32,
            void* out_bf16, int rows, int D, float eps, cudaStream_t stream,
            float* in_copy = nullptr, float* mean_out = nullptr, float* rstd_out = nullptr) {
  ProfileScope prof(PROF_LN, static_cast<double>(rows) * D * 10.0, stream);
  ln_post_kernel<<<(rows + 7) / 8, 256, 0, stream>>>(in, in_rows, gamma, beta, out_f32,
                                                     static_cast<__nv_bfloat16*>(out_bf16), rows, D,
                                                     eps, in_copy, mean_out, rstd_out);
  VITK_CHECK_LAUNCH("ln_post_kernel");
  return VITK_OK;
}

// ---------------------------------------------------------------------------------------------
// class_head and sigmoid(bbox_head) on the decoder output (evaluation.py:191-194): one warp per
// query row, fp32 weights (n_cls + 4 rows of D, L1/L2 resident), fp32 accumulation.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
det_heads_kernel(const float* __restrict__ x, const float* __restrict__ cw,
                 const float* __restrict__ cb, const float* __restrict__ bw,
                 const float* __restrict__ bb, float* __restrict__ cls_out,
                 float* __restrict__ box_out, int rows, int D, int n_cls) {
  const int row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  const float4* xr = reinterpret_cast<const float4*>(x + static_cast<size_t>(row) * D);
  const int nvec = D >> 2;
  float4 v[kLnVec];
#pragma unroll
  for (int j = 0; j < kLnVec; ++j) {
    const int i = lane + 32 * j;
    v[j] = (i < nvec) ? xr[i] : make_float4(0.f, 0.f, 0.f, 0.f);
  }
  for (int o = 0; o < n_cls + 4; ++o) {
    const float4* wr = reinterpret_cast<const float4*>(
        (o < n_cls ? cw + static_cast<size_t>(o) * D : bw + static_cast<size_t>(o - n_cls) * D));
    float acc = 0.f;
#pragma unroll
    for (int j = 0; j < kLnVec; ++j) {
      const int i = lane + 32 * j;
      if (i < nvec) {
        const float4 w = __ldg(wr + i);
        acc += (v[j].x * w.x + v[j].y * w.y) + (v[j].z * w.z + v[j].w * w.w);
      }
    }
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, s);
    if (lane == 0) {
      if (o < n_cls) {
        cls_out[static_cast<size_t>(row) * n_cls + o] = acc + cb[o];
      } else {
        const float z = acc + bb[o - n_cls];
        box_out[static_cast<size_t>(row) * 4 + (o - n_cls)] = 1.f / (1.f + __expf(-z));
      }
    }
  }
}

struct HeadDims {
  int B, Ntok, skip, P, D, H, hd, F, L, Q, C;
  long long M, Mm;  // query rows, encoder token rows
};

struct HeadWorkspace {
  float* x;    // decoder stream f32 [M, D]
  void* xb;    // bf16 [M, D]
  void* qkv;   // bf16 [M, 3D]   (cross-attention: the q projection lives in its first D columns)
  void* ctx;   // bf16 [M, D]
  void* h;     // bf16 [M, F]
  void* mem;   // encoder tokens bf16 [Mm, D]
  void* kv;    // their K/V projections for every layer, bf16 [Mm, L*2D]
  float* xq;   // layer-0 self-attention block on the bare queries, f32 [Q, D]
  void* xqb;   // bf16 [Q, D]
  size_t bytes;
};

HeadWorkspace carve(const HeadDims& d, void* base) {
  Carver c(base);
  HeadWorkspace w;
  const size_t D = d.D;
  w.x = static_cast<float*>(c.take(d.M * D * 4));
  w.xb = c.take(d.M * D * 2);
  w.qkv = c.take(d.M * 3 * D * 2);
  w.ctx = c.take(d.M * D * 2);
  w.h = c.take(d.M * static_cast<size_t>(d.F) * 2);
  w.mem = c.take(d.Mm * D * 2);
  w.kv = c.take(d.Mm * static_cast<size_t>(d.L) * 2 * D * 2);
  w.xq = static_cast<float*>(c.take(static_cast<size_t>(d.Q) * D * 4));
  w.xqb = c.take(static_cast<size_t>(d.Q) * D * 2);
  w.bytes = c.off;
  return w;
}

int check(const VitkDetectionHeadConfig* cfg, int batch, int n_tokens, int skip, HeadDims* d) {
  VITK_REQUIRE(cfg != nullptr, "detection head: config is null");
  VITK_REQUIRE(batch > 0 && n_tokens > 0 && skip >= 0 && skip < n_tokens,
               "detection head: bad batch %d / tokens %d / skipped prefix %d", batch, n_tokens, skip);
  VITK_REQUIRE(cfg->embed_dim > 0 && cfg->num_heads > 0 && cfg->embed_dim % cfg->num_heads == 0,
               "detection head: embed_dim %d must be divisible by num_heads %d", cfg->embed_dim,
               cfg->num_heads);
  d->hd = cfg->embed_dim / cfg->num_heads;
  VITK_REQUIRE(d->hd == 32 || d->hd == 64 || d->hd == 96 || d->hd == 128,
               "detection head: head_dim %d unsupported (32, 64, 96 or 128)", d->hd);
  VITK_REQUIRE(cfg->embed_dim % 8 == 0 && cfg->embed_dim <= 128 * kLnVec && cfg->ffn_dim > 0 &&
                   cfg->ffn_dim % 8 == 0,
               "detection head: embed_dim (<= %d) and ffn_dim must be multiples of 8", 128 * kLnVec);
  VITK_REQUIRE(cfg->num_layers > 0 && cfg->num_queries > 0 && cfg->num_outputs > 0,
               "detection head: layers, queries and outputs must be positive");
  d->B = batch;
  d->Ntok = n_tokens;
  d->skip = skip;
  d->P = n_tokens - skip;
  d->D = cfg->embed_dim;
  d->H = cfg->num_heads;
  d->F = cfg->ffn_dim;
  d->L = cfg->num_layers;
  d->Q = cfg->num_queries;
  d->C = cfg->num_outputs;
  d->M = static_cast<long long>(batch) * d->Q;
  d->Mm = static_cast<long long>(batch) * n_tokens;
  VITK_REQUIRE(d->M < (1ll << 29) && d->Mm < (1ll << 29), "detection head: batch too large");
  VITK_REQUIRE(cfg->dropout_p >= 0.f && cfg->dropout_p < 1.f, "detection head: dropout_p %g outside "
               "[0, 1)", static_cast<double>(cfg->dropout_p));
  if (cfg->dropout_p > 0.f)   // element indices of the masks are 32-bit; the fused LayerNorm backward
    VITK_REQUIRE(cfg->embed_dim <= 768 && d->M * static_cast<long long>(cfg->ffn_dim) < (1ll << 32),
                 "detection head: dropout needs embed_dim <= 768 and batch * queries * ffn_dim < 2^32");
  return VITK_OK;
}

int head_forward(const VitkDetectionHeadConfig* cfg, const VitkDetectionHeadWeights* w,
                 const float* tokens, const HeadDims& d, float* class_logits, float* bbox,
                 const HeadWorkspace& ws, cudaStream_t stream) {
  const int D = d.D, M = static_cast<int>(d.M), Q = d.Q;
  const long long imgD = static_cast<long long>(Q) * D;
  const __nv_bfloat16* qkv = static_cast<const __nv_bfloat16*>(ws.qkv);
  const __nv_bfloat16* kv = static_cast<const __nv_bfloat16*>(ws.kv);
  const int ldkv = d.L * 2 * D;
  // -- memory = features[:, skip:, :] (evaluation.py:235): bf16 operand, then K and V of every
  //    layer's multihead_attn in one GEMM (rows of the skipped prefix tokens are computed and
  //    never read)
  VITK_TRY(cast_f32_to_bf16(tokens, ws.mem, d.Mm * D, stream));
  VITK_TRY(linear_fwd(ws.mem, D, w->ca_kv_w, static_cast<int>(d.Mm), ldkv, D, EPI_BF16, w->ca_kv_b,
                      nullptr, 0, ws.kv, nullptr, ldkv, stream));
  for (int l = 0; l < d.L; ++l) {
    const VitkDecoderLayerWeights& lw = w->layers[l];
    // ---- x = norm1(x + self_attn(x, x, x))
    if (l == 0) {
      // object_queries.unsqueeze(0).expand(B, -1, -1) (evaluation.py:186): identical for every
      // image, so the block runs on Q rows and norm1 broadcasts its result
      VITK_CHECK_CUDA(cudaMemcpyAsync(ws.xq, w->object_queries, static_cast<size_t>(Q) * D * 4,
                                      cudaMemcpyDeviceToDevice, stream));
      VITK_TRY(cast_f32_to_bf16(w->object_queries, ws.xqb, static_cast<long long>(Q) * D, stream));
      VITK_TRY(linear_fwd(ws.xqb, D, lw.sa_in_w, Q, 3 * D, D, EPI_BF16, lw.sa_in_b, nullptr, 0,
                          ws.qkv, nullptr, 3 * D, stream));
      const AttnXSrc src{qkv, 0, 3 * D, qkv + D, qkv + 2 * D, 0, 3 * D};
      VITK_TRY(attention_src_fwd(src, ws.ctx, imgD, D, nullptr, 1, Q, Q, d.H, d.hd, stream));
      VITK_TRY(linear_fwd(ws.ctx, D, lw.sa_out_w, Q, D, D, EPI_RESID_F32, lw.sa_out_b, ws.xq, D,
                          ws.xq, nullptr, D, stream));
      VITK_TRY(ln_post(ws.xq, Q, lw.norm1_w, lw.norm1_b, ws.x, ws.xb, M, D, cfg->ln_eps, stream));
    } else {
      VITK_TRY(linear_fwd(ws.xb, D, lw.sa_in_w, M, 3 * D, D, EPI_BF16, lw.sa_in_b, nullptr, 0,
                          ws.qkv, nullptr, 3 * D, stream));
      const long long img = static_cast<long long>(Q) * 3 * D;
      const AttnXSrc src{qkv, img, 3 * D, qkv + D, qkv + 2 * D, img, 3 * D};
      VITK_TRY(attention_src_fwd(src, ws.ctx, imgD, D, nullptr, d.B, Q, Q, d.H, d.hd, stream));
      VITK_TRY(linear_fwd(ws.ctx, D, lw.sa_out_w, M, D, D, EPI_RESID_F32, lw.sa_out_b, ws.x, D,
                          ws.x, nullptr, D, stream));
      VITK_TRY(ln_post(ws.x, M, lw.norm1_w, lw.norm1_b, ws.x, ws.xb, M, D, cfg->ln_eps, stream));
    }
    // ---- x = norm2(x + multihead_attn(x, memory, memory))
    VITK_TRY(linear_fwd(ws.xb, D, lw.ca_q_w, M, D, D, EPI_BF16, lw.ca_q_b, nullptr, 0, ws.qkv,
                        nullptr, D, stream));
    {
      const __nv_bfloat16* kl = kv + static_cast<size_t>(d.skip) * ldkv + static_cast<size_t>(l) * 2 * D;
      const AttnXSrc src{qkv, imgD, D, kl, kl + D, static_cast<long long>(d.Ntok) * ldkv, ldkv};
      VITK_TRY(attention_src_fwd(src, ws.ctx, imgD, D, nullptr, d.B, Q, d.P, d.H, d.hd, stream));
    }
    VITK_TRY(linear_fwd(ws.ctx, D, lw.ca_out_w, M, D, D, EPI_RESID_F32, lw.ca_out_b, ws.x, D, ws.x,
                        nullptr, D, stream));
    VITK_TRY(ln_post(ws.x, M, lw.norm2_w, lw.norm2_b, ws.x, ws.xb, M, D, cfg->ln_eps, stream));
    // ---- x = norm3(x + linear2(relu(linear1(x))))
    VITK_TRY(linear_fwd(ws.xb, D, lw.ff1_w, M, d.F, D, EPI_RELU_BF16, lw.ff1_b, nullptr, 0, ws.h,
                        nullptr, d.F, stream));
    VITK_TRY(linear_fwd(ws.h, d.F, lw.ff2_w, M, D, d.F, EPI_RESID_F32, lw.ff2_b, ws.x, D, ws.x,
                        nullptr, D, stream));
    VITK_TRY(ln_post(ws.x, M, lw.norm3_w, lw.norm3_b, ws.x, ws.xb, M, D, cfg->ln_eps, stream));
  }
  {
    ProfileScope prof(PROF_OTHER, static_cast<double>(M) * D * 4.0, stream);
    det_heads_kernel<<<(M + 7) / 8, 256, 0, stream>>>(ws.x, w->class_w, w->class_b, w->bbox_w,
                                                      w->bbox_b, class_logits, bbox, M, D, d.C);
    VITK_CHECK_LAUNCH("det_heads_kernel");
  }
  return VITK_OK;
}

// =============================================================================================
// Training through the head (train.py:842-845 inside the forward of :1441-1444, differentiated by
// losses.backward() at :1455): the arithmetic above with every activation the backward needs
// kept.  cfg->dropout_p > 0 applies nn.TransformerDecoderLayer's dropout at its six sites per
// layer (dropout.cuh: DROP_DEC_*) with masks that are regenerated, never stored; layer 0 then runs
// on all batch * Q rows (every image draws its own masks) and the attention with dropped
// probabilities uses the CUDA-core kernel.
// =============================================================================================
struct SavedLayer {
  void *xb_in, *qkv, *ctx_sa;     // self-attention operands (layer 0: Q rows, else M rows)
  float *lse_sa, *r1, *mean1, *rstd1;
  void *xb1, *qc, *ctx_ca;
  float *lse_ca, *r2, *mean2, *rstd2;
  void *xb2, *h;
  float *r3, *mean3, *rstd3;
};
struct SavedHead {
  void* mem;      // bf16 [Mm, D]
  void* kv;       // bf16 [Mm, L*2D]
  float* xfinal;  // f32 [M, D] decoder output (input of class_head / bbox_head)
  void* xb_last;  // bf16 [M, D] norm3 output of the last layer (unused by the backward)
  char* layers;   // L blocks of layer_bytes
  size_t layer_bytes, bytes;
};

SavedLayer carve_layer(const HeadDims& d, int l, char* base, size_t* bytes) {
  Carver c(base);
  SavedLayer s;
  // every layer gets the same (largest) layout so that layer_bytes is one number
  (void)l;
  const size_t M = d.M, D = d.D, F = d.F;
  s.xb_in = c.take(M * D * 2);
  s.qkv = c.take(M * 3 * D * 2);
  s.ctx_sa = c.take(M * D * 2);
  s.lse_sa = static_cast<float*>(c.take(static_cast<size_t>(d.B) * d.H * d.Q * 4));
  s.r1 = static_cast<float*>(c.take(M * D * 4));
  s.mean1 = static_cast<float*>(c.take(M * 4));
  s.rstd1 = static_cast<float*>(c.take(M * 4));
  s.xb1 = c.take(M * D * 2);
  s.qc = c.take(M * D * 2);
  s.ctx_ca = c.take(M * D * 2);
  s.lse_ca = static_cast<float*>(c.take(static_cast<size_t>(d.B) * d.H * d.Q * 4));
  s.r2 = static_cast<float*>(c.take(M * D * 4));
  s.mean2 = static_cast<float*>(c.take(M * 4));
  s.rstd2 = static_cast<float*>(c.take(M * 4));
  s.xb2 = c.take(M * D * 2);
  s.h = c.take(M * F * 2);
  s.r3 = static_cast<float*>(c.take(M * D * 4));
  s.mean3 = static_cast<float*>(c.take(M * 4));
  s.rstd3 = static_cast<float*>(c.take(M * 4));
  if (bytes) *bytes = c.off;
  return s;
}

SavedHead carve_saved(const HeadDims& d, void* base) {
  Carver c(base);
  SavedHead s;
  const size_t D = d.D;
  s.mem = c.take(d.Mm * D * 2);
  s.kv = c.take(d.Mm * static_cast<size_t>(d.L) * 2 * D * 2);
  s.xfinal = static_cast<float*>(c.take(d.M * D * 4));
  s.xb_last = c.take(d.M * D * 2);
  carve_layer(d, 0, nullptr, &s.layer_bytes);
  s.layers = static_cast<char*>(c.take(s.layer_bytes * d.L));
  s.bytes = c.off;
  return s;
}

struct HeadTrainWs {
  float* x;      // forward: decoder stream f32 [M, D]; backward: gradient w.r.t. the stream
  float* xq;     // forward: layer-0 block on the bare queries f32 [Q, D]; backward: its gradient
  void* dxb;     // bf16 [M, D]
  void* dh;      // bf16 [M, F]
  void* dctx;    // bf16 [M, D]
  void* dqkv;    // bf16 [M, 3D]
  void* dkv;     // bf16 [Mm, L*2D]
  void* dsumb;   // bf16 [Q, D]
  float* dz;     // f32 [M, C + 4]
  size_t bytes;
};

HeadTrainWs carve_train_ws(const HeadDims& d, void* base) {
  Carver c(base);
  HeadTrainWs w;
  const size_t D = d.D;
  w.x = static_cast<float*>(c.take(d.M * D * 4));
  w.xq = static_cast<float*>(c.take(static_cast<size_t>(d.Q) * D * 4));
  w.dxb = c.take(d.M * D * 2);
  w.dh = c.take(d.M * static_cast<size_t>(d.F) * 2);
  w.dctx = c.take(d.M * D * 2);
  w.dqkv = c.take(d.M * 3 * D * 2);
  w.dkv = c.take(d.Mm * static_cast<size_t>(d.L) * 2 * D * 2);
  w.dsumb = c.take(static_cast<size_t>(d.Q) * D * 2);
  w.dz = static_cast<float*>(c.take(d.M * static_cast<size_t>(d.C + 4) * 4));
  w.bytes = c.off;
  return w;
}

struct HeadDrop {
  float p;
  uint32_t seed;
  bool on() const { return p > 0.f; }
  DropParams at(int site, int layer) const { return make_drop_params(p, seed, site, layer); }
};

// out_f32[row] = in[row % in_rows] (+ bf16 copy): object_queries.unsqueeze(0).expand(B, -1, -1)
__global__ void __launch_bounds__(256)
broadcast_rows_kernel(const float* __restrict__ in, int in_rows, float* __restrict__ out_f32,
                      __nv_bfloat16* __restrict__ out_bf16, long long rows, int D) {
  const long long i = (blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x) * 4;
  if (i >= rows * D) return;
  const long long row = i / D;
  const int col = static_cast<int>(i - row * D);
  const float4 v = *reinterpret_cast<const float4*>(in + (row % in_rows) * D + col);
  *reinterpret_cast<float4*>(out_f32 + i) = v;
  uint2 pk;
  pk.x = pack_bf16x2(v.x, v.y);
  pk.y = pack_bf16x2(v.z, v.w);
  *reinterpret_cast<uint2*>(out_bf16 + i) = pk;
}

int head_forward_train(const VitkDetectionHeadConfig* cfg, const VitkDetectionHeadWeights* w,
                       const float* tokens, const HeadDims& d, float* class_logits, float* bbox,
                       const SavedHead& sv, const HeadTrainWs& ws, cudaStream_t stream) {
  const int D = d.D, M = static_cast<int>(d.M), Q = d.Q;
  const long long imgD = static_cast<long long>(Q) * D;
  const HeadDrop drop{cfg->dropout_p, static_cast<uint32_t>(cfg->seed)};
  const __nv_bfloat16* kv = static_cast<const __nv_bfloat16*>(sv.kv);
  const int ldkv = d.L * 2 * D;
  VITK_TRY(cast_f32_to_bf16(tokens, sv.mem, d.Mm * D, stream));
  VITK_TRY(linear_fwd(sv.mem, D, w->ca_kv_w, static_cast<int>(d.Mm), ldkv, D, EPI_BF16, w->ca_kv_b,
                      nullptr, 0, sv.kv, nullptr, ldkv, stream));
  for (int l = 0; l < d.L; ++l) {
    const VitkDecoderLayerWeights& lw = w->layers[l];
    const SavedLayer sl = carve_layer(d, l, sv.layers + l * sv.layer_bytes, nullptr);
    const __nv_bfloat16* qkv = static_cast<const __nv_bfloat16*>(sl.qkv);
    if (l == 0 && drop.on()) {
      broadcast_rows_kernel<<<static_cast<unsigned>((d.M * D / 4 + 255) / 256), 256, 0, stream>>>(
          w->object_queries, Q, ws.x, static_cast<__nv_bfloat16*>(sl.xb_in), d.M, D);
      VITK_CHECK_LAUNCH("broadcast_rows_kernel");
    }
    if (l == 0 && !drop.on()) {
      VITK_CHECK_CUDA(cudaMemcpyAsync(ws.xq, w->object_queries, static_cast<size_t>(Q) * D * 4,
                                      cudaMemcpyDeviceToDevice, stream));
      VITK_TRY(cast_f32_to_bf16(w->object_queries, sl.xb_in, static_cast<long long>(Q) * D, stream));
      VITK_TRY(linear_fwd(sl.xb_in, D, lw.sa_in_w, Q, 3 * D, D, EPI_BF16, lw.sa_in_b, nullptr, 0,
                          sl.qkv, nullptr, 3 * D, stream));
      const AttnXSrc src{qkv, 0, 3 * D, qkv + D, qkv + 2 * D, 0, 3 * D};
      VITK_TRY(attention_src_fwd(src, sl.ctx_sa, imgD, D, sl.lse_sa, 1, Q, Q, d.H, d.hd, stream));
      VITK_TRY(linear_fwd(sl.ctx_sa, D, lw.sa_out_w, Q, D, D, EPI_RESID_F32, lw.sa_out_b, ws.xq, D,
                          ws.xq, nullptr, D, stream));
      VITK_TRY(ln_post(ws.xq, Q, lw.norm1_w, lw.norm1_b, ws.x, sl.xb1, M, D, cfg->ln_eps, stream,
                       sl.r1, sl.mean1, sl.rstd1));
    } else {
      // sl.xb_in was written by the previous layer's norm3
      VITK_TRY(linear_fwd(sl.xb_in, D, lw.sa_in_w, M, 3 * D, D, EPI_BF16, lw.sa_in_b, nullptr, 0,
                          sl.qkv, nullptr, 3 * D, stream));
      const long long img = static_cast<long long>(Q) * 3 * D;
      const AttnXSrc src{qkv, img, 3 * D, qkv + D, qkv + 2 * D, img, 3 * D};
      const DropParams drop_sa = drop.at(DROP_DEC_SA_ATTN, l);
      VITK_TRY(attention_src_fwd(src, sl.ctx_sa, imgD, D, sl.lse_sa, d.B, Q, Q, d.H, d.hd, stream,
                                 &drop_sa));
      VITK_TRY(linear_fwd(sl.ctx_sa, D, lw.sa_out_w, M, D, D, EPI_RESID_F32, lw.sa_out_b, ws.x, D,
                          ws.x, nullptr, D, stream, drop.at(DROP_DEC_SA_OUT, l)));
      VITK_TRY(ln_post(ws.x, M, lw.norm1_w, lw.norm1_b, ws.x, sl.xb1, M, D, cfg->ln_eps, stream,
                       sl.r1, sl.mean1, sl.rstd1));
    }
    VITK_TRY(linear_fwd(sl.xb1, D, lw.ca_q_w, M, D, D, EPI_BF16, lw.ca_q_b, nullptr, 0, sl.qc,
                        nullptr, D, stream));
    {
      const __nv_bfloat16* kl = kv + static_cast<size_t>(d.skip) * ldkv + static_cast<size_t>(l) * 2 * D;
      const AttnXSrc src{sl.qc, imgD, D, kl, kl + D, static_cast<long long>(d.Ntok) * ldkv, ldkv};
      const DropParams drop_ca = drop.at(DROP_DEC_CA_ATTN, l);
      VITK_TRY(attention_src_fwd(src, sl.ctx_ca, imgD, D, sl.lse_ca, d.B, Q, d.P, d.H, d.hd, stream,
                                 &drop_ca));
    }
    VITK_TRY(linear_fwd(sl.ctx_ca, D, lw.ca_out_w, M, D, D, EPI_RESID_F32, lw.ca_out_b, ws.x, D,
                        ws.x, nullptr, D, stream, drop.at(DROP_DEC_CA_OUT, l)));
    VITK_TRY(ln_post(ws.x, M, lw.norm2_w, lw.norm2_b, ws.x, sl.xb2, M, D, cfg->ln_eps, stream, sl.r2,
                     sl.mean2, sl.rstd2));
    VITK_TRY(linear_fwd(sl.xb2, D, lw.ff1_w, M, d.F, D, EPI_RELU_BF16, lw.ff1_b, nullptr, 0, sl.h,
                        nullptr, d.F, stream, drop.at(DROP_DEC_FFN, l)));
    VITK_TRY(linear_fwd(sl.h, d.F, lw.ff2_w, M, D, d.F, EPI_RESID_F32, lw.ff2_b, ws.x, D, ws.x,
                        nullptr, D, stream, drop.at(DROP_DEC_FF2, l)));
    const bool last = (l == d.L - 1);
    void* xb_next = last ? sv.xb_last
                         : carve_layer(d, l + 1, sv.layers + (l + 1) * sv.layer_bytes, nullptr).xb_in;
    VITK_TRY(ln_post(ws.x, M, lw.norm3_w, lw.norm3_b, last ? sv.xfinal : ws.x, xb_next, M, D,
                     cfg->ln_eps, stream, sl.r3, sl.mean3, sl.rstd3));
  }
  {
    ProfileScope prof(PROF_OTHER, static_cast<double>(M) * D * 4.0, stream);
    det_heads_kernel<<<(M + 7) / 8, 256, 0, stream>>>(sv.xfinal, w->class_w, w->class_b, w->bbox_w,
                                                      w->bbox_b, class_logits, bbox, M, D, d.C);
    VITK_CHECK_LAUNCH("det_heads_kernel");
  }
  return VITK_OK;
}

// ---- backward kernels -----------------------------------------------------------------------
// class_head / bbox_head backward, one warp per query row: dz[row] = (d_logits, d_box * s (1 - s))
// with s the sigmoid the forward returned, dx[row, :] = dz . [class_w; bbox_w].
__global__ void __launch_bounds__(256)
det_heads_bwd_dx_kernel(const float* __restrict__ d_logits, const float* __restrict__ d_box,
                        const float* __restrict__ box, const float* __restrict__ cw,
                        const float* __restrict__ bw, float* __restrict__ dz, float* __restrict__ dx,
                        int rows, int D, int n_cls) {
  const int row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  const int n_out = n_cls + 4;
  float* dzr = dz + static_cast<size_t>(row) * n_out;
  for (int o = lane; o < n_out; o += 32) {
    float g;
    if (o < n_cls) {
      g = d_logits[static_cast<size_t>(row) * n_cls + o];
    } else {
      const float s = box[static_cast<size_t>(row) * 4 + (o - n_cls)];
      g = d_box[static_cast<size_t>(row) * 4 + (o - n_cls)] * s * (1.f - s);
    }
    dzr[o] = g;
  }
  __syncwarp();
  const int nvec = D >> 2;
  for (int i = lane; i < nvec; i += 32) {
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int o = 0; o < n_out; ++o) {
      const float g = dzr[o];
      const float4 wv = __ldg(reinterpret_cast<const float4*>(
                                  o < n_cls ? cw + static_cast<size_t>(o) * D
                                            : bw + static_cast<size_t>(o - n_cls) * D) + i);
      acc.x = fmaf(g, wv.x, acc.x);
      acc.y = fmaf(g, wv.y, acc.y);
      acc.z = fmaf(g, wv.z, acc.z);
      acc.w = fmaf(g, wv.w, acc.w);
    }
    *reinterpret_cast<float4*>(dx + static_cast<size_t>(row) * D + 4 * i) = acc;
  }
}

// dW[o, c] += sum_rows dz[row, o] x[row, c], db[o] += sum_rows dz[row, o]: thread = column c of one
// output o, a slice of the rows per blockIdx.z, one atomic per thread.
__global__ void __launch_bounds__(256)
det_heads_bwd_w_kernel(const float* __restrict__ dz, const float* __restrict__ x,
                       float* __restrict__ dcw, float* __restrict__ dcb, float* __restrict__ dbw,
                       float* __restrict__ dbb, int rows, int D, int n_cls, int rows_per_slice) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  const int o = blockIdx.y;
  const int n_out = n_cls + 4;
  const int r0 = blockIdx.z * rows_per_slice;
  const int r1 = min(rows, r0 + rows_per_slice);
  if (c >= D) return;
  float acc = 0.f, accb = 0.f;
  for (int r = r0; r < r1; ++r) {
    const float g = __ldg(dz + static_cast<size_t>(r) * n_out + o);
    acc = fmaf(g, x[static_cast<size_t>(r) * D + c], acc);
    accb += g;
  }
  float* dw = o < n_cls ? dcw + static_cast<size_t>(o) * D : dbw + static_cast<size_t>(o - n_cls) * D;
  atomicAdd(dw + c, acc);
  if (c == 0) atomicAdd(o < n_cls ? dcb + o : dbb + (o - n_cls), accb);
}

// dh <- scale * dh where the forward's (dropped) ReLU output h was positive, else 0: h > 0 means
// pre-activation > 0 AND kept by the FFN dropout, scale = 1 / (1 - p) (bf16, 8 elements per thread)
__global__ void __launch_bounds__(256)
relu_bwd_kernel(__nv_bfloat16* __restrict__ dh, const __nv_bfloat16* __restrict__ h, long long n8,
                float scale) {
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n8;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    uint4 g = reinterpret_cast<uint4*>(dh)[i];
    const uint4 a = __ldg(reinterpret_cast<const uint4*>(h) + i);
    auto mask = [](uint32_t gv, uint32_t av) {
      // bf16 > 0: sign bit clear and not zero
      const uint32_t lo = ((av & 0x8000u) == 0u && (av & 0x7fffu) != 0u) ? 0x0000ffffu : 0u;
      const uint32_t hi = ((av & 0x80000000u) == 0u && (av & 0x7fff0000u) != 0u) ? 0xffff0000u : 0u;
      return gv & (lo | hi);
    };
    g.x = mask(g.x, a.x);
    g.y = mask(g.y, a.y);
    g.z = mask(g.z, a.z);
    g.w = mask(g.w, a.w);
    if (scale != 1.f) {
      g.x = pack_bf16x2(bf16lo_to_f32(g.x) * scale, bf16hi_to_f32(g.x) * scale);
      g.y = pack_bf16x2(bf16lo_to_f32(g.y) * scale, bf16hi_to_f32(g.y) * scale);
      g.z = pack_bf16x2(bf16lo_to_f32(g.z) * scale, bf16hi_to_f32(g.z) * scale);
      g.w = pack_bf16x2(bf16lo_to_f32(g.w) * scale, bf16hi_to_f32(g.w) * scale);
    }
    reinterpret_cast<uint4*>(dh)[i] = g;
  }
}

// out[q, :] = sum_b in[b, q, :]  (layer 0: every image saw the same queries)
__global__ void __launch_bounds__(256)
batch_sum_kernel(const float* __restrict__ in, float* __restrict__ out, int B, long long per_image) {
  const long long i = (blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x) * 4;
  if (i >= per_image) return;
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int b = 0; b < B; ++b) {
    const float4 v = *reinterpret_cast<const float4*>(in + b * per_image + i);
    acc.x += v.x;
    acc.y += v.y;
    acc.z += v.z;
    acc.w += v.w;
  }
  *reinterpret_cast<float4*>(out + i) = acc;
}

__global__ void __launch_bounds__(256)
accumulate_kernel(float* __restrict__ dst, const float* __restrict__ src, long long n) {
  const long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
  if (i < n) dst[i] += src[i];
}

// norm backward in place on the fp32 gradient stream: dx <- LN'(dx), bf16 copy, dgamma / dbeta
// accumulated, column sums of the result into `colsum` (the bias gradient of the Linear whose
// output the normalised sum received)
// `drop`: mask of the branch output the bf16 copy enters (dropout1 / 2 / 3 of the decoder layer)
int norm_bwd(float* dx, void* dxb, const float* r, const float* mean, const float* rstd,
             const float* gamma, float* dgamma, float* dbeta, float* colsum, int rows, int D,
             cudaStream_t stream, const DropParams& drop = DropParams()) {
  return layernorm_bwd(dx, 1, D, r, D, mean, rstd, gamma, dx, D, 0, dxb, D, dgamma, dbeta, rows, D,
                       stream, colsum, drop.thresh != 0u ? &drop : nullptr);
}

int head_backward(const VitkDetectionHeadConfig* cfg, const VitkDetectionHeadWeights* w,
                  const VitkDetectionHeadWeightsT* wt, const VitkDetectionHeadGrads* g,
                  const float* d_logits, const float* d_box, const float* box, const HeadDims& d,
                  float* d_tokens, const SavedHead& sv, const HeadTrainWs& ws, cudaStream_t stream) {
  const HeadDrop drop{cfg->dropout_p, static_cast<uint32_t>(cfg->seed)};
  const int D = d.D, M = static_cast<int>(d.M), Q = d.Q, F = d.F;
  const int ldkv = d.L * 2 * D;
  const long long imgD = static_cast<long long>(Q) * D;
  // ---- class_head / bbox_head
  {
    ProfileScope prof(PROF_OTHER, static_cast<double>(M) * D * 8.0, stream);
    det_heads_bwd_dx_kernel<<<(M + 7) / 8, 256, 0, stream>>>(d_logits, d_box, box, w->class_w,
                                                             w->bbox_w, ws.dz, ws.x, M, D, d.C);
    VITK_CHECK_LAUNCH("det_heads_bwd_dx_kernel");
    const int slices = 32;
    const int rps = (M + slices - 1) / slices;
    det_heads_bwd_w_kernel<<<dim3((D + 255) / 256, d.C + 4, slices), 256, 0, stream>>>(
        ws.dz, sv.xfinal, g->class_w, g->class_b, g->bbox_w, g->bbox_b, M, D, d.C, rps);
    VITK_CHECK_LAUNCH("det_heads_bwd_w_kernel");
  }
  // rows of the skipped prefix tokens never received keys / values: their gradient is zero
  if (d.skip > 0)
    VITK_CHECK_CUDA(cudaMemset2DAsync(ws.dkv, static_cast<size_t>(d.Ntok) * ldkv * 2, 0,
                                      static_cast<size_t>(d.skip) * ldkv * 2, d.B, stream));
  __nv_bfloat16* dkv = static_cast<__nv_bfloat16*>(ws.dkv);
  __nv_bfloat16* dqkv = static_cast<__nv_bfloat16*>(ws.dqkv);
  const __nv_bfloat16* kv = static_cast<const __nv_bfloat16*>(sv.kv);
  for (int l = d.L - 1; l >= 0; --l) {
    const VitkDecoderLayerWeights& lw = w->layers[l];
    const VitkDecoderLayerWeightsT& lt = wt->layers[l];
    const VitkDecoderLayerGrads& lg = g->layers[l];
    const SavedLayer sl = carve_layer(d, l, sv.layers + l * sv.layer_bytes, nullptr);
    // ---- x = norm3(x2 + linear2(relu(linear1(x2))))
    VITK_TRY(norm_bwd(ws.x, ws.dxb, sl.r3, sl.mean3, sl.rstd3, lw.norm3_w, lg.norm3_w, lg.norm3_b,
                      lg.ff2_b, M, D, stream, drop.at(DROP_DEC_FF2, l)));
    VITK_TRY(linear_dgrad(ws.dxb, D, lt.ff2_wt, M, F, EPI_BF16, nullptr, ws.dh, 0.f, stream));
    {
      const long long n8 = static_cast<long long>(M) * F / 8;
      ProfileScope prof(PROF_OTHER, static_cast<double>(M) * F * 6.0, stream);
      relu_bwd_kernel<<<sm_count() * 8, 256, 0, stream>>>(
          static_cast<__nv_bfloat16*>(ws.dh), static_cast<const __nv_bfloat16*>(sl.h), n8,
          drop.at(DROP_DEC_FFN, l).scale);
      VITK_CHECK_LAUNCH("relu_bwd_kernel");
    }
    VITK_TRY(linear_wgrad(ws.dxb, D, sl.h, F, M, lg.ff2_w, nullptr, stream));
    VITK_TRY(linear_dgrad(ws.dh, F, lt.ff1_wt, M, D, EPI_F32, nullptr, ws.x, 1.f, stream));
    VITK_TRY(linear_wgrad(ws.dh, F, sl.xb2, D, M, lg.ff1_w, lg.ff1_b, stream));
    // ---- x2 = norm2(x1 + multihead_attn(x1, memory, memory))
    VITK_TRY(norm_bwd(ws.x, ws.dxb, sl.r2, sl.mean2, sl.rstd2, lw.norm2_w, lg.norm2_w, lg.norm2_b,
                      lg.ca_out_b, M, D, stream, drop.at(DROP_DEC_CA_OUT, l)));
    VITK_TRY(linear_dgrad(ws.dxb, D, lt.ca_out_wt, M, D, EPI_BF16, nullptr, ws.dctx, 0.f, stream));
    VITK_TRY(linear_wgrad(ws.dxb, D, sl.ctx_ca, D, M, lg.ca_out_w, nullptr, stream));
    {
      const size_t koff = static_cast<size_t>(d.skip) * ldkv + static_cast<size_t>(l) * 2 * D;
      const AttnXSrc src{sl.qc, imgD, D, kv + koff, kv + koff + D,
                         static_cast<long long>(d.Ntok) * ldkv, ldkv};
      const DropParams drop_ca = drop.at(DROP_DEC_CA_ATTN, l);
      VITK_TRY(attention_src_bwd(src, sl.ctx_ca, ws.dctx, imgD, D, sl.lse_ca, dqkv, imgD, D,
                                  dkv + koff, dkv + koff + D, static_cast<long long>(d.Ntok) * ldkv,
                                  ldkv, d.B, Q, d.P, d.H, d.hd, stream, &drop_ca));
    }
    VITK_TRY(linear_dgrad(dqkv, D, lt.ca_q_wt, M, D, EPI_F32, nullptr, ws.x, 1.f, stream));
    VITK_TRY(linear_wgrad(dqkv, D, sl.xb1, D, M, lg.ca_q_w, lg.ca_q_b, stream));
    // ---- x1 = norm1(x0 + self_attn(x0, x0, x0))
    if (l > 0 || drop.on()) {
      VITK_TRY(norm_bwd(ws.x, ws.dxb, sl.r1, sl.mean1, sl.rstd1, lw.norm1_w, lg.norm1_w, lg.norm1_b,
                        lg.sa_out_b, M, D, stream, drop.at(DROP_DEC_SA_OUT, l)));
      VITK_TRY(linear_dgrad(ws.dxb, D, lt.sa_out_wt, M, D, EPI_BF16, nullptr, ws.dctx, 0.f,
                            stream));
      VITK_TRY(linear_wgrad(ws.dxb, D, sl.ctx_sa, D, M, lg.sa_out_w, nullptr, stream));
      const __nv_bfloat16* qkv = static_cast<const __nv_bfloat16*>(sl.qkv);
      const long long img = static_cast<long long>(Q) * 3 * D;
      const AttnXSrc src{qkv, img, 3 * D, qkv + D, qkv + 2 * D, img, 3 * D};
      const DropParams drop_sa = drop.at(DROP_DEC_SA_ATTN, l);
      VITK_TRY(attention_src_bwd(src, sl.ctx_sa, ws.dctx, imgD, D, sl.lse_sa, dqkv, img, 3 * D,
                                  dqkv + D, dqkv + 2 * D, img, 3 * D, d.B, Q, Q, d.H, d.hd, stream,
                                  &drop_sa));
      VITK_TRY(linear_dgrad(dqkv, 3 * D, lt.sa_in_wt, M, D, EPI_F32, nullptr, ws.x, 1.f, stream));
      VITK_TRY(linear_wgrad(dqkv, 3 * D, sl.xb_in, D, M, lg.sa_in_w, lg.sa_in_b, stream));
      if (l == 0) {
        // (dropout: layer 0 ran on every image's own copy of the queries) d queries = sum over images
        batch_sum_kernel<<<static_cast<unsigned>((imgD / 4 + 255) / 256), 256, 0, stream>>>(
            ws.x, ws.xq, d.B, imgD);
        VITK_CHECK_LAUNCH("batch_sum_kernel");
        accumulate_kernel<<<static_cast<unsigned>((imgD + 255) / 256), 256, 0, stream>>>(
            g->object_queries, ws.xq, imgD);
        VITK_CHECK_LAUNCH("accumulate_kernel");
      }
    } else {
      // the block ran once on the bare queries and norm1 broadcast it: LayerNorm's backward is
      // linear in the incoming gradient, so the gradients of the images are summed first
      {
        ProfileScope prof(PROF_OTHER, static_cast<double>(M) * D * 4.0, stream);
        batch_sum_kernel<<<static_cast<unsigned>((imgD / 4 + 255) / 256), 256, 0, stream>>>(
            ws.x, ws.xq, d.B, imgD);
        VITK_CHECK_LAUNCH("batch_sum_kernel");
      }
      VITK_TRY(norm_bwd(ws.xq, ws.dsumb, sl.r1, sl.mean1, sl.rstd1, lw.norm1_w, lg.norm1_w,
                        lg.norm1_b, lg.sa_out_b, Q, D, stream));
      VITK_TRY(linear_dgrad(ws.dsumb, D, lt.sa_out_wt, Q, D, EPI_BF16, nullptr, ws.dctx, 0.f,
                            stream));
      VITK_TRY(linear_wgrad(ws.dsumb, D, sl.ctx_sa, D, Q, lg.sa_out_w, nullptr, stream));
      const __nv_bfloat16* qkv = static_cast<const __nv_bfloat16*>(sl.qkv);
      const AttnXSrc src{qkv, 0, 3 * D, qkv + D, qkv + 2 * D, 0, 3 * D};
      VITK_TRY(attention_src_bwd(src, sl.ctx_sa, ws.dctx, 0, D, sl.lse_sa, dqkv, 0, 3 * D, dqkv + D,
                          dqkv + 2 * D, 0, 3 * D, 1, Q, Q, d.H, d.hd, stream, nullptr));
      VITK_TRY(linear_dgrad(dqkv, 3 * D, lt.sa_in_wt, Q, D, EPI_F32, nullptr, ws.xq, 1.f, stream));
      VITK_TRY(linear_wgrad(dqkv, 3 * D, sl.xb_in, D, Q, lg.sa_in_w, lg.sa_in_b, stream));
      accumulate_kernel<<<static_cast<unsigned>((imgD + 255) / 256), 256, 0, stream>>>(
          g->object_queries, ws.xq, imgD);
      VITK_CHECK_LAUNCH("accumulate_kernel");
    }
  }
  // ---- K / V projections of the memory (all layers at once) and the encoder features
  if (d_tokens != nullptr)
    VITK_TRY(linear_dgrad(ws.dkv, ldkv, wt->ca_kv_wt, static_cast<int>(d.Mm), D, EPI_F32, nullptr,
                          d_tokens, 0.f, stream));
  VITK_TRY(linear_wgrad(ws.dkv, ldkv, sv.mem, D, static_cast<int>(d.Mm), g->ca_kv_w, g->ca_kv_b,
                        stream));
  return VITK_OK;
}

}  // namespace
}  // namespace vitk

using namespace vitk;

extern "C" {

int vitk_detection_head_workspace_bytes(const VitkDetectionHeadConfig* cfg, int batch, int n_tokens,
                                        int skip_tokens, size_t* out_bytes) {
  HeadDims d;
  VITK_TRY(check(cfg, batch, n_tokens, skip_tokens, &d));
  VITK_REQUIRE(out_bytes != nullptr, "detection head: out_bytes is null");
  *out_bytes = carve(d, nullptr).bytes;
  return VITK_OK;
}

int vitk_detection_head_forward(const VitkDetectionHeadConfig* cfg,
                                const VitkDetectionHeadWeights* w, const float* tokens, int batch,
                                int n_tokens, int skip_tokens, float* class_logits_out,
                                float* bbox_out, void* workspace, size_t workspace_bytes,
                                vitk_stream_t stream) {
  HeadDims d;
  VITK_TRY(check(cfg, batch, n_tokens, skip_tokens, &d));
  VITK_REQUIRE(w != nullptr && w->layers != nullptr && w->object_queries != nullptr &&
                   w->ca_kv_w != nullptr && w->class_w != nullptr && w->bbox_w != nullptr,
               "detection head: weights are null");
  VITK_REQUIRE(tokens && class_logits_out && bbox_out && workspace,
               "detection head: null tokens / outputs / workspace");
  VITK_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 1023) == 0,
               "detection head: workspace must be 1024-byte aligned");
  VITK_REQUIRE(device_cc() >= 100, "detection head: requires an sm_100 device (found sm_%d)",
               device_cc());
  const HeadWorkspace ws = carve(d, workspace);
  if (workspace_bytes < ws.bytes)
    return set_error(VITK_ERR_WORKSPACE, "detection head: workspace of %zu bytes < %zu required",
                     workspace_bytes, ws.bytes);
  return head_forward(cfg, w, tokens, d, class_logits_out, bbox_out, ws,
                      static_cast<cudaStream_t>(stream));
}

int vitk_detection_head_train_bytes(const VitkDetectionHeadConfig* cfg, int batch, int n_tokens,
                                    int skip_tokens, size_t* saved_bytes, size_t* workspace_bytes) {
  HeadDims d;
  VITK_TRY(check(cfg, batch, n_tokens, skip_tokens, &d));
  VITK_REQUIRE(saved_bytes != nullptr && workspace_bytes != nullptr,
               "detection head (train): null size outputs");
  *saved_bytes = carve_saved(d, nullptr).bytes;
  *workspace_bytes = carve_train_ws(d, nullptr).bytes;
  return VITK_OK;
}

int vitk_detection_head_forward_train(const VitkDetectionHeadConfig* cfg,
                                      const VitkDetectionHeadWeights* w, const float* tokens,
                                      int batch, int n_tokens, int skip_tokens,
                                      float* class_logits_out, float* bbox_out, void* saved,
                                      size_t saved_bytes, void* workspace, size_t workspace_bytes,
                                      vitk_stream_t stream) {
  HeadDims d;
  VITK_TRY(check(cfg, batch, n_tokens, skip_tokens, &d));
  VITK_REQUIRE(w != nullptr && w->layers != nullptr && w->object_queries != nullptr &&
                   w->ca_kv_w != nullptr && w->class_w != nullptr && w->bbox_w != nullptr,
               "detection head: weights are null");
  VITK_REQUIRE(tokens && class_logits_out && bbox_out && workspace && saved,
               "detection head (train): null tokens / outputs / buffers");
  VITK_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 1023) == 0 &&
                   (reinterpret_cast<uintptr_t>(saved) & 1023) == 0,
               "detection head (train): buffers must be 1024-byte aligned");
  VITK_REQUIRE(device_cc() >= 100, "detection head: requires an sm_100 device (found sm_%d)",
               device_cc());
  const SavedHead sv = carve_saved(d, saved);
  const HeadTrainWs ws = carve_train_ws(d, workspace);
  if (saved_bytes < sv.bytes || workspace_bytes < ws.bytes)
    return set_error(VITK_ERR_WORKSPACE, "detection head (train): buffers of %zu / %zu bytes < %zu "
                     "/ %zu required", saved_bytes, workspace_bytes, sv.bytes, ws.bytes);
  return head_forward_train(cfg, w, tokens, d, class_logits_out, bbox_out, sv, ws,
                            static_cast<cudaStream_t>(stream));
}

int vitk_detection_head_backward(const VitkDetectionHeadConfig* cfg,
                                 const VitkDetectionHeadWeights* w,
                                 const VitkDetectionHeadWeightsT* wt,
                                 const VitkDetectionHeadGrads* grads, const float* d_class_logits,
                                 const float* d_bbox, const float* bbox, int batch, int n_tokens,
                                 int skip_tokens, float* d_tokens_out, void* saved, void* workspace,
                                 vitk_stream_t stream) {
  HeadDims d;
  VITK_TRY(check(cfg, batch, n_tokens, skip_tokens, &d));
  VITK_REQUIRE(w && wt && grads && w->layers && wt->layers && grads->layers && wt->ca_kv_wt,
               "detection head (backward): null weights / gradients");
  VITK_REQUIRE(grads->object_queries && grads->ca_kv_w && grads->ca_kv_b && grads->class_w &&
                   grads->class_b && grads->bbox_w && grads->bbox_b,
               "detection head (backward): gradient struct has null members");
  VITK_REQUIRE(d_class_logits && d_bbox && bbox && saved && workspace,
               "detection head (backward): null gradients / buffers");
  const SavedHead sv = carve_saved(d, saved);
  const HeadTrainWs ws = carve_train_ws(d, workspace);
  return head_backward(cfg, w, wt, grads, d_class_logits, d_bbox, bbox, d, d_tokens_out, sv, ws,
                       static_cast<cudaStream_t>(stream));
}

}  // extern "C"
