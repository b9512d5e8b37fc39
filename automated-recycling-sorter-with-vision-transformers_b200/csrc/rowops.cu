// HBM-bound row kernels of the encoder: LayerNorm, patch extraction (im2col of non-overlapping
// patches), prefix-token rows, CLS-row LayerNorm + classifier head, dtype casts.
// All are vectorised (16-byte accesses), coalesced along the feature dimension, warp-per-row where
// a row reduction is needed.
#include "rowops.cuh"

#include <cuda_bf16.h>

#include "common.h"
#include "ptx.cuh"

namespace vitk {
using namespace ptx;

namespace {

constexpr int kLnMaxVec = 8;  // 8 float4 per lane -> D <= 1024

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

__device__ __forceinline__ void store4(float* p, float a, float b, float c, float d) {
  *reinterpret_cast<float4*>(p) = make_float4(a, b, c, d);
}
__device__ __forceinline__ void store4(__nv_bfloat16* p, float a, float b, float c, float d) {
  uint2 pk;
  pk.x = pack_bf16x2(a, b);
  pk.y = pack_bf16x2(c, d);
  *reinterpret_cast<uint2*>(p) = pk;
}

// nn.LayerNorm(D), eps inside the sqrt, biased variance (reference train.py:581-582,586,590;
// evaluation.py:136,156). One warp per row, two-pass statistics in registers.
// Five resident blocks per SM (48 registers): 40 warps of loads in flight instead of 32; same-box
// A/B (tests/ab_forward.py): 41.1 -> 40.1 us for 50 432 x 768 rows.  Six (40 registers) spills
// and is 60 % slower; streaming (ld.global.cs) loads are 2.6x slower.
template <typename OutT>
__global__ void __launch_bounds__(256, 5)
layernorm_fwd_kernel(const float* __restrict__ x, long long in_stride,
                     const float* __restrict__ gamma, const float* __restrict__ beta,
                     OutT* __restrict__ y, long long out_stride, float* __restrict__ mean_out,
                     float* __restrict__ rstd_out, float* __restrict__ x_copy, int rows, int D,
                     float eps, int descending) {
  int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (warp >= rows) return;
  if (descending) warp = rows - 1 - warp;  // blocks are scheduled in index order
  const float* xr = x + static_cast<long long>(warp) * in_stride;
  const int nvec = D >> 2;
  float4 v[kLnMaxVec];
  float s = 0.f;
#pragma unroll
  for (int j = 0; j < kLnMaxVec; ++j) {
    const int i = lane + 32 * j;
    if (i < nvec) {
      v[j] = *reinterpret_cast<const float4*>(xr + 4 * i);
      if (x_copy != nullptr)
        *reinterpret_cast<float4*>(x_copy + static_cast<long long>(warp) * D + 4 * i) = v[j];
      s += (v[j].x + v[j].y) + (v[j].z + v[j].w);
    }
  }
  const float mean = warp_sum(s) / static_cast<float>(D);
  float sq = 0.f;
#pragma unroll
  for (int j = 0; j < kLnMaxVec; ++j) {
    const int i = lane + 32 * j;
    if (i < nvec) {
      const float a = v[j].x - mean, b = v[j].y - mean, c = v[j].z - mean, d = v[j].w - mean;
      sq += (a * a + b * b) + (c * c + d * d);
    }
  }
  const float rstd = rsqrtf(warp_sum(sq) / static_cast<float>(D) + eps);
  if (lane == 0) {
    if (mean_out) mean_out[warp] = mean;
    if (rstd_out) rstd_out[warp] = rstd;
  }
  OutT* yr = y + static_cast<long long>(warp) * out_stride;
#pragma unroll
  for (int j = 0; j < kLnMaxVec; ++j) {
    const int i = lane + 32 * j;
    if (i < nvec) {
      const float4 g = __ldg(reinterpret_cast<const float4*>(gamma) + i);
      const float4 b = __ldg(reinterpret_cast<const float4*>(beta) + i);
      store4(yr + 4 * i, (v[j].x - mean) * rstd * g.x + b.x, (v[j].y - mean) * rstd * g.y + b.y,
             (v[j].z - mean) * rstd * g.z + b.z, (v[j].w - mean) * rstd * g.w + b.w);
    }
  }
}

// images f32 NCHW [B,C,S,S] -> patch rows bf16 [B*P, C*p*p], column order (c, kh, kw) ==
// conv.weight.reshape(D, -1) (reference train.py:505-515). Each thread moves 8 pixels of one
// image row: 32-byte read, 16-byte write.
__global__ void __launch_bounds__(256)
patchify_kernel(const float* __restrict__ img, __nv_bfloat16* __restrict__ out, int B, int C, int S,
                int p) {
  const int groups_per_row = S >> 3;
  const long long total = static_cast<long long>(B) * C * S * groups_per_row;
  const int grid_w = S / p;
  const int P = grid_w * grid_w;
  const int Kp = C * p * p;
  for (long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; idx < total;
       idx += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int xg = static_cast<int>(idx % groups_per_row);
    long long t = idx / groups_per_row;
    const int y = static_cast<int>(t % S);
    t /= S;
    const int c = static_cast<int>(t % C);
    const int b = static_cast<int>(t / C);
    const float4* src = reinterpret_cast<const float4*>(img + idx * 8);
    const float4 a0 = __ldg(src), a1 = __ldg(src + 1);
    const int x0 = xg * 8;
    const int px = x0 / p, kw0 = x0 - px * p;
    const int py = y / p, kh = y - py * p;
    const long long row = static_cast<long long>(b) * P + py * grid_w + px;
    const int col = c * p * p + kh * p + kw0;
    uint4 pk;
    pk.x = pack_bf16x2(a0.x, a0.y);
    pk.y = pack_bf16x2(a0.z, a0.w);
    pk.z = pack_bf16x2(a1.x, a1.y);
    pk.w = pack_bf16x2(a1.z, a1.w);
    *reinterpret_cast<uint4*>(out + row * Kp + col) = pk;
  }
}

// The input edge of the reference's data pipeline fused into the patch gather: 8-bit RGB images in
// the decoder's layout (HWC, [B, S, S, 3]) -> A.Normalize(mean, std) -> ToTensorV2 (evaluation.py:
// 362-364, train.py:442-443) -> bf16 patch rows.  The normalisation is evaluated exactly as the
// reference does it in fp32 - (u / 255 - mean) / std with IEEE divisions - so the patch rows are
// bit-identical to patchify(normalised f32 image); the host sends 1 byte per value instead of 4.
// Thread = 8 pixels of one image row: 24-byte read, three 16-byte writes (one per channel plane).
__global__ void __launch_bounds__(256)
patchify_u8_kernel(const unsigned char* __restrict__ img, __nv_bfloat16* __restrict__ out, int B,
                   int S, int p, float m0, float m1, float m2, float s0, float s1, float s2) {
  const int groups_per_row = S >> 3;
  const long long total = static_cast<long long>(B) * S * groups_per_row;
  const int grid_w = S / p;
  const int P = grid_w * grid_w;
  const int Kp = 3 * p * p;
  for (long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; idx < total;
       idx += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int xg = static_cast<int>(idx % groups_per_row);
    long long t = idx / groups_per_row;
    const int y = static_cast<int>(t % S);
    const int b = static_cast<int>(t / S);
    const uint2* src = reinterpret_cast<const uint2*>(img + idx * 24);
    const uint2 a = __ldg(src), bb = __ldg(src + 1), cc = __ldg(src + 2);
    const unsigned int w[6] = {a.x, a.y, bb.x, bb.y, cc.x, cc.y};
    float v[3][8];
#pragma unroll
    for (int k = 0; k < 24; ++k) {
      const float u = static_cast<float>((w[k >> 2] >> (8 * (k & 3))) & 0xFFu);
      const int ch = k % 3;
      const float mean = ch == 0 ? m0 : (ch == 1 ? m1 : m2);
      const float sd = ch == 0 ? s0 : (ch == 1 ? s1 : s2);
      v[ch][k / 3] = __fdiv_rn(__fsub_rn(__fdiv_rn(u, 255.0f), mean), sd);
    }
    const int x0 = xg * 8;
    const int px = x0 / p, kw0 = x0 - px * p;
    const int py = y / p, kh = y - py * p;
    const long long row = static_cast<long long>(b) * P + py * grid_w + px;
#pragma unroll
    for (int ch = 0; ch < 3; ++ch) {
      uint4 pk;
      pk.x = pack_bf16x2(v[ch][0], v[ch][1]);
      pk.y = pack_bf16x2(v[ch][2], v[ch][3]);
      pk.z = pack_bf16x2(v[ch][4], v[ch][5]);
      pk.w = pack_bf16x2(v[ch][6], v[ch][7]);
      *reinterpret_cast<uint4*>(out + row * Kp + ch * p * p + kh * p + kw0) = pk;
    }
  }
}

// x[b, t, :] = token[t] + pos[t]  for the n_prefix learned tokens (CLS, and DIST for DeiT)
// (reference evaluation.py:145-149, train.py:669-680).
__global__ void prefix_tokens_kernel(float* __restrict__ x, const float* __restrict__ cls,
                                     const float* __restrict__ dist, const float* __restrict__ pos,
                                     int B, int Ntok, int D, int n_prefix) {
  const int nvec = D >> 2;
  const long long total = static_cast<long long>(B) * n_prefix * nvec;
  for (long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; idx < total;
       idx += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int i = static_cast<int>(idx % nvec);
    const int t = static_cast<int>((idx / nvec) % n_prefix);
    const int b = static_cast<int>(idx / (static_cast<long long>(nvec) * n_prefix));
    const float4 tok = __ldg(reinterpret_cast<const float4*>(t == 0 ? cls : dist) + i);
    const float4 pe = __ldg(reinterpret_cast<const float4*>(pos + static_cast<long long>(t) * D) + i);
    float* dst = x + (static_cast<long long>(b) * Ntok + t) * D + 4 * i;
    store4(dst, tok.x + pe.x, tok.y + pe.y, tok.z + pe.z, tok.w + pe.w);
  }
}

// Final LayerNorm on the CLS row only + Linear(D, n_classes): logits[b, c].
// (north_star's classifier: Linear(D,6) on features[:,0]; LN per evaluation.py:156.)
// One block of 128 threads per image; the normalised row lives in shared memory.
__global__ void __launch_bounds__(128)
cls_head_kernel(const float* __restrict__ x, long long row_stride, const float* __restrict__ gamma,
                const float* __restrict__ beta, const float* __restrict__ head_w,
                const float* __restrict__ head_b, float* __restrict__ feat_out,
                float* __restrict__ logits, int D, int n_classes, float eps) {
  extern __shared__ float srow[];  // D floats + 8 scratch
  float* red = srow + D;
  const int b = blockIdx.x;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const float* xr = x + static_cast<long long>(b) * row_stride;
  float s = 0.f;
  for (int i = tid; i < D; i += 128) {
    const float v = xr[i];
    srow[i] = v;
    s += v;
  }
  s = warp_sum(s);
  if (lane == 0) red[warp] = s;
  __syncthreads();
  const float mean = (red[0] + red[1] + red[2] + red[3]) / static_cast<float>(D);
  __syncthreads();
  float sq = 0.f;
  for (int i = tid; i < D; i += 128) {
    const float d = srow[i] - mean;
    sq += d * d;
  }
  sq = warp_sum(sq);
  if (lane == 0) red[warp] = sq;
  __syncthreads();
  const float rstd = rsqrtf((red[0] + red[1] + red[2] + red[3]) / static_cast<float>(D) + eps);
  for (int i = tid; i < D; i += 128) {
    const float v = (srow[i] - mean) * rstd * gamma[i] + beta[i];
    srow[i] = v;
    if (feat_out) feat_out[static_cast<long long>(b) * D + i] = v;
  }
  __syncthreads();
  for (int c = warp; c < n_classes; c += 4) {
    const float* w = head_w + static_cast<long long>(c) * D;
    float acc = 0.f;
    for (int i = lane; i < D; i += 32) acc = fmaf(srow[i], __ldg(w + i), acc);
    acc = warp_sum(acc);
    if (lane == 0) logits[static_cast<long long>(b) * n_classes + c] = acc + head_b[c];
  }
}

__global__ void __launch_bounds__(256)
cast_f32_bf16_kernel(const float* __restrict__ in, __nv_bfloat16* __restrict__ out, long long n) {
  const long long nvec = n >> 3;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < nvec;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const float4 a = __ldg(reinterpret_cast<const float4*>(in) + 2 * i);
    const float4 b = __ldg(reinterpret_cast<const float4*>(in) + 2 * i + 1);
    uint4 pk;
    pk.x = pack_bf16x2(a.x, a.y);
    pk.y = pack_bf16x2(a.z, a.w);
    pk.z = pack_bf16x2(b.x, b.y);
    pk.w = pack_bf16x2(b.z, b.w);
    reinterpret_cast<uint4*>(out)[i] = pk;
  }
  // tail
  const long long tail0 = nvec << 3;
  for (long long i = tail0 + blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<long long>(gridDim.x) * blockDim.x)
    out[i] = __float2bfloat16_rn(in[i]);
}

// ---- LayerNorm folded into the GEMMs around it (gemm_sm100.cuh: GemmEpilogue::ln_part) ---------
// Entry of the chain (block 0, after token assembly): bf16 copy of the rows and their (sum,
// sum of squares) as a single partial.  One warp per row; reads 4 B, writes 2 B per element.
__global__ void __launch_bounds__(256, 5)
row_stats_kernel(const float* __restrict__ x, long long in_stride, __nv_bfloat16* __restrict__ y,
                 long long out_stride, float2* __restrict__ part, int rows, int D, int descending) {
  int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (warp >= rows) return;
  if (descending) warp = rows - 1 - warp;
  const float* xr = x + static_cast<long long>(warp) * in_stride;
  __nv_bfloat16* yr = y + static_cast<long long>(warp) * out_stride;
  const int nvec = D >> 2;
  float s = 0.f, q = 0.f;
#pragma unroll
  for (int j = 0; j < kLnMaxVec; ++j) {
    const int i = lane + 32 * j;
    if (i < nvec) {
      const float4 v = *reinterpret_cast<const float4*>(xr + 4 * i);
      s += (v.x + v.y) + (v.z + v.w);
      q += (v.x * v.x + v.y * v.y) + (v.z * v.z + v.w * v.w);
      store4(yr + 4 * i, v.x, v.y, v.z, v.w);
    }
  }
  s = warp_sum(s);
  q = warp_sum(q);
  if (lane == 0) part[warp] = make_float2(s, q);
}

// Weights of Linear(LayerNorm(.)) for the folded form: one warp per output feature n.
//   w_out[n,k] = bf16(W[n,k] * gamma[k] - m_n),  m_n = mean_k(W[n,k] * gamma[k]): the row is
//   centred, so sum_k x[k] w_out[n,k] = sum_k (x[k] - mean(x)) gamma[k] W[n,k] up to
//   mean(x) * rowsum[n], where rowsum[n] = sum_k float(w_out[n,k]) is what bf16 rounding leaves
//   of the row sum (~1e-3 for ViT weights; returned for inspection);
//   bias_out[n] = b[n] + sum_k W[n,k] * beta[k].
__global__ void __launch_bounds__(256)
ln_fold_kernel(const float* __restrict__ W, const float* __restrict__ gamma,
               const float* __restrict__ beta, const float* __restrict__ b,
               __nv_bfloat16* __restrict__ w_out, float* __restrict__ rowsum,
               float* __restrict__ bias_out, int N, int K) {
  const int n = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (n >= N) return;
  const float* wr = W + static_cast<long long>(n) * K;
  __nv_bfloat16* wo = w_out + static_cast<long long>(n) * K;
  float t = 0.f, c = 0.f;
  for (int k = lane; k < K; k += 32) {
    const float w = wr[k];
    t = fmaf(w, gamma[k], t);
    c = fmaf(w, beta[k], c);
  }
  const float m = warp_sum(t) / static_cast<float>(K);
  c = warp_sum(c);
  float s = 0.f;
  for (int k = lane; k < K; k += 32) {
    const __nv_bfloat16 r = __float2bfloat16_rn(fmaf(wr[k], gamma[k], -m));
    wo[k] = r;
    s += __bfloat162float(r);
  }
  s = warp_sum(s);
  if (lane == 0) {
    if (rowsum != nullptr) rowsum[n] = s;
    bias_out[n] = (b != nullptr ? b[n] : 0.f) + c;
  }
}

int grid_for(long long work_items, int block, int max_blocks_per_sm = 8) {
  long long g = (work_items + block - 1) / block;
  const long long cap = static_cast<long long>(sm_count()) * max_blocks_per_sm;
  if (g > cap) g = cap;
  if (g < 1) g = 1;
  return static_cast<int>(g);
}

}  // namespace

int layernorm_fwd(const float* x, long long in_stride, const float* gamma, const float* beta,
                  void* y, int y_is_f32, long long out_stride, float* mean_out, float* rstd_out,
                  int rows, int D, float eps, cudaStream_t stream, float* x_copy) {
  VITK_REQUIRE(x && gamma && beta && y, "layernorm: null operand");
  VITK_REQUIRE(rows > 0, "layernorm: rows must be positive");
  VITK_REQUIRE(D % 4 == 0 && D <= 128 * kLnMaxVec, "layernorm: D=%d unsupported (need D%%4==0, D<=%d)",
               D, 128 * kLnMaxVec);
  VITK_REQUIRE(in_stride % 4 == 0 && out_stride % 4 == 0, "layernorm: strides must be multiples of 4");
  const int block = 256;
  const int grid = (rows + 7) / 8;
  ProfileScope prof(PROF_LN, static_cast<double>(rows) * D * (4.0 + (y_is_f32 ? 4.0 : 2.0)), stream);
  const int descending = sweep_next();
  if (y_is_f32)
    layernorm_fwd_kernel<float><<<grid, block, 0, stream>>>(
        x, in_stride, gamma, beta, static_cast<float*>(y), out_stride, mean_out, rstd_out, x_copy,
        rows, D, eps, descending);
  else
    layernorm_fwd_kernel<__nv_bfloat16><<<grid, block, 0, stream>>>(
        x, in_stride, gamma, beta, static_cast<__nv_bfloat16*>(y), out_stride, mean_out, rstd_out,
        x_copy, rows, D, eps, descending);
  VITK_CHECK_LAUNCH("layernorm_fwd_kernel");
  return VITK_OK;
}

int row_stats(const float* x, long long in_stride, void* y_bf16, long long out_stride, float2* part,
              int rows, int D, cudaStream_t stream) {
  VITK_REQUIRE(x && y_bf16 && part, "row_stats: null operand");
  VITK_REQUIRE(rows > 0 && D % 4 == 0 && D <= 128 * kLnMaxVec,
               "row_stats: need rows > 0, D %% 4 == 0, D <= %d", 128 * kLnMaxVec);
  VITK_REQUIRE(in_stride % 4 == 0 && out_stride % 4 == 0, "row_stats: strides must be multiples of 4");
  ProfileScope prof(PROF_LN, static_cast<double>(rows) * D * 6.0, stream);
  const int descending = sweep_next();
  row_stats_kernel<<<(rows + 7) / 8, 256, 0, stream>>>(
      x, in_stride, static_cast<__nv_bfloat16*>(y_bf16), out_stride, part, rows, D, descending);
  VITK_CHECK_LAUNCH("row_stats_kernel");
  return VITK_OK;
}

int ln_fold(const float* W, const float* gamma, const float* beta, const float* b, void* w_out_bf16,
            float* colsum, float* bias_out, int N, int K, cudaStream_t stream) {
  VITK_REQUIRE(W && gamma && beta && w_out_bf16 && bias_out, "ln_fold: null operand");
  VITK_REQUIRE(N > 0 && K > 0, "ln_fold: empty matrix");
  ln_fold_kernel<<<(N + 7) / 8, 256, 0, stream>>>(W, gamma, beta, b,
                                                  static_cast<__nv_bfloat16*>(w_out_bf16), colsum,
                                                  bias_out, N, K);
  VITK_CHECK_LAUNCH("ln_fold_kernel");
  return VITK_OK;
}

int patchify(const float* img, void* out_bf16, int B, int C, int S, int p, cudaStream_t stream) {
  VITK_REQUIRE(img && out_bf16, "patchify: null operand");
  VITK_REQUIRE(B > 0 && C > 0 && S > 0 && p > 0, "patchify: bad shape");
  VITK_REQUIRE(S % p == 0 && p % 8 == 0, "patchify: need image %% patch == 0 and patch %% 8 == 0");
  const long long work = static_cast<long long>(B) * C * S * (S / 8);
  ProfileScope prof(PROF_PATCH, static_cast<double>(B) * C * S * S * 6.0, stream);
  patchify_kernel<<<grid_for(work, 256, 16), 256, 0, stream>>>(
      img, static_cast<__nv_bfloat16*>(out_bf16), B, C, S, p);
  VITK_CHECK_LAUNCH("patchify_kernel");
  return VITK_OK;
}

int patchify_u8(const unsigned char* img_hwc, void* out_bf16, int B, int S, int p, const float* mean,
                const float* stddev, cudaStream_t stream) {
  VITK_REQUIRE(img_hwc && out_bf16 && mean && stddev, "patchify_u8: null operand");
  VITK_REQUIRE(B > 0 && S > 0 && p > 0 && S % p == 0 && p % 8 == 0,
               "patchify_u8: need image %% patch == 0 and patch %% 8 == 0");
  VITK_REQUIRE((reinterpret_cast<uintptr_t>(img_hwc) & 7) == 0, "patchify_u8: images must be 8-byte aligned");
  const long long work = static_cast<long long>(B) * S * (S / 8);
  ProfileScope prof(PROF_PATCH, static_cast<double>(B) * 3 * S * S * 3.0, stream);
  patchify_u8_kernel<<<grid_for(work, 256, 16), 256, 0, stream>>>(
      img_hwc, static_cast<__nv_bfloat16*>(out_bf16), B, S, p, mean[0], mean[1], mean[2], stddev[0],
      stddev[1], stddev[2]);
  VITK_CHECK_LAUNCH("patchify_u8_kernel");
  return VITK_OK;
}

// post_process_predictions (evaluation.py:403-404): class_probs = softmax(logits, -1);
// max_probs, predicted = max(class_probs[:, :-1]) (the last class is "background" for the detector;
// the 6-class classifier keeps all).  One warp per row; scores / labels leave as f32 / i64.
__global__ void __launch_bounds__(256)
postprocess_scores_kernel(const float* __restrict__ logits, int rows, int C, int exclude_last,
                          float* __restrict__ scores, long long* __restrict__ labels,
                          float* __restrict__ probs) {
  const int row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  const float* lr = logits + static_cast<long long>(row) * C;
  float m = -INFINITY;
  for (int c = lane; c < C; c += 32) m = fmaxf(m, lr[c]);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  float sum = 0.f;
  for (int c = lane; c < C; c += 32) sum += __expf(lr[c] - m);
  sum = warp_sum(sum);
  const int Cc = exclude_last ? C - 1 : C;
  float best = -1.f;
  int arg = 0;
  for (int c = lane; c < C; c += 32) {
    const float pr = __expf(lr[c] - m) / sum;
    if (probs != nullptr) probs[static_cast<long long>(row) * C + c] = pr;
    if (c < Cc && pr > best) {
      best = pr;
      arg = c;
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float ob = __shfl_xor_sync(0xffffffffu, best, o);
    const int oa = __shfl_xor_sync(0xffffffffu, arg, o);
    if (ob > best || (ob == best && oa < arg)) {   // first maximum wins, as torch.max does
      best = ob;
      arg = oa;
    }
  }
  if (lane == 0) {
    if (scores != nullptr) scores[row] = best;
    if (labels != nullptr) labels[row] = arg;
  }
}

// post_process_predictions (evaluation.py:393-426) for a whole batch in one launch: per query
// softmax -> best non-background class (as above), `max_probs > confidence_threshold`, and the
// boolean-mask compaction `bbox_coords[confident_mask]` etc. - kept queries of image b move to the
// front of row b of the outputs in query order, counts[b] says how many.  One block per image.
constexpr int kDetMaxQueries = 1024;

__global__ void __launch_bounds__(128)
postprocess_detections_kernel(const float* __restrict__ logits, const float* __restrict__ boxes,
                              int Q, int C, float threshold, int* __restrict__ counts,
                              float* __restrict__ boxes_out, long long* __restrict__ labels_out,
                              float* __restrict__ scores_out) {
  __shared__ float s_score[kDetMaxQueries];
  __shared__ int s_label[kDetMaxQueries];
  __shared__ int s_pos[kDetMaxQueries];  // output slot, or -1 when the query is filtered out
  const int b = blockIdx.x;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int qi = warp; qi < Q; qi += 4) {
    const float* lr = logits + (static_cast<long long>(b) * Q + qi) * C;
    float m = -INFINITY;
    for (int c = lane; c < C; c += 32) m = fmaxf(m, lr[c]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    float sum = 0.f;
    for (int c = lane; c < C; c += 32) sum += __expf(lr[c] - m);
    sum = warp_sum(sum);
    float best = -1.f;
    int arg = 0;
    for (int c = lane; c < C - 1; c += 32) {
      const float pr = __expf(lr[c] - m) / sum;
      if (pr > best) {
        best = pr;
        arg = c;
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float ob = __shfl_xor_sync(0xffffffffu, best, o);
      const int oa = __shfl_xor_sync(0xffffffffu, arg, o);
      if (ob > best || (ob == best && oa < arg)) {
        best = ob;
        arg = oa;
      }
    }
    if (lane == 0) {
      s_score[qi] = best;
      s_label[qi] = arg;
    }
  }
  __syncthreads();
  if (warp == 0) {
    int base = 0;
    for (int q0 = 0; q0 < Q; q0 += 32) {
      const int qi = q0 + lane;
      const bool keep = qi < Q && s_score[qi] > threshold;
      const unsigned bal = __ballot_sync(0xffffffffu, keep);
      if (qi < Q) s_pos[qi] = keep ? base + __popc(bal & ((1u << lane) - 1u)) : -1;
      base += __popc(bal);
    }
    if (lane == 0) counts[b] = base;
  }
  __syncthreads();
  for (int qi = threadIdx.x; qi < Q; qi += blockDim.x) {
    const int pos = s_pos[qi];
    if (pos >= 0) {
      const long long o = static_cast<long long>(b) * Q + pos;
      scores_out[o] = s_score[qi];
      labels_out[o] = s_label[qi];
      reinterpret_cast<float4*>(boxes_out)[o] =
          reinterpret_cast<const float4*>(boxes)[static_cast<long long>(b) * Q + qi];
    }
  }
}

int postprocess_detections(const float* logits, const float* boxes, int batch, int Q, int C,
                           float threshold, int* counts, float* boxes_out, long long* labels_out,
                           float* scores_out, cudaStream_t stream) {
  VITK_REQUIRE(logits && boxes && counts && boxes_out && labels_out && scores_out,
               "postprocess_detections: null operand");
  VITK_REQUIRE(batch > 0 && Q > 0 && Q <= kDetMaxQueries && C > 1,
               "postprocess_detections: need batch > 0, 1 <= queries <= %d, classes + background > 1",
               kDetMaxQueries);
  VITK_REQUIRE(((reinterpret_cast<uintptr_t>(boxes) | reinterpret_cast<uintptr_t>(boxes_out)) & 15) == 0,
               "postprocess_detections: boxes must be 16-byte aligned");
  postprocess_detections_kernel<<<batch, 128, 0, stream>>>(logits, boxes, Q, C, threshold, counts,
                                                           boxes_out, labels_out, scores_out);
  VITK_CHECK_LAUNCH("postprocess_detections_kernel");
  return VITK_OK;
}

int postprocess_scores(const float* logits, int rows, int C, int exclude_last, float* scores,
                       long long* labels, float* probs, cudaStream_t stream) {
  VITK_REQUIRE(logits && rows > 0 && C > (exclude_last ? 1 : 0), "postprocess_scores: bad argument");
  postprocess_scores_kernel<<<(rows + 7) / 8, 256, 0, stream>>>(logits, rows, C, exclude_last, scores,
                                                                labels, probs);
  VITK_CHECK_LAUNCH("postprocess_scores_kernel");
  return VITK_OK;
}

// Linear(D, n_out) on a few fp32 rows (+ optional L2 normalisation of each output row): the CLS
// consumers of the reference - `triplet_projection` + F.normalize (train.py:833-838).  One block
// per row; the row is staged in shared memory, each warp owns every 8th output.
__global__ void __launch_bounds__(256)
linear_rows_kernel(const float* __restrict__ x, long long row_stride, const float* __restrict__ w,
                   const float* __restrict__ b, float* __restrict__ out, int D, int n_out,
                   int l2_normalize) {
  extern __shared__ float s_lin[];  // D inputs, then n_out outputs, then 8 partial sums
  float* s_x = s_lin;
  float* s_y = s_lin + D;
  float* s_part = s_y + n_out;
  const int row = blockIdx.x;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const float* xr = x + static_cast<long long>(row) * row_stride;
  for (int i = threadIdx.x; i < D; i += blockDim.x) s_x[i] = xr[i];
  __syncthreads();
  for (int o = warp; o < n_out; o += 8) {
    const float* wr = w + static_cast<long long>(o) * D;
    float acc = 0.f;
    for (int i = lane; i < D; i += 32) acc = fmaf(s_x[i], __ldg(wr + i), acc);
    acc = warp_sum(acc);
    if (lane == 0) s_y[o] = acc + (b != nullptr ? b[o] : 0.f);
  }
  __syncthreads();
  float scale = 1.f;
  if (l2_normalize) {
    float sq = 0.f;
    for (int o = threadIdx.x; o < n_out; o += blockDim.x) sq += s_y[o] * s_y[o];
    sq = warp_sum(sq);
    if (lane == 0) s_part[warp] = sq;
    __syncthreads();
    float tot = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) tot += s_part[i];
    scale = 1.f / fmaxf(sqrtf(tot), 1e-12f);  // F.normalize: x / max(||x||, eps)
  }
  for (int o = threadIdx.x; o < n_out; o += blockDim.x)
    out[static_cast<long long>(row) * n_out + o] = s_y[o] * scale;
}

int linear_rows(const float* x, long long row_stride, const float* w, const float* b, float* out,
                int rows, int D, int n_out, int l2_normalize, cudaStream_t stream) {
  VITK_REQUIRE(x && w && out, "linear_rows: null operand");
  VITK_REQUIRE(rows > 0 && D > 0 && n_out > 0 && D + n_out <= 11000,
               "linear_rows: bad shape rows=%d D=%d n_out=%d", rows, D, n_out);
  linear_rows_kernel<<<rows, 256, (D + n_out + 8) * sizeof(float), stream>>>(
      x, row_stride, w, b, out, D, n_out, l2_normalize);
  VITK_CHECK_LAUNCH("linear_rows_kernel");
  return VITK_OK;
}

// Backward of out = x W^T + b on a few rows (the head on the CLS rows under the autograd bridge,
// train.py:833-838,1455): thread = input feature k; dx[r,k] = sum_o dy[r,o] W[o,k],
// dW[o,k] = sum_r dy[r,o] x[r,k], db[o] = sum_r dy[r,o].  dy is staged in shared memory.
__global__ void __launch_bounds__(128)
linear_rows_bwd_kernel(const float* __restrict__ x, long long row_stride,
                       const float* __restrict__ w, const float* __restrict__ dy,
                       float* __restrict__ dx, float* __restrict__ dw, float* __restrict__ db,
                       int rows, int D, int n_out) {
  extern __shared__ float s_dy[];  // [rows, n_out]
  for (int i = threadIdx.x; i < rows * n_out; i += blockDim.x) s_dy[i] = dy[i];
  __syncthreads();
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (blockIdx.x == 0 && db != nullptr)
    for (int o = threadIdx.x; o < n_out; o += blockDim.x) {
      float acc = 0.f;
      for (int r = 0; r < rows; ++r) acc += s_dy[r * n_out + o];
      db[o] = acc;
    }
  if (k >= D) return;
  if (dx != nullptr)
    for (int r = 0; r < rows; ++r) {
      float acc = 0.f;
      for (int o = 0; o < n_out; ++o) acc = fmaf(s_dy[r * n_out + o], __ldg(w + (long long)o * D + k), acc);
      dx[static_cast<long long>(r) * D + k] = acc;
    }
  if (dw != nullptr)
    for (int o = 0; o < n_out; ++o) {
      float acc = 0.f;
      for (int r = 0; r < rows; ++r)
        acc = fmaf(s_dy[r * n_out + o], __ldg(x + static_cast<long long>(r) * row_stride + k), acc);
      dw[static_cast<long long>(o) * D + k] = acc;
    }
}

int linear_rows_bwd(const float* x, long long row_stride, const float* w, const float* dy,
                    float* dx, float* dw, float* db, int rows, int D, int n_out,
                    cudaStream_t stream) {
  VITK_REQUIRE(x && w && dy, "linear_rows_bwd: null operand");
  VITK_REQUIRE(rows > 0 && D > 0 && n_out > 0 && static_cast<long long>(rows) * n_out <= 48 * 1024,
               "linear_rows_bwd: rows * n_out = %d * %d exceeds the staged 48 K values", rows, n_out);
  const size_t smem = static_cast<size_t>(rows) * n_out * sizeof(float);
  if (smem > 48 * 1024)
    VITK_TRY(opt_in_smem<linear_rows_bwd_kernel>(192 * 1024, "linear_rows_bwd_kernel"));
  linear_rows_bwd_kernel<<<(D + 127) / 128, 128, smem, stream>>>(x, row_stride, w, dy, dx, dw, db,
                                                                 rows, D, n_out);
  VITK_CHECK_LAUNCH("linear_rows_bwd_kernel");
  return VITK_OK;
}

int prefix_tokens(float* x, const float* cls, const float* dist, const float* pos, int B, int Ntok,
                  int D, int n_prefix, cudaStream_t stream) {
  VITK_REQUIRE(x && cls && pos, "prefix_tokens: null operand");
  VITK_REQUIRE(n_prefix == 1 || (n_prefix == 2 && dist), "prefix_tokens: n_prefix must be 1 or 2");
  VITK_REQUIRE(D % 4 == 0, "prefix_tokens: D %% 4 != 0");
  const long long work = static_cast<long long>(B) * n_prefix * (D / 4);
  prefix_tokens_kernel<<<grid_for(work, 256), 256, 0, stream>>>(x, cls, dist, pos, B, Ntok, D,
                                                                n_prefix);
  VITK_CHECK_LAUNCH("prefix_tokens_kernel");
  return VITK_OK;
}

int cls_head(const float* x, long long row_stride, const float* gamma, const float* beta,
             const float* head_w, const float* head_b, float* feat_out, float* logits, int B, int D,
             int n_classes, float eps, cudaStream_t stream) {
  VITK_REQUIRE(x && gamma && beta && head_w && head_b && logits, "cls_head: null operand");
  VITK_REQUIRE(B > 0 && D > 0 && n_classes > 0, "cls_head: bad shape");
  cls_head_kernel<<<B, 128, (D + 8) * sizeof(float), stream>>>(x, row_stride, gamma, beta, head_w,
                                                               head_b, feat_out, logits, D,
                                                               n_classes, eps);
  VITK_CHECK_LAUNCH("cls_head_kernel");
  return VITK_OK;
}

int cast_f32_to_bf16(const float* in, void* out, long long n, cudaStream_t stream) {
  VITK_REQUIRE(in && out && n > 0, "cast: bad argument");
  VITK_REQUIRE((reinterpret_cast<uintptr_t>(in) & 15) == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0,
               "cast: pointers must be 16-byte aligned");
  cast_f32_bf16_kernel<<<grid_for(n / 8 + 1, 256), 256, 0, stream>>>(
      in, static_cast<__nv_bfloat16*>(out), n);
  VITK_CHECK_LAUNCH("cast_f32_bf16_kernel");
  return VITK_OK;
}

}  // namespace vitk
