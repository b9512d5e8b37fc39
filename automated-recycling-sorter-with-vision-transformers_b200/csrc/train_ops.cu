// Row / elementwise kernels of the training step (reference train.py:1441-1460): LayerNorm
// backward, bias-gradient column sums, cross-entropy + classifier-head backward on the CLS rows,
// token/position-embedding gradients, weight transposes and the fused multi-tensor AdamW of
// train.py:1598-1602.  All HBM-bound: vectorised 8/16-byte accesses, warp-per-row reductions,
// shared-memory partials before global atomics.
#include "train_ops.cuh"

#include <cuda_bf16.h>

#include "common.h"
#include "ptx.cuh"

namespace vitk {
using namespace ptx;

namespace {

constexpr int kLnMaxVec = 8;  // D <= 1024

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

__device__ __forceinline__ float4 load4(const float* p) { return *reinterpret_cast<const float4*>(p); }
__device__ __forceinline__ float4 load4(const __nv_bfloat16* p) {
  const uint2 u = *reinterpret_cast<const uint2*>(p);
  return make_float4(bf16lo_to_f32(u.x), bf16hi_to_f32(u.x), bf16lo_to_f32(u.y), bf16hi_to_f32(u.y));
}

int grid_for(long long work_items, int block, int max_blocks_per_sm = 8) {
  long long g = (work_items + block - 1) / block;
  const long long cap = static_cast<long long>(sm_count()) * max_blocks_per_sm;
  if (g > cap) g = cap;
  if (g < 1) g = 1;
  return static_cast<int>(g);
}

// ------------------------------------------------------------------------------------------------
// LayerNorm backward.  y = (x - mean) * rstd * gamma + beta  (reference nn.LayerNorm, train.py:581).
//   dx = rstd * (g - mean_D(g) - xhat * mean_D(g * xhat)),  g = dy * gamma
//   dgamma += sum_rows dy * xhat ;  dbeta += sum_rows dy
// dx_io: if add_resid, the residual-stream gradient already stored there is added (pre-LN block:
// x feeds both the LN and the skip connection).  Optionally emits a bf16 copy of the result (the
// A operand of the next dgrad GEMM).
// ------------------------------------------------------------------------------------------------
// dy row fragments are kept in their storage type between the passes (bf16: 2 registers per 4
// elements) to stay within the register budget of 3 resident CTAs per SM.
template <typename T> struct RawVec;
template <> struct RawVec<float> {
  using type = float4;
  static __device__ __forceinline__ type load(const float* p) { return *reinterpret_cast<const float4*>(p); }
  static __device__ __forceinline__ float4 f4(const type& v) { return v; }
};
template <> struct RawVec<__nv_bfloat16> {
  using type = uint2;
  static __device__ __forceinline__ type load(const __nv_bfloat16* p) { return *reinterpret_cast<const uint2*>(p); }
  static __device__ __forceinline__ float4 f4(const type& u) {
    return make_float4(bf16lo_to_f32(u.x), bf16hi_to_f32(u.x), bf16lo_to_f32(u.y), bf16hi_to_f32(u.y));
  }
};

// Kernel A: dx (warp per row). Only the raw row (x, dy) stays in registers between the two
// passes - NVEC float4 each - so that 4 CTAs of 256 threads are resident per SM; gamma is
// re-read from L1.  The residual-gradient row is requested before the reductions so that its
// DRAM round trip overlaps them.
template <typename DyT, int NVEC>
__global__ void __launch_bounds__(256, 3)
layernorm_bwd_dx_kernel(const DyT* __restrict__ dy, long long dy_stride, const float* __restrict__ x,
                        long long x_stride, const float* __restrict__ mean,
                        const float* __restrict__ rstd, const float* __restrict__ gamma,
                        float* __restrict__ dx_io, long long dx_stride, int add_resid,
                        __nv_bfloat16* __restrict__ dx_bf16, long long dxb_stride, int rows, int D) {
  const int nvec = D >> 2;
  const int lane = threadIdx.x & 31;
  const long long r = (static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  if (r >= rows) return;
  const float mu = mean[r], rs = rstd[r];
  const float inv_d = 1.f / static_cast<float>(D);
  using RV = RawVec<DyT>;
  float4 xv[NVEC], pv[NVEC];
  typename RV::type dr[NVEC];
  float s1 = 0.f, s2 = 0.f;
#pragma unroll
  for (int j = 0; j < NVEC; ++j) {
    const int i = lane + 32 * j;
    if (i < nvec) {
      xv[j] = load4(x + r * x_stride + 4 * i);
      dr[j] = RV::load(dy + r * dy_stride + 4 * i);
      pv[j] = add_resid ? *reinterpret_cast<const float4*>(dx_io + r * dx_stride + 4 * i)
                        : make_float4(0.f, 0.f, 0.f, 0.f);
    }
  }
#pragma unroll
  for (int j = 0; j < NVEC; ++j) {
    const int i = lane + 32 * j;
    if (i < nvec) {
      const float4 gm = __ldg(reinterpret_cast<const float4*>(gamma) + i);
      const float4 dvj = RV::f4(dr[j]);
      const float g0 = dvj.x * gm.x, g1 = dvj.y * gm.y, g2 = dvj.z * gm.z, g3 = dvj.w * gm.w;
      s1 += (g0 + g1) + (g2 + g3);
      s2 += (g0 * (xv[j].x - mu) + g1 * (xv[j].y - mu)) + (g2 * (xv[j].z - mu) + g3 * (xv[j].w - mu));
    }
  }
  s1 = warp_sum(s1) * inv_d;
  s2 = warp_sum(s2) * rs * inv_d;  // mean_D(g * xhat)
#pragma unroll
  for (int j = 0; j < NVEC; ++j) {
    const int i = lane + 32 * j;
    if (i < nvec) {
      const float4 gm = __ldg(reinterpret_cast<const float4*>(gamma) + i);
      const float4 dvj = RV::f4(dr[j]);
      float4 o;
      o.x = rs * (dvj.x * gm.x - s1 - (xv[j].x - mu) * rs * s2) + pv[j].x;
      o.y = rs * (dvj.y * gm.y - s1 - (xv[j].y - mu) * rs * s2) + pv[j].y;
      o.z = rs * (dvj.z * gm.z - s1 - (xv[j].z - mu) * rs * s2) + pv[j].z;
      o.w = rs * (dvj.w * gm.w - s1 - (xv[j].w - mu) * rs * s2) + pv[j].w;
      *reinterpret_cast<float4*>(dx_io + r * dx_stride + 4 * i) = o;
      if (dx_bf16 != nullptr) {
        uint2 pk;
        pk.x = pack_bf16x2(o.x, o.y);
        pk.y = pack_bf16x2(o.z, o.w);
        *reinterpret_cast<uint2*>(dx_bf16 + r * dxb_stride + 4 * i) = pk;
      }
    }
  }
}

// Fused variant: dx AND the parameter gradients in one pass over dy / x (the separate column
// reduction of kernel B re-reads both: +50 % HBM traffic).  Persistent warps walk rows gw, gw + W,
// ... and keep their dgamma / dbeta partial sums for the 4 * NVEC columns of each lane in
// registers; one shared-memory reduction across the 8 warps and one global atomic per column and
// CTA at the end.
template <typename DyT, int NVEC>
__global__ void __launch_bounds__(256, 2)
layernorm_bwd_fused_kernel(const DyT* __restrict__ dy, long long dy_stride,
                           const float* __restrict__ x, long long x_stride,
                           const float* __restrict__ mean, const float* __restrict__ rstd,
                           const float* __restrict__ gamma, float* __restrict__ dx_io,
                           long long dx_stride, int add_resid, __nv_bfloat16* __restrict__ dx_bf16,
                           long long dxb_stride, float* __restrict__ dgamma,
                           float* __restrict__ dbeta, float* __restrict__ dx_colsum, int rows,
                           int D, DropParams drop) {
  // per-warp column buffer: during the row loop it accumulates the column sums of the bf16 result
  // (dx_colsum: the bias gradient of the Linear whose output gradient this is - saves the separate
  // column-sum pass over dx_bf16); afterwards it carries the cross-warp reduction of dgamma / dbeta
  __shared__ float s_red[8][128 * NVEC];
  const int nvec = D >> 2;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const long long gw = static_cast<long long>(blockIdx.x) * 8 + warp;
  const long long W = static_cast<long long>(gridDim.x) * 8;
  const float inv_d = 1.f / static_cast<float>(D);
  using RV = RawVec<DyT>;
  float4 ag[NVEC], ab[NVEC];
#pragma unroll
  for (int j = 0; j < NVEC; ++j) {
    ag[j] = make_float4(0.f, 0.f, 0.f, 0.f);
    ab[j] = make_float4(0.f, 0.f, 0.f, 0.f);
    const int i = lane + 32 * j;
    if (dx_colsum != nullptr && i < nvec)
      *reinterpret_cast<float4*>(&s_red[warp][4 * i]) = make_float4(0.f, 0.f, 0.f, 0.f);
  }
  for (long long r = gw; r < rows; r += W) {
    const float mu = mean[r], rs = rstd[r];
    float4 xv[NVEC], pv[NVEC];
    typename RV::type dr[NVEC];
#pragma unroll
    for (int j = 0; j < NVEC; ++j) {
      const int i = lane + 32 * j;
      if (i < nvec) {
        xv[j] = load4(x + r * x_stride + 4 * i);
        dr[j] = RV::load(dy + r * dy_stride + 4 * i);
        // requested now so that its DRAM round trip overlaps the reductions
        pv[j] = add_resid ? *reinterpret_cast<const float4*>(dx_io + r * dx_stride + 4 * i)
                          : make_float4(0.f, 0.f, 0.f, 0.f);
      }
    }
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int j = 0; j < NVEC; ++j) {
      const int i = lane + 32 * j;
      if (i < nvec) {
        const float4 d = RV::f4(dr[j]);
        // xhat in place of x; dgamma += dy * xhat, dbeta += dy
        xv[j].x = (xv[j].x - mu) * rs;
        xv[j].y = (xv[j].y - mu) * rs;
        xv[j].z = (xv[j].z - mu) * rs;
        xv[j].w = (xv[j].w - mu) * rs;
        ag[j].x = fmaf(d.x, xv[j].x, ag[j].x);
        ag[j].y = fmaf(d.y, xv[j].y, ag[j].y);
        ag[j].z = fmaf(d.z, xv[j].z, ag[j].z);
        ag[j].w = fmaf(d.w, xv[j].w, ag[j].w);
        ab[j].x += d.x;
        ab[j].y += d.y;
        ab[j].z += d.z;
        ab[j].w += d.w;
        const float4 gm = __ldg(reinterpret_cast<const float4*>(gamma) + i);  // L1 resident
        const float g0 = d.x * gm.x, g1 = d.y * gm.y, g2 = d.z * gm.z, g3 = d.w * gm.w;
        s1 += (g0 + g1) + (g2 + g3);
        s2 += (g0 * xv[j].x + g1 * xv[j].y) + (g2 * xv[j].z + g3 * xv[j].w);
      }
    }
    s1 = warp_sum(s1) * inv_d;
    s2 = warp_sum(s2) * inv_d;  // mean_D(g * xhat)
#pragma unroll
    for (int j = 0; j < NVEC; ++j) {
      const int i = lane + 32 * j;
      if (i < nvec) {
        const float4 d = RV::f4(dr[j]);
        const float4 gm = __ldg(reinterpret_cast<const float4*>(gamma) + i);
        float4 o;
        o.x = rs * (d.x * gm.x - s1 - xv[j].x * s2) + pv[j].x;
        o.y = rs * (d.y * gm.y - s1 - xv[j].y * s2) + pv[j].y;
        o.z = rs * (d.z * gm.z - s1 - xv[j].z * s2) + pv[j].z;
        o.w = rs * (d.w * gm.w - s1 - xv[j].w * s2) + pv[j].w;
        *reinterpret_cast<float4*>(dx_io + r * dx_stride + 4 * i) = o;
        if (dx_bf16 != nullptr) {
          // the bf16 copy is the gradient entering the next branch; if that branch's output was
          // dropped in the forward, its mask (element index = row * D + column) is applied here
          float4 ob = o;
          if (drop.thresh != 0u) {
            const uint32_t pair0 = (static_cast<uint32_t>(r) * static_cast<uint32_t>(D) + 4u * i) >> 1;
            const uint32_t b0 = drop_bits(pair0, drop.key), b1 = drop_bits(pair0 + 1u, drop.key);
            ob.x = drop_keep_lo(b0, drop.thresh) ? o.x * drop.scale : 0.f;
            ob.y = drop_keep_hi(b0, drop.thresh) ? o.y * drop.scale : 0.f;
            ob.z = drop_keep_lo(b1, drop.thresh) ? o.z * drop.scale : 0.f;
            ob.w = drop_keep_hi(b1, drop.thresh) ? o.w * drop.scale : 0.f;
          }
          uint2 pk;
          pk.x = pack_bf16x2(ob.x, ob.y);
          pk.y = pack_bf16x2(ob.z, ob.w);
          *reinterpret_cast<uint2*>(dx_bf16 + r * dxb_stride + 4 * i) = pk;
          if (dx_colsum != nullptr) {   // sums of the ROUNDED values, as a pass over dx_bf16 gives
            float4 acc = *reinterpret_cast<float4*>(&s_red[warp][4 * i]);
            acc.x += bf16lo_to_f32(pk.x);
            acc.y += bf16hi_to_f32(pk.x);
            acc.z += bf16lo_to_f32(pk.y);
            acc.w += bf16hi_to_f32(pk.y);
            *reinterpret_cast<float4*>(&s_red[warp][4 * i]) = acc;
          }
        }
      }
    }
  }
  // ---- column sums of the result, then the per-warp partial sums of dgamma and dbeta through the
  //      same buffer
  if (dx_colsum != nullptr) {
    __syncthreads();
    for (int col = threadIdx.x; col < D; col += 256) {
      float acc = 0.f;
#pragma unroll
      for (int w = 0; w < 8; ++w) acc += s_red[w][col];
      atomicAdd(dx_colsum + col, acc);
    }
    __syncthreads();
  }
#pragma unroll
  for (int pass = 0; pass < 2; ++pass) {
#pragma unroll
    for (int j = 0; j < NVEC; ++j) {
      const int i = lane + 32 * j;
      if (i < nvec)
        *reinterpret_cast<float4*>(&s_red[warp][4 * i]) = pass == 0 ? ag[j] : ab[j];
    }
    __syncthreads();
    float* out = pass == 0 ? dgamma : dbeta;
    for (int col = threadIdx.x; col < D; col += 256) {
      float acc = 0.f;
#pragma unroll
      for (int w = 0; w < 8; ++w) acc += s_red[w][col];
      atomicAdd(out + col, acc);
    }
    __syncthreads();
  }
}

// Kernel B: dgamma / dbeta - a column reduction over rows. Thread = 4 columns, block = 64 threads
// (256 columns) x 4 row lanes, each block sweeps `rows_per_block` rows.
template <typename DyT>
__global__ void __launch_bounds__(256)
layernorm_bwd_params_kernel(const DyT* __restrict__ dy, long long dy_stride,
                            const float* __restrict__ x, long long x_stride,
                            const float* __restrict__ mean, const float* __restrict__ rstd,
                            float* __restrict__ dgamma, float* __restrict__ dbeta, int rows, int D,
                            int rows_per_block) {
  __shared__ float4 s_g[4][64], s_b[4][64];
  const int tcol = threadIdx.x & 63, trow = threadIdx.x >> 6;
  const int col = blockIdx.x * 256 + tcol * 4;
  const int r_begin = blockIdx.y * rows_per_block;
  const int r_end = min(rows, r_begin + rows_per_block);
  float4 ag = make_float4(0, 0, 0, 0), ab = make_float4(0, 0, 0, 0);
  if (col < D) {
#pragma unroll 4
    for (int r = r_begin + trow; r < r_end; r += 4) {
      const float mu = __ldg(mean + r), rs = __ldg(rstd + r);
      const float4 xv = load4(x + r * x_stride + col);
      const float4 d = load4(dy + r * dy_stride + col);
      ag.x = fmaf(d.x, (xv.x - mu) * rs, ag.x);
      ag.y = fmaf(d.y, (xv.y - mu) * rs, ag.y);
      ag.z = fmaf(d.z, (xv.z - mu) * rs, ag.z);
      ag.w = fmaf(d.w, (xv.w - mu) * rs, ag.w);
      ab.x += d.x;
      ab.y += d.y;
      ab.z += d.z;
      ab.w += d.w;
    }
  }
  s_g[trow][tcol] = ag;
  s_b[trow][tcol] = ab;
  __syncthreads();
  if (trow == 0 && col < D) {
#pragma unroll
    for (int k = 1; k < 4; ++k) {
      const float4 a = s_g[k][tcol], b = s_b[k][tcol];
      ag.x += a.x; ag.y += a.y; ag.z += a.z; ag.w += a.w;
      ab.x += b.x; ab.y += b.y; ab.z += b.z; ab.w += b.w;
    }
    atomicAdd(dgamma + col + 0, ag.x);
    atomicAdd(dgamma + col + 1, ag.y);
    atomicAdd(dgamma + col + 2, ag.z);
    atomicAdd(dgamma + col + 3, ag.w);
    atomicAdd(dbeta + col + 0, ab.x);
    atomicAdd(dbeta + col + 1, ab.y);
    atomicAdd(dbeta + col + 2, ab.z);
    atomicAdd(dbeta + col + 3, ab.w);
  }
}

// ------------------------------------------------------------------------------------------------
// out[n] += scale * sum_m Y[m, n]  (bias gradients; Y bf16 [M, ld]).  Each thread owns 8 columns.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
colsum_bf16_kernel(const __nv_bfloat16* __restrict__ y, long long ld, int M, int N,
                   float* __restrict__ out, int rows_per_block) {
  __shared__ float s_acc[4][512];
  const int tcol = threadIdx.x & 63;  // 64 threads x 8 columns = 512-column strip
  const int trow = threadIdx.x >> 6;  // 4 row lanes
  const int col0 = blockIdx.x * 512 + tcol * 8;
  const int r_begin = blockIdx.y * rows_per_block;
  const int r_end = min(M, r_begin + rows_per_block);
  float acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  if (col0 < N) {
#pragma unroll 4
    for (int r = r_begin + trow; r < r_end; r += 4) {
      const uint4 u = __ldg(reinterpret_cast<const uint4*>(y + r * ld + col0));
      acc[0] += bf16lo_to_f32(u.x);
      acc[1] += bf16hi_to_f32(u.x);
      acc[2] += bf16lo_to_f32(u.y);
      acc[3] += bf16hi_to_f32(u.y);
      acc[4] += bf16lo_to_f32(u.z);
      acc[5] += bf16hi_to_f32(u.z);
      acc[6] += bf16lo_to_f32(u.w);
      acc[7] += bf16hi_to_f32(u.w);
    }
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) s_acc[trow][tcol * 8 + j] = acc[j];
  __syncthreads();
  for (int c = threadIdx.x; c < 512; c += 256) {
    const int col = blockIdx.x * 512 + c;
    if (col < N) atomicAdd(out + col, s_acc[0][c] + s_acc[1][c] + s_acc[2][c] + s_acc[3][c]);
  }
}

// ------------------------------------------------------------------------------------------------
// Classifier tail, forward + backward in one pass over the CLS rows (north_star's 6-class head on
// features[:,0]; loss = mean cross-entropy, cf. F.cross_entropy):
//   feat = LN_f(x[b, 0]) ; logits = feat W^T + b ; loss += scale * (lse - logit[label])
//   dlogits = scale * (softmax - onehot) ; dfeat = dlogits W ; dx[b, 0] = LN_f backward(dfeat)
// One block per image.  dx must be zero elsewhere (the caller memsets it).
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128)
cls_loss_bwd_kernel(const float* __restrict__ x, long long row_stride, const float* __restrict__ gamma,
                    const float* __restrict__ beta, const float* __restrict__ head_w,
                    const float* __restrict__ head_b, const long long* __restrict__ labels,
                    float scale, float eps, int D, int C, float* __restrict__ logits_out,
                    float* __restrict__ loss_out, float* __restrict__ feat_out,
                    float* __restrict__ dlogits_out, float* __restrict__ dx,
                    __nv_bfloat16* __restrict__ dx_bf16, float* __restrict__ dgamma,
                    float* __restrict__ dbeta) {
  extern __shared__ float sm[];  // xhat[D], feat/dfeat[D], red[8], logit[C], dl[C]
  float* xhat = sm;
  float* feat = sm + D;
  float* red = sm + 2 * D;
  float* logit = red + 8;
  float* dl = logit + C;
  const int b = blockIdx.x;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const float* xr = x + b * row_stride;
  auto block_sum = [&](float v) {
    v = warp_sum(v);
    __syncthreads();
    if (lane == 0) red[warp] = v;
    __syncthreads();
    return red[0] + red[1] + red[2] + red[3];
  };
  float s = 0.f;
  for (int i = tid; i < D; i += 128) {
    xhat[i] = xr[i];
    s += xhat[i];
  }
  const float mean = block_sum(s) / D;
  float sq = 0.f;
  for (int i = tid; i < D; i += 128) {
    const float d = xhat[i] - mean;
    sq += d * d;
  }
  const float rstd = rsqrtf(block_sum(sq) / D + eps);
  for (int i = tid; i < D; i += 128) {
    const float h = (xhat[i] - mean) * rstd;
    xhat[i] = h;
    const float f = h * gamma[i] + beta[i];
    feat[i] = f;
    if (feat_out) feat_out[static_cast<long long>(b) * D + i] = f;
  }
  __syncthreads();
  for (int c = warp; c < C; c += 4) {
    const float* w = head_w + static_cast<long long>(c) * D;
    float acc = 0.f;
    for (int i = lane; i < D; i += 32) acc = fmaf(feat[i], __ldg(w + i), acc);
    acc = warp_sum(acc);
    if (lane == 0) logit[c] = acc + head_b[c];
  }
  __syncthreads();
  if (tid == 0) {
    float m = -INFINITY;
    for (int c = 0; c < C; ++c) m = fmaxf(m, logit[c]);
    float z = 0.f;
    for (int c = 0; c < C; ++c) z += expf(logit[c] - m);
    const float lse = m + logf(z);
    const int lab = static_cast<int>(labels[b]);
    for (int c = 0; c < C; ++c) {
      const float p = expf(logit[c] - lse);
      dl[c] = scale * (p - (c == lab ? 1.f : 0.f));
      if (logits_out) logits_out[static_cast<long long>(b) * C + c] = logit[c];
      if (dlogits_out) dlogits_out[static_cast<long long>(b) * C + c] = dl[c];
    }
    if (loss_out) atomicAdd(loss_out, scale * (lse - logit[lab]));
  }
  __syncthreads();
  // dfeat (reuse feat[]), then LayerNorm backward of the row
  float s1 = 0.f, s2 = 0.f;
  for (int i = tid; i < D; i += 128) {
    float df = 0.f;
    for (int c = 0; c < C; ++c) df = fmaf(dl[c], __ldg(head_w + static_cast<long long>(c) * D + i), df);
    if (dgamma) {
      atomicAdd(dgamma + i, df * xhat[i]);
      atomicAdd(dbeta + i, df);
    }
    const float g = df * gamma[i];
    feat[i] = g;
    s1 += g;
    s2 += g * xhat[i];
  }
  s1 = block_sum(s1) / D;
  s2 = block_sum(s2) / D;
  for (int i = tid; i < D; i += 128) {
    const float o = rstd * (feat[i] - s1 - xhat[i] * s2);
    dx[b * row_stride + i] = o;
    if (dx_bf16) dx_bf16[b * row_stride + i] = __float2bfloat16_rn(o);
  }
}

// dW[c, :] = sum_b dlogits[b, c] * feat[b, :] ; db[c] = sum_b dlogits[b, c].
// Block = (class, 64 feature columns); 4 thread groups split the batch, unrolled so that the loads
// of a group are in flight together (the first version walked the batch serially in 6 blocks:
// 116 us of pure load latency for 0.6 MFLOP).
__global__ void __launch_bounds__(256)
head_wgrad_kernel(const float* __restrict__ dlogits, const float* __restrict__ feat, int B, int D,
                  int C, float* __restrict__ dW, float* __restrict__ db) {
  __shared__ float s_part[4][64];
  __shared__ float s_db[4];
  const int c = blockIdx.x;
  const int col = blockIdx.y * 64 + (threadIdx.x & 63);
  const int g = threadIdx.x >> 6;
  float acc = 0.f, accb = 0.f;
  if (col < D) {
#pragma unroll 8
    for (int b = g; b < B; b += 4) {
      const float dl = __ldg(dlogits + b * C + c);
      acc = fmaf(dl, __ldg(feat + static_cast<long long>(b) * D + col), acc);
      accb += dl;
    }
  }
  s_part[g][threadIdx.x & 63] = acc;
  if ((threadIdx.x & 63) == 0) s_db[g] = accb;
  __syncthreads();
  if (g == 0 && col < D)
    dW[static_cast<long long>(c) * D + col] +=
        (s_part[0][threadIdx.x] + s_part[1][threadIdx.x]) + (s_part[2][threadIdx.x] + s_part[3][threadIdx.x]);
  if (threadIdx.x == 0 && blockIdx.y == 0) db[c] += (s_db[0] + s_db[1]) + (s_db[2] + s_db[3]);
}

// ------------------------------------------------------------------------------------------------
// Token-assembly backward (x = cat(cls[, dist], patches) + pos, evaluation.py:145-149):
//   dpos[t, :] += sum_b dx[b, t, :]   (dcls = dpos[0], ddist = dpos[1] are copied by the caller)
//   dxp[b*P + p, :] = bf16(dx[b, prefix + p, :])   (A operand of the patch-embedding wgrad)
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
token_grads_kernel(const float* __restrict__ dx, int B, int Ntok, int D, int prefix,
                   float* __restrict__ dpos, float* __restrict__ dcls, float* __restrict__ ddist,
                   __nv_bfloat16* __restrict__ dxp) {
  const int nvec = D >> 2;
  const long long total = static_cast<long long>(Ntok) * nvec;
  for (long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; idx < total;
       idx += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int i = static_cast<int>(idx % nvec);
    const int t = static_cast<int>(idx / nvec);
    float4 acc = make_float4(0, 0, 0, 0);
    for (int b = 0; b < B; ++b) {
      const float4 v = *reinterpret_cast<const float4*>(dx + (static_cast<long long>(b) * Ntok + t) * D + 4 * i);
      acc.x += v.x;
      acc.y += v.y;
      acc.z += v.z;
      acc.w += v.w;
      if (t >= prefix && dxp != nullptr) {
        uint2 pk;
        pk.x = pack_bf16x2(v.x, v.y);
        pk.y = pack_bf16x2(v.z, v.w);
        *reinterpret_cast<uint2*>(dxp + (static_cast<long long>(b) * (Ntok - prefix) + (t - prefix)) * D + 4 * i) = pk;
      }
    }
    float* dst = dpos + static_cast<long long>(t) * D + 4 * i;
    float4 p = *reinterpret_cast<float4*>(dst);
    p.x += acc.x;
    p.y += acc.y;
    p.z += acc.z;
    p.w += acc.w;
    *reinterpret_cast<float4*>(dst) = p;
    float* tok = (t == 0) ? dcls : ((t == 1 && prefix == 2) ? ddist : nullptr);
    if (tok != nullptr) {  // x[b, t] = token + pos[t]  ->  same gradient as pos[t]
      float4 q = *reinterpret_cast<float4*>(tok + 4 * i);
      q.x += acc.x;
      q.y += acc.y;
      q.z += acc.z;
      q.w += acc.w;
      *reinterpret_cast<float4*>(tok + 4 * i) = q;
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Batched bf16 transposes (W [R, C] -> W^T [C, R]): the dgrad GEMMs consume nn.Linear weights as
// K-major operands with the roles of the two dimensions swapped.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
transpose_batched_kernel(const TransposeBatch tb) {
  __shared__ __nv_bfloat16 tile[64][66];
  int job = 0;
  int t = blockIdx.x;
  while (job < tb.n && t >= tb.tiles[job]) {
    t -= tb.tiles[job];
    ++job;
  }
  if (job >= tb.n) return;
  const int R = tb.rows[job], Cc = tb.cols[job];
  const __nv_bfloat16* src = static_cast<const __nv_bfloat16*>(tb.src[job]);
  __nv_bfloat16* dst = static_cast<__nv_bfloat16*>(tb.dst[job]);
  const int tiles_c = (Cc + 63) / 64;
  const int r0 = (t / tiles_c) * 64, c0 = (t % tiles_c) * 64;
  // full tiles of 16-byte aligned matrices (every Linear weight of the models): 16-byte global
  // accesses on both sides, eight elements per thread (206 -> ~90 us for the 85 M weights of
  // ViT-B/16: the 2-byte form kept too few bytes in flight)
  const bool vec = (R % 8 == 0) && (Cc % 8 == 0) && r0 + 64 <= R && c0 + 64 <= Cc &&
                   (reinterpret_cast<uintptr_t>(src) & 15) == 0 &&
                   (reinterpret_cast<uintptr_t>(dst) & 15) == 0;
  if (vec) {
    for (int v = threadIdx.x; v < 512; v += 256) {
      const int r = v >> 3, cv = v & 7;
      const uint4 q = __ldg(reinterpret_cast<const uint4*>(
          src + static_cast<long long>(r0 + r) * Cc + c0 + cv * 8));
      uint32_t* t32 = reinterpret_cast<uint32_t*>(&tile[r][cv * 8]);   // rows are 4-byte aligned
      t32[0] = q.x;
      t32[1] = q.y;
      t32[2] = q.z;
      t32[3] = q.w;
    }
    __syncthreads();
    for (int v = threadIdx.x; v < 512; v += 256) {
      const int c = v >> 3, rv = v & 7;
      const unsigned short* col = reinterpret_cast<const unsigned short*>(&tile[rv * 8][c]);
      uint32_t w[4];
#pragma unroll
      for (int k = 0; k < 4; ++k)
        w[k] = static_cast<uint32_t>(col[(2 * k) * 66]) |
               (static_cast<uint32_t>(col[(2 * k + 1) * 66]) << 16);
      *reinterpret_cast<uint4*>(dst + static_cast<long long>(c0 + c) * R + r0 + rv * 8) =
          make_uint4(w[0], w[1], w[2], w[3]);
    }
    return;
  }
  const int tx = threadIdx.x & 63, ty = threadIdx.x >> 6;
  for (int r = ty; r < 64; r += 4)
    if (r0 + r < R && c0 + tx < Cc) tile[r][tx] = src[static_cast<long long>(r0 + r) * Cc + c0 + tx];
  __syncthreads();
  for (int c = ty; c < 64; c += 4)
    if (c0 + c < Cc && r0 + tx < R) dst[static_cast<long long>(c0 + c) * R + r0 + tx] = tile[tx][c];
}

// ------------------------------------------------------------------------------------------------
// Fused AdamW over one flat parameter arena (train.py:1598-1602: one group, decoupled weight decay
// on EVERY parameter, betas (0.9, 0.999), eps 1e-8; update rule of torch.optim.AdamW):
//   p *= 1 - lr*wd ; m = b1 m + (1-b1) g ; v = b2 v + (1-b2) g^2
//   p -= (lr / bc1) * m / (sqrt(v) / sqrt(bc2) + eps)
// One launch for all 85.8 M parameters; also refreshes the bf16 shadow the GEMMs read.
// Traffic: 16 B read + 12 B write (+2 B shadow) per parameter.
// ------------------------------------------------------------------------------------------------
// guard (optional): {non-finite flag of this step's gradients, steps skipped so far}.  With the flag
// set the launch does nothing - the reference's `scaler.step(optimizer)` skips the optimizer step
// when a gradient is inf / nan (train.py:1456, 1615) - and skipped steps do not advance Adam's
// step counter, so the bias corrections are evaluated here, per block, for step - skipped.
__global__ void __launch_bounds__(256)
adamw_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
             float* __restrict__ v, __nv_bfloat16* __restrict__ shadow, long long n, float decay,
             float b1, float b2, float omb1, float omb2, float step_size, float inv_sqrt_bc2,
             float eps, float grad_scale, const int* __restrict__ guard, double lr, double beta1,
             double beta2, int step) {
  if (guard != nullptr) {
    if (guard[0] != 0) return;
    const int skipped = guard[1];
    if (skipped != 0) {   // uniform across the grid; the common case keeps the host's constants
      __shared__ float s_fix[2];
      if (threadIdx.x == 0) {
        const int t = step - skipped;
        s_fix[0] = static_cast<float>(lr / (1.0 - pow(beta1, static_cast<double>(t))));
        s_fix[1] = static_cast<float>(1.0 / sqrt(1.0 - pow(beta2, static_cast<double>(t))));
      }
      __syncthreads();
      step_size = s_fix[0];
      inv_sqrt_bc2 = s_fix[1];
    }
  }
  const long long nvec = n >> 2;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < nvec;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    float4 pv = reinterpret_cast<float4*>(p)[i];
    const float4 gv = reinterpret_cast<const float4*>(g)[i];
    float4 mv = reinterpret_cast<float4*>(m)[i];
    float4 vv = reinterpret_cast<float4*>(v)[i];
    float* pp = reinterpret_cast<float*>(&pv);
    const float* gp = reinterpret_cast<const float*>(&gv);
    float* mp = reinterpret_cast<float*>(&mv);
    float* vp = reinterpret_cast<float*>(&vv);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const float gr = gp[k] * grad_scale;
      pp[k] *= decay;
      mp[k] = b1 * mp[k] + omb1 * gr;
      vp[k] = b2 * vp[k] + omb2 * gr * gr;
      const float denom = sqrtf(vp[k]) * inv_sqrt_bc2 + eps;
      pp[k] -= step_size * (mp[k] / denom);
    }
    reinterpret_cast<float4*>(p)[i] = pv;
    reinterpret_cast<float4*>(m)[i] = mv;
    reinterpret_cast<float4*>(v)[i] = vv;
    if (shadow != nullptr) {
      uint2 pk;
      pk.x = pack_bf16x2(pv.x, pv.y);
      pk.y = pack_bf16x2(pv.z, pv.w);
      reinterpret_cast<uint2*>(shadow)[i] = pk;
    }
  }
  // tail (n not a multiple of 4)
  for (long long i = (nvec << 2) + blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
       i < n; i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const float gr = g[i] * grad_scale;
    float pv = p[i] * decay;
    const float mv = b1 * m[i] + omb1 * gr;
    const float vv = b2 * v[i] + omb2 * gr * gr;
    pv -= step_size * (mv / (sqrtf(vv) * inv_sqrt_bc2 + eps));
    p[i] = pv;
    m[i] = mv;
    v[i] = vv;
    if (shadow != nullptr) shadow[i] = __float2bfloat16_rn(pv);
  }
}

// ------------------------------------------------------------------------------------------------
// Stand-alone dropout passes (thread = one element pair = one hash).
// ------------------------------------------------------------------------------------------------
template <int MODE>  // 0: f32 in place, 1: f32 -> bf16, 2: keep mask bytes
__global__ void __launch_bounds__(256)
dropout_kernel(float* __restrict__ x, __nv_bfloat16* __restrict__ out_bf16,
               unsigned char* __restrict__ out_mask, long long n_pairs, DropParams d) {
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n_pairs;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const uint32_t bits = drop_bits(static_cast<uint32_t>(i), d.key);
    const bool k0 = d.thresh == 0u || drop_keep_lo(bits, d.thresh);
    const bool k1 = d.thresh == 0u || drop_keep_hi(bits, d.thresh);
    if constexpr (MODE == 2) {
      out_mask[2 * i] = k0 ? 1 : 0;
      out_mask[2 * i + 1] = k1 ? 1 : 0;
    } else {
      const float2 v = reinterpret_cast<const float2*>(x)[i];
      const float a = k0 ? v.x * d.scale : 0.f, b = k1 ? v.y * d.scale : 0.f;
      if constexpr (MODE == 0) reinterpret_cast<float2*>(x)[i] = make_float2(a, b);
      else reinterpret_cast<uint32_t*>(out_bf16)[i] = pack_bf16x2(a, b);
    }
  }
}

// SetCriterion.loss_labels (train.py:1220-1239): F.cross_entropy(logits, targets, weight) = the
// weighted mean  sum_i w[t_i] nll_i / sum_i w[t_i].  Pass 1: thread = row, log-sum-exp over the few
// classes, block-reduced (sum w nll, sum w) -> two atomics per block.  Pass 2: loss and
// dlogits[i, c] = grad_scale * w[t_i] (softmax_ic - [c == t_i]) / sum w.
__global__ void __launch_bounds__(256)
wce_sums_kernel(const float* __restrict__ logits, const long long* __restrict__ targets,
                const float* __restrict__ weight, int rows, int C, float* __restrict__ sums) {
  __shared__ float s_red[2][8];
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  float wn = 0.f, ws = 0.f;
  if (r < rows) {
    const float* lr = logits + static_cast<long long>(r) * C;
    float m = -INFINITY;
    for (int c = 0; c < C; ++c) m = fmaxf(m, lr[c]);
    float z = 0.f;
    for (int c = 0; c < C; ++c) z += __expf(lr[c] - m);
    const long long t = targets[r];
    if (t >= 0 && t < C) {   // (F.cross_entropy's ignore_index rows carry no weight)
      const float w = weight != nullptr ? weight[t] : 1.f;
      wn = w * (m + __logf(z) - lr[t]);
      ws = w;
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    wn += __shfl_xor_sync(0xffffffffu, wn, o);
    ws += __shfl_xor_sync(0xffffffffu, ws, o);
  }
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0) {
    s_red[0][warp] = wn;
    s_red[1][warp] = ws;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    float a = 0.f, b = 0.f;
    for (int i = 0; i < 8; ++i) {
      a += s_red[0][i];
      b += s_red[1][i];
    }
    atomicAdd(sums, a);
    atomicAdd(sums + 1, b);
  }
}

__global__ void __launch_bounds__(256)
wce_grad_kernel(const float* __restrict__ logits, const long long* __restrict__ targets,
                const float* __restrict__ weight, int rows, int C, const float* __restrict__ sums,
                float* __restrict__ loss_out, float* __restrict__ dlogits, float grad_scale) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  const float wsum = sums[1];
  if (r == 0 && loss_out != nullptr) *loss_out = sums[0] / wsum;
  if (dlogits == nullptr || r >= rows) return;
  const float* lr = logits + static_cast<long long>(r) * C;
  float* dr = dlogits + static_cast<long long>(r) * C;
  const long long t = targets[r];
  if (t < 0 || t >= C) {
    for (int c = 0; c < C; ++c) dr[c] = 0.f;
    return;
  }
  float m = -INFINITY;
  for (int c = 0; c < C; ++c) m = fmaxf(m, lr[c]);
  float z = 0.f;
  for (int c = 0; c < C; ++c) z += __expf(lr[c] - m);
  const float k = grad_scale * (weight != nullptr ? weight[t] : 1.f) / wsum;
  const float inv_z = 1.f / z;
  for (int c = 0; c < C; ++c) dr[c] = k * (__expf(lr[c] - m) * inv_z - (c == t ? 1.f : 0.f));
}

}  // namespace

int dropout_f32_inplace(float* x, long long n, const DropParams& d, cudaStream_t stream) {
  VITK_REQUIRE(x && n > 0 && n % 2 == 0 && n < (1ll << 32), "dropout: bad argument");
  ProfileScope prof(PROF_OTHER, static_cast<double>(n) * 8.0, stream);
  dropout_kernel<0><<<grid_for(n / 2, 256, 16), 256, 0, stream>>>(x, nullptr, nullptr, n / 2, d);
  VITK_CHECK_LAUNCH("dropout_kernel");
  return VITK_OK;
}
int dropout_cast_bf16(const float* x, void* out_bf16, long long n, const DropParams& d,
                      cudaStream_t stream) {
  VITK_REQUIRE(x && out_bf16 && n > 0 && n % 2 == 0 && n < (1ll << 32), "dropout: bad argument");
  ProfileScope prof(PROF_OTHER, static_cast<double>(n) * 6.0, stream);
  dropout_kernel<1><<<grid_for(n / 2, 256, 16), 256, 0, stream>>>(
      const_cast<float*>(x), static_cast<__nv_bfloat16*>(out_bf16), nullptr, n / 2, d);
  VITK_CHECK_LAUNCH("dropout_kernel");
  return VITK_OK;
}
int dropout_keep_mask(unsigned char* out, long long n, const DropParams& d, cudaStream_t stream) {
  VITK_REQUIRE(out && n > 0 && n % 2 == 0 && n < (1ll << 32), "dropout: bad argument");
  dropout_kernel<2><<<grid_for(n / 2, 256, 16), 256, 0, stream>>>(nullptr, nullptr, out, n / 2, d);
  VITK_CHECK_LAUNCH("dropout_kernel");
  return VITK_OK;
}

int layernorm_bwd(const void* dy, int dy_is_f32, long long dy_stride, const float* x,
                  long long x_stride, const float* mean, const float* rstd, const float* gamma,
                  float* dx_io, long long dx_stride, int add_resid, void* dx_bf16,
                  long long dxb_stride, float* dgamma, float* dbeta, int rows, int D,
                  cudaStream_t stream, float* dx_colsum, const DropParams* drop) {
  VITK_REQUIRE(dy && x && mean && rstd && gamma && dx_io, "layernorm_bwd: null operand");
  const DropParams dp = drop != nullptr ? *drop : DropParams();
  const bool dropping = dp.thresh != 0u;
  VITK_REQUIRE(rows > 0 && D % 4 == 0 && D <= 128 * kLnMaxVec, "layernorm_bwd: bad shape");
  VITK_REQUIRE((dgamma == nullptr) == (dbeta == nullptr), "layernorm_bwd: dgamma/dbeta together");
  const int block = 256;
  const int grid = (rows + 7) / 8;
  const __nv_bfloat16* dyb = static_cast<const __nv_bfloat16*>(dy);
  const float* dyf = static_cast<const float*>(dy);
  const int nv = (D / 4 + 31) / 32;
  VITK_REQUIRE(dx_colsum == nullptr || dx_bf16 != nullptr,
               "layernorm_bwd: dx_colsum needs the bf16 output");
  VITK_REQUIRE(!dropping || (dx_bf16 != nullptr && dxb_stride == D &&
                             static_cast<long long>(rows) * D < (1ll << 32)),
               "layernorm_bwd: the dropout mask applies to a dense bf16 output");
  if (dgamma != nullptr && nv <= 6) {
    // one pass: dx and the parameter gradients together
    ProfileScope prof(PROF_LN, static_cast<double>(rows) * D * (dy_is_f32 ? 14.0 : 12.0), stream);
    int fgrid = sm_count() * 2;
    if (fgrid > (rows + 7) / 8) fgrid = (rows + 7) / 8;
    __nv_bfloat16* dxb = static_cast<__nv_bfloat16*>(dx_bf16);
#define VITK_LN_FUSED(T, PTR, NV)                                                                 \
  layernorm_bwd_fused_kernel<T, NV><<<fgrid, block, 0, stream>>>(                                 \
      PTR, dy_stride, x, x_stride, mean, rstd, gamma, dx_io, dx_stride, add_resid, dxb, dxb_stride, \
      dgamma, dbeta, dx_colsum, rows, D, dp)
    if (dy_is_f32) {
      if (nv <= 2) VITK_LN_FUSED(float, dyf, 2);
      else if (nv <= 4) VITK_LN_FUSED(float, dyf, 4);
      else VITK_LN_FUSED(float, dyf, 6);
    } else {
      if (nv <= 2) VITK_LN_FUSED(__nv_bfloat16, dyb, 2);
      else if (nv <= 4) VITK_LN_FUSED(__nv_bfloat16, dyb, 4);
      else VITK_LN_FUSED(__nv_bfloat16, dyb, 6);
    }
#undef VITK_LN_FUSED
    VITK_CHECK_LAUNCH("layernorm_bwd_fused_kernel");
    return VITK_OK;
  }
  VITK_REQUIRE(!dropping, "layernorm_bwd: dropout needs the fused kernel (parameter gradients, D <= 768)");
  if (dgamma != nullptr) {
    // parameter gradients first: they read dy / x only, before dx_io is updated in place
    const int strips = (D + 255) / 256;
    int chunks = (sm_count() * 6 + strips - 1) / strips;
    if (chunks > (rows + 15) / 16) chunks = (rows + 15) / 16;
    if (chunks < 1) chunks = 1;
    const int rows_per_block = (rows + chunks - 1) / chunks;
    chunks = (rows + rows_per_block - 1) / rows_per_block;
    ProfileScope prof(PROF_LN, static_cast<double>(rows) * D * (dy_is_f32 ? 8.0 : 6.0), stream);
    if (dy_is_f32)
      layernorm_bwd_params_kernel<float><<<dim3(strips, chunks), block, 0, stream>>>(
          dyf, dy_stride, x, x_stride, mean, rstd, dgamma, dbeta, rows, D, rows_per_block);
    else
      layernorm_bwd_params_kernel<__nv_bfloat16><<<dim3(strips, chunks), block, 0, stream>>>(
          dyb, dy_stride, x, x_stride, mean, rstd, dgamma, dbeta, rows, D, rows_per_block);
    VITK_CHECK_LAUNCH("layernorm_bwd_params_kernel");
  }
  ProfileScope prof(PROF_LN, static_cast<double>(rows) * D * (dy_is_f32 ? 14.0 : 12.0), stream);
  __nv_bfloat16* dxb = static_cast<__nv_bfloat16*>(dx_bf16);
#define VITK_LN_BWD(T, PTR, NV)                                                                  \
  layernorm_bwd_dx_kernel<T, NV><<<grid, block, 0, stream>>>(PTR, dy_stride, x, x_stride, mean,  \
                                                             rstd, gamma, dx_io, dx_stride,       \
                                                             add_resid, dxb, dxb_stride, rows, D)
  if (dy_is_f32) {
    if (nv <= 2) VITK_LN_BWD(float, dyf, 2);
    else if (nv <= 4) VITK_LN_BWD(float, dyf, 4);
    else if (nv <= 6) VITK_LN_BWD(float, dyf, 6);
    else VITK_LN_BWD(float, dyf, 8);
  } else {
    if (nv <= 2) VITK_LN_BWD(__nv_bfloat16, dyb, 2);
    else if (nv <= 4) VITK_LN_BWD(__nv_bfloat16, dyb, 4);
    else if (nv <= 6) VITK_LN_BWD(__nv_bfloat16, dyb, 6);
    else VITK_LN_BWD(__nv_bfloat16, dyb, 8);
  }
#undef VITK_LN_BWD
  VITK_CHECK_LAUNCH("layernorm_bwd_dx_kernel");
  if (dx_colsum != nullptr) {
    VITK_REQUIRE(dx_bf16 != nullptr, "layernorm_bwd: dx_colsum needs the bf16 output");
    return colsum_bf16(dx_bf16, dxb_stride, rows, D, dx_colsum, stream);
  }
  return VITK_OK;
}

int colsum_bf16(const void* y, long long ld, int M, int N, float* out, cudaStream_t stream) {
  VITK_REQUIRE(y && out && M > 0 && N > 0 && N % 8 == 0 && ld % 8 == 0, "colsum: bad argument");
  const int strips = (N + 511) / 512;
  int chunks = (sm_count() * 12 + strips - 1) / strips;
  if (chunks > (M + 31) / 32) chunks = (M + 31) / 32;
  if (chunks < 1) chunks = 1;
  const int rows_per_block = (M + chunks - 1) / chunks;
  chunks = (M + rows_per_block - 1) / rows_per_block;
  ProfileScope prof(PROF_OTHER, static_cast<double>(M) * N * 2.0, stream);
  colsum_bf16_kernel<<<dim3(strips, chunks), 256, 0, stream>>>(
      static_cast<const __nv_bfloat16*>(y), ld, M, N, out, rows_per_block);
  VITK_CHECK_LAUNCH("colsum_bf16_kernel");
  return VITK_OK;
}

int cls_loss_bwd(const float* x, long long row_stride, const float* gamma, const float* beta,
                 const float* head_w, const float* head_b, const long long* labels, float scale,
                 float eps, int B, int D, int C, float* logits_out, float* loss_out, float* feat_ws,
                 float* dlogits_ws, float* dx, void* dx_bf16, float* dgamma, float* dbeta,
                 float* dhead_w, float* dhead_b, cudaStream_t stream) {
  VITK_REQUIRE(x && gamma && beta && head_w && head_b && labels && dx && feat_ws && dlogits_ws,
               "cls_loss_bwd: null operand");
  VITK_REQUIRE(B > 0 && D > 0 && C > 0 && C <= 1024, "cls_loss_bwd: bad shape");
  const size_t smem = (2 * static_cast<size_t>(D) + 8 + 2 * C) * sizeof(float);
  cls_loss_bwd_kernel<<<B, 128, smem, stream>>>(x, row_stride, gamma, beta, head_w, head_b, labels,
                                                scale, eps, D, C, logits_out, loss_out, feat_ws,
                                                dlogits_ws, dx,
                                                static_cast<__nv_bfloat16*>(dx_bf16), dgamma, dbeta);
  VITK_CHECK_LAUNCH("cls_loss_bwd_kernel");
  if (dhead_w != nullptr) {
    VITK_REQUIRE(dhead_b != nullptr, "cls_loss_bwd: dhead_b missing");
    head_wgrad_kernel<<<dim3(C, (D + 63) / 64), 256, 0, stream>>>(dlogits_ws, feat_ws, B, D, C,
                                                                  dhead_w, dhead_b);
    VITK_CHECK_LAUNCH("head_wgrad_kernel");
  }
  return VITK_OK;
}

int token_grads(const float* dx, int B, int Ntok, int D, int prefix, float* dpos, float* dcls,
                float* ddist, void* dxp_bf16, cudaStream_t stream) {
  VITK_REQUIRE(dx && dpos && dcls && D % 4 == 0, "token_grads: bad argument");
  VITK_REQUIRE(prefix == 1 || ddist != nullptr, "token_grads: ddist missing");
  const long long work = static_cast<long long>(Ntok) * (D / 4);
  token_grads_kernel<<<grid_for(work, 256), 256, 0, stream>>>(
      dx, B, Ntok, D, prefix, dpos, dcls, ddist, static_cast<__nv_bfloat16*>(dxp_bf16));
  VITK_CHECK_LAUNCH("token_grads_kernel");
  return VITK_OK;
}

int transpose_batched(const TransposeBatch& tb, cudaStream_t stream) {
  VITK_REQUIRE(tb.n > 0 && tb.n <= kMaxTransposeJobs, "transpose: bad job count");
  int total = 0;
  for (int i = 0; i < tb.n; ++i) total += tb.tiles[i];
  transpose_batched_kernel<<<total, 256, 0, stream>>>(tb);
  VITK_CHECK_LAUNCH("transpose_batched_kernel");
  return VITK_OK;
}

// guard[0] |= any(!isfinite(g)); 16-byte loads, one atomic per block that saw one.
__global__ void __launch_bounds__(256)
nonfinite_scan_kernel(const float* __restrict__ g, long long n, int* __restrict__ guard) {
  const long long nvec = n >> 2;
  bool bad = false;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < nvec;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const float4 v = reinterpret_cast<const float4*>(g)[i];
    // x - x is 0 for finite x, nan for inf / nan
    bad |= !(((v.x - v.x) + (v.y - v.y)) + ((v.z - v.z) + (v.w - v.w)) == 0.f);
  }
  for (long long i = (nvec << 2) + blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
       i < n; i += static_cast<long long>(gridDim.x) * blockDim.x)
    bad |= !(g[i] - g[i] == 0.f);
  if (__syncthreads_or(bad) && threadIdx.x == 0) atomicOr(guard, 1);
}

__global__ void guard_finish_kernel(int* guard) {
  if (guard[0] != 0) guard[1] += 1;
}

int grad_guard_scan(const float* g, long long n, int* guard, int reset, cudaStream_t stream) {
  VITK_REQUIRE(g && guard && n > 0, "grad_guard_scan: bad argument");
  VITK_REQUIRE((reinterpret_cast<uintptr_t>(g) & 15) == 0, "grad_guard_scan: 16-byte alignment");
  if (reset) VITK_CHECK_CUDA(cudaMemsetAsync(guard, 0, sizeof(int), stream));
  ProfileScope prof(PROF_OPT, static_cast<double>(n) * 4.0, stream);
  nonfinite_scan_kernel<<<grid_for(n / 4 + 1, 256, 8), 256, 0, stream>>>(g, n, guard);
  VITK_CHECK_LAUNCH("nonfinite_scan_kernel");
  return VITK_OK;
}

int grad_guard_finish(int* guard, cudaStream_t stream) {
  VITK_REQUIRE(guard != nullptr, "grad_guard_finish: null guard");
  guard_finish_kernel<<<1, 1, 0, stream>>>(guard);
  VITK_CHECK_LAUNCH("guard_finish_kernel");
  return VITK_OK;
}

int adamw_flat(float* p, const float* g, float* m, float* v, void* shadow_bf16, long long n,
               double lr, double beta1, double beta2, double eps, double weight_decay, int step,
               float grad_scale, cudaStream_t stream, const int* guard) {
  VITK_REQUIRE(p && g && m && v && n > 0 && step >= 1, "adamw: bad argument");
  VITK_REQUIRE((reinterpret_cast<uintptr_t>(p) & 15) == 0 && (reinterpret_cast<uintptr_t>(g) & 15) == 0 &&
                   (reinterpret_cast<uintptr_t>(m) & 15) == 0 && (reinterpret_cast<uintptr_t>(v) & 15) == 0,
               "adamw: arenas must be 16-byte aligned");
  // hyper-parameters are combined in double and rounded once, as torch.optim.AdamW does
  const double bc1 = 1.0 - pow(beta1, step);
  const double bc2 = 1.0 - pow(beta2, step);
  const float step_size = static_cast<float>(lr / bc1);
  const float inv_sqrt_bc2 = static_cast<float>(1.0 / sqrt(bc2));
  const float decay = static_cast<float>(1.0 - lr * weight_decay);
  ProfileScope prof(PROF_OPT, static_cast<double>(n) * 30.0, stream);
  adamw_kernel<<<grid_for(n / 4 + 1, 256, 8), 256, 0, stream>>>(
      p, g, m, v, static_cast<__nv_bfloat16*>(shadow_bf16), n, decay, static_cast<float>(beta1),
      static_cast<float>(beta2), static_cast<float>(1.0 - beta1), static_cast<float>(1.0 - beta2),
      step_size, inv_sqrt_bc2, static_cast<float>(eps), grad_scale, guard, lr, beta1, beta2, step);
  VITK_CHECK_LAUNCH("adamw_kernel");
  return VITK_OK;
}

int weighted_cross_entropy(const float* logits, const long long* targets, const float* weight,
                           int rows, int C, float* loss_out, float* sums_ws, float* dlogits,
                           float grad_scale, cudaStream_t stream) {
  VITK_REQUIRE(logits && targets && sums_ws && (loss_out || dlogits),
               "weighted_cross_entropy: null operand");
  VITK_REQUIRE(rows > 0 && C > 0 && C <= 4096, "weighted_cross_entropy: bad shape %d x %d", rows, C);
  VITK_CHECK_CUDA(cudaMemsetAsync(sums_ws, 0, 2 * sizeof(float), stream));
  ProfileScope prof(PROF_OTHER, static_cast<double>(rows) * C * 12.0, stream);
  const int grid = (rows + 255) / 256;
  wce_sums_kernel<<<grid, 256, 0, stream>>>(logits, targets, weight, rows, C, sums_ws);
  VITK_CHECK_LAUNCH("wce_sums_kernel");
  wce_grad_kernel<<<grid, 256, 0, stream>>>(logits, targets, weight, rows, C, sums_ws, loss_out,
                                            dlogits, grad_scale);
  VITK_CHECK_LAUNCH("wce_grad_kernel");
  return VITK_OK;
}

}  // namespace vitk
