// Attention core for every shape the tcgen05 kernels do not cover, forward AND backward, with the
// log-sum-exp output and the attention-probability dropout the training step needs:
//   * head_dim 8 .. 128 in steps of 8 - the reference's shipped Config trains D = 400 with 25 heads
//     of dimension 16 (train.py:1345-1356); nothing else here handles head_dim 16;
//   * more than 256 tokens in the backward (a 384 px fine-tune has 577), dropout beyond 208 tokens.
// softmax(q k^T / sqrt(hd)) v per (image, head) on the packed qkv activation - reference
// train.py:536-549, scores divided AFTER the product (:543), dropout on the probabilities (:545).
//
// Plain CUDA-core kernels (fp32 arithmetic on bf16 operands staged in shared memory), written for
// coverage, not for the roofline: these shapes are 4-8 % of a step's FLOPs and none of the
// BASELINE configurations.  One warp owns a query row (or, in the second backward pass, a key
// row); lanes stride over the keys for the score products and over the head dimension for the
// probability-weighted sums, so no value ever crosses a warp.
//   forward        : S row -> softmax (+ lse) -> dropout -> O row
//   backward pass 1: per query row  dS row, dQ row            (K, V resident in shared memory)
//   backward pass 2: per key row    P / dS column, dK, dV row (Q, dO resident in shared memory)
// Both backward passes recompute the probabilities from the saved log-sum-exp with the same
// accumulation order as the forward.
#include <cuda_bf16.h>

#include "attention_kernels.cuh"
#include "common.h"
#include "ptx.cuh"
#include "train_ops.cuh"

namespace vitk {
using namespace ptx;

namespace {

constexpr int kGenWarps = 8;
constexpr int kGenThreads = kGenWarps * 32;
constexpr int kGenMaxKeysPerLane = 32;  // N <= 1024
constexpr int kGenRowsPerBlock = 32;    // query (or key) rows per block: K/V staged once per block

__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ float warp_add(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// rows [0, N) of one head's q / k / v (or of ctx / d_ctx: `ld` and `col0` select the matrix) into
// shared memory as bf16 rows of `hdp` elements (hd + 8: a 16-byte pad staggers the banks)
__device__ __forceinline__ void stage_rows(__nv_bfloat16* dst, const __nv_bfloat16* src, long long ld,
                                           int N, int hd, int hdp) {
  const int vec_per_row = hd >> 3;
  for (int idx = threadIdx.x; idx < N * vec_per_row; idx += blockDim.x) {
    const int r = idx / vec_per_row, c = idx - r * vec_per_row;
    *reinterpret_cast<uint4*>(dst + r * hdp + 8 * c) =
        __ldg(reinterpret_cast<const uint4*>(src + r * ld + 8 * c));
  }
}

// dot(a[0..hd) fp32 in shared memory (same address for every lane: broadcast), b row bf16)
__device__ __forceinline__ float dot_row(const float* a, const __nv_bfloat16* b, int hd) {
  float acc = 0.f;
  for (int c = 0; c < hd; c += 8) {
    const uint4 v = *reinterpret_cast<const uint4*>(b + c);
    acc = fmaf(a[c + 0], bf16lo_to_f32(v.x), acc);
    acc = fmaf(a[c + 1], bf16hi_to_f32(v.x), acc);
    acc = fmaf(a[c + 2], bf16lo_to_f32(v.y), acc);
    acc = fmaf(a[c + 3], bf16hi_to_f32(v.y), acc);
    acc = fmaf(a[c + 4], bf16lo_to_f32(v.z), acc);
    acc = fmaf(a[c + 5], bf16hi_to_f32(v.z), acc);
    acc = fmaf(a[c + 6], bf16lo_to_f32(v.w), acc);
    acc = fmaf(a[c + 7], bf16hi_to_f32(v.w), acc);
  }
  return acc;
}

// out[d] (d = lane, lane + 32, ..) = sum_j w[j] * rows[j][d]   (w fp32 in shared memory)
__device__ __forceinline__ void weighted_sum(const float* w, const __nv_bfloat16* rows, int n, int hd,
                                             int hdp, int lane, float (&out)[4]) {
  out[0] = out[1] = out[2] = out[3] = 0.f;
  for (int j = 0; j < n; ++j) {
    const float wj = w[j];
    const __nv_bfloat16* r = rows + j * hdp;
#pragma unroll
    for (int q = 0; q < 4; ++q)
      if (lane + 32 * q < hd) out[q] = fmaf(wj, __bfloat162float(r[lane + 32 * q]), out[q]);
  }
}

struct GenParams {
  const __nv_bfloat16* qkv;   // [B*N, 3*D]
  const __nv_bfloat16* ctx;   // backward: [B*N, D]
  const __nv_bfloat16* dctx;  // backward: [B*N, D]
  __nv_bfloat16* out;         // forward: ctx; backward: dqkv [B*N, 3*D]
  float* lse;                 // [B, H, N] natural log of the row sums of exp(scaled scores)
  int N, H, hd, hdp, Nk;      // Nk = N rounded up to 16: row pitch of the dropout element index
  float scale;
  DropParams drop;
};

__device__ __forceinline__ bool keep_prob(const GenParams& p, int bh, int i, int j) {
  if (p.drop.thresh == 0u) return true;
  const uint32_t idx = (static_cast<uint32_t>(bh) * static_cast<uint32_t>(p.N) +
                        static_cast<uint32_t>(i)) * static_cast<uint32_t>(p.Nk) +
                       static_cast<uint32_t>(j);
  return drop_keep(idx, p.drop.key, p.drop.thresh);
}

// shared memory: K [N][hdp], V [N][hdp] (bf16), then per warp: q [hd] fp32 and p [N] fp32
__global__ void __launch_bounds__(kGenThreads)
attn_gen_fwd_kernel(const GenParams p) {
  extern __shared__ __align__(16) uint8_t smem_gen[];
  const int N = p.N, hd = p.hd, hdp = p.hdp, D = p.H * hd;
  __nv_bfloat16* sK = reinterpret_cast<__nv_bfloat16*>(smem_gen);
  __nv_bfloat16* sV = sK + N * hdp;
  float* sw = reinterpret_cast<float*>(sV + N * hdp);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* sq = sw + warp * (hd + N);
  float* sp = sq + hd;
  const int bh = blockIdx.y, b = bh / p.H, h = bh - b * p.H;
  const __nv_bfloat16* base = p.qkv + static_cast<long long>(b) * N * 3 * D + h * hd;
  stage_rows(sK, base + D, 3ll * D, N, hd, hdp);
  stage_rows(sV, base + 2 * D, 3ll * D, N, hd, hdp);
  __syncthreads();
  const int i_end = min(N, (blockIdx.x + 1) * kGenRowsPerBlock);
  for (int i = blockIdx.x * kGenRowsPerBlock + warp; i < i_end; i += kGenWarps) {
    for (int d = lane; d < hd; d += 32) sq[d] = __bfloat162float(base[static_cast<long long>(i) * 3 * D + d]);
    __syncwarp();
    float s[kGenMaxKeysPerLane];
    float m = -INFINITY;
#pragma unroll
    for (int t = 0; t < kGenMaxKeysPerLane; ++t) {
      const int j = lane + 32 * t;
      if (j < N) {
        s[t] = dot_row(sq, sK + j * hdp, hd) * p.scale;   // (q . k) / sqrt(hd), train.py:543
        m = fmaxf(m, s[t]);
      }
    }
    m = warp_max(m);
    float sum = 0.f;
#pragma unroll
    for (int t = 0; t < kGenMaxKeysPerLane; ++t) {
      const int j = lane + 32 * t;
      if (j < N) {
        s[t] = __expf(s[t] - m);
        sum += s[t];
      }
    }
    sum = warp_add(sum);
    const float inv = 1.f / sum;
    if (lane == 0 && p.lse != nullptr) p.lse[static_cast<long long>(bh) * N + i] = m + __logf(sum);
#pragma unroll
    for (int t = 0; t < kGenMaxKeysPerLane; ++t) {
      const int j = lane + 32 * t;
      if (j < N) sp[j] = keep_prob(p, bh, i, j) ? s[t] * inv * p.drop.scale : 0.f;
    }
    __syncwarp();
    float o[4];
    weighted_sum(sp, sV, N, hd, hdp, lane, o);
    __nv_bfloat16* orow = p.out + (static_cast<long long>(b) * N + i) * D + h * hd;
#pragma unroll
    for (int q = 0; q < 4; ++q)
      if (lane + 32 * q < hd) orow[lane + 32 * q] = __float2bfloat16_rn(o[q]);
    __syncwarp();
  }
}

// Backward.  pass 0 (query rows): dQ_i = sum_j dS_ij K_j;  pass 1 (key rows): dK_j = sum_i dS_ij Q_i,
// dV_j = sum_i P~_ij dO_i, with P = exp(S - lse), P~ = dropout(P), dP = dropout-mask(dO V^T),
// dS = P (dP - rowsum(dO * O)) / sqrt(hd).
// shared memory: A [N][hdp], Bm [N][hdp] (bf16: K, V in pass 0; Q, dO in pass 1), lse [N], Drow [N]
// fp32 (pass 1), then per warp: two fp32 vectors [hd] and two fp32 arrays [N].
__global__ void __launch_bounds__(kGenThreads)
attn_gen_bwd_kernel(const GenParams p) {
  extern __shared__ __align__(16) uint8_t smem_gen[];
  const int N = p.N, hd = p.hd, hdp = p.hdp, D = p.H * hd;
  const int pass = blockIdx.z;
  __nv_bfloat16* sA = reinterpret_cast<__nv_bfloat16*>(smem_gen);
  __nv_bfloat16* sB = sA + N * hdp;
  float* s_lse = reinterpret_cast<float*>(sB + N * hdp);
  float* s_drow = s_lse + N;
  float* sw = s_drow + N;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* v0 = sw + warp * (2 * hd + 2 * N);   // pass 0: q_i        pass 1: k_j
  float* v1 = v0 + hd;                        // pass 0: dO_i       pass 1: v_j
  float* w0 = v1 + hd;                        // pass 0: dS row     pass 1: dS column
  float* w1 = w0 + N;                         // pass 0: -          pass 1: P~ column
  const int bh = blockIdx.y, b = bh / p.H, h = bh - b * p.H;
  const long long row0 = static_cast<long long>(b) * N;
  const __nv_bfloat16* qkv = p.qkv + row0 * 3 * D + h * hd;
  const __nv_bfloat16* ctx = p.ctx + row0 * D + h * hd;
  const __nv_bfloat16* dctx = p.dctx + row0 * D + h * hd;
  __nv_bfloat16* dqkv = p.out + row0 * 3 * D + h * hd;
  if (pass == 0) {
    stage_rows(sA, qkv + D, 3ll * D, N, hd, hdp);       // K
    stage_rows(sB, qkv + 2 * D, 3ll * D, N, hd, hdp);   // V
  } else {
    stage_rows(sA, qkv, 3ll * D, N, hd, hdp);           // Q
    stage_rows(sB, dctx, D, N, hd, hdp);                // dO
    for (int i = threadIdx.x; i < N; i += blockDim.x) s_lse[i] = p.lse[static_cast<long long>(bh) * N + i];
  }
  __syncthreads();
  if (pass == 1) {
    // Drow_i = dO_i . O_i for every query row of this head
    for (int i = warp; i < N; i += kGenWarps) {
      float acc = 0.f;
      for (int d = lane; d < hd; d += 32)
        acc = fmaf(__bfloat162float(sB[i * hdp + d]), __bfloat162float(ctx[static_cast<long long>(i) * D + d]), acc);
      acc = warp_add(acc);
      if (lane == 0) s_drow[i] = acc;
    }
    __syncthreads();
  }
  const int r_end = min(N, (blockIdx.x + 1) * kGenRowsPerBlock);
  for (int r = blockIdx.x * kGenRowsPerBlock + warp; r < r_end; r += kGenWarps) {
    if (pass == 0) {
      const int i = r;
      for (int d = lane; d < hd; d += 32) {
        v0[d] = __bfloat162float(qkv[static_cast<long long>(i) * 3 * D + d]);
        v1[d] = __bfloat162float(dctx[static_cast<long long>(i) * D + d]);
      }
      float dr = 0.f;
      for (int d = lane; d < hd; d += 32)
        dr = fmaf(__bfloat162float(dctx[static_cast<long long>(i) * D + d]),
                  __bfloat162float(ctx[static_cast<long long>(i) * D + d]), dr);
      dr = warp_add(dr);
      const float lse_i = p.lse[static_cast<long long>(bh) * N + i];
      __syncwarp();
      for (int j = lane; j < N; j += 32) {
        const float pij = __expf(dot_row(v0, sA + j * hdp, hd) * p.scale - lse_i);
        float dp = dot_row(v1, sB + j * hdp, hd);
        dp = keep_prob(p, bh, i, j) ? dp * p.drop.scale : 0.f;
        w0[j] = pij * (dp - dr) * p.scale;
      }
      __syncwarp();
      float o[4];
      weighted_sum(w0, sA, N, hd, hdp, lane, o);
      __nv_bfloat16* out = dqkv + static_cast<long long>(i) * 3 * D;
#pragma unroll
      for (int q = 0; q < 4; ++q)
        if (lane + 32 * q < hd) out[lane + 32 * q] = __float2bfloat16_rn(o[q]);
    } else {
      const int j = r;
      for (int d = lane; d < hd; d += 32) {
        v0[d] = __bfloat162float(qkv[static_cast<long long>(j) * 3 * D + D + d]);
        v1[d] = __bfloat162float(qkv[static_cast<long long>(j) * 3 * D + 2 * D + d]);
      }
      __syncwarp();
      for (int i = lane; i < N; i += 32) {
        // same products and accumulation order as pass 0 / the forward (d ascending)
        const float pij = __expf(dot_row(v0, sA + i * hdp, hd) * p.scale - s_lse[i]);
        float dp = dot_row(v1, sB + i * hdp, hd);
        const bool keep = keep_prob(p, bh, i, j);
        dp = keep ? dp * p.drop.scale : 0.f;
        w0[i] = pij * (dp - s_drow[i]) * p.scale;
        w1[i] = keep ? pij * p.drop.scale : 0.f;
      }
      __syncwarp();
      float dk[4], dv[4];
      weighted_sum(w0, sA, N, hd, hdp, lane, dk);
      weighted_sum(w1, sB, N, hd, hdp, lane, dv);
      __nv_bfloat16* out = dqkv + static_cast<long long>(j) * 3 * D;
#pragma unroll
      for (int q = 0; q < 4; ++q)
        if (lane + 32 * q < hd) {
          out[D + lane + 32 * q] = __float2bfloat16_rn(dk[q]);
          out[2 * D + lane + 32 * q] = __float2bfloat16_rn(dv[q]);
        }
    }
    __syncwarp();
  }
}

// ---------------------------------------------------------------------------------------------
// Generic-source form (decoder layers of the detection head under training, train.py:691-731 /
// 842-845 differentiated at :1455): queries, keys / values, context and every gradient have their
// own base pointer, row pitch and per-image pitch, and there may be a different number of queries
// and keys (100 object queries against 196 patch tokens).  Same arithmetic as the kernels above.
// ---------------------------------------------------------------------------------------------
struct XParams {
  const __nv_bfloat16 *q, *k, *v, *ctx, *dctx;
  __nv_bfloat16 *out, *dq, *dk, *dv;
  float* lse;
  long long q_img, kv_img, ctx_img, dq_img, dkv_img;
  int ldq, ldkv, ldc, lddq, lddkv;
  int Nq, Nk, H, hd, hdp;
  int Nkp;      // keys rounded up to 16: row pitch of the dropout element index
  float scale;
  DropParams drop;
};

__device__ __forceinline__ bool keep_prob_x(const XParams& p, int bh, int i, int j) {
  if (p.drop.thresh == 0u) return true;
  const uint32_t idx = (static_cast<uint32_t>(bh) * static_cast<uint32_t>(p.Nq) +
                        static_cast<uint32_t>(i)) * static_cast<uint32_t>(p.Nkp) +
                       static_cast<uint32_t>(j);
  return drop_keep(idx, p.drop.key, p.drop.thresh);
}

// forward: K, V of the head resident in shared memory; one warp per query row
__global__ void __launch_bounds__(kGenThreads)
attn_xgen_fwd_kernel(const XParams p) {
  extern __shared__ __align__(16) uint8_t smem_gen[];
  const int Nk = p.Nk, hd = p.hd, hdp = p.hdp;
  __nv_bfloat16* sK = reinterpret_cast<__nv_bfloat16*>(smem_gen);
  __nv_bfloat16* sV = sK + Nk * hdp;
  float* sw = reinterpret_cast<float*>(sV + Nk * hdp);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* sq = sw + warp * (hd + Nk);
  float* sp = sq + hd;
  const int bh = blockIdx.y, b = bh / p.H, h = bh - b * p.H;
  stage_rows(sK, p.k + b * p.kv_img + h * hd, p.ldkv, Nk, hd, hdp);
  stage_rows(sV, p.v + b * p.kv_img + h * hd, p.ldkv, Nk, hd, hdp);
  __syncthreads();
  const __nv_bfloat16* qb = p.q + b * p.q_img + h * hd;
  const int i_end = min(p.Nq, (blockIdx.x + 1) * kGenRowsPerBlock);
  for (int i = blockIdx.x * kGenRowsPerBlock + warp; i < i_end; i += kGenWarps) {
    for (int d = lane; d < hd; d += 32) sq[d] = __bfloat162float(qb[static_cast<long long>(i) * p.ldq + d]);
    __syncwarp();
    float s[kGenMaxKeysPerLane];
    float m = -INFINITY;
#pragma unroll
    for (int t = 0; t < kGenMaxKeysPerLane; ++t) {
      const int j = lane + 32 * t;
      if (j < Nk) {
        s[t] = dot_row(sq, sK + j * hdp, hd) * p.scale;
        m = fmaxf(m, s[t]);
      }
    }
    m = warp_max(m);
    float sum = 0.f;
#pragma unroll
    for (int t = 0; t < kGenMaxKeysPerLane; ++t) {
      const int j = lane + 32 * t;
      if (j < Nk) {
        s[t] = __expf(s[t] - m);
        sum += s[t];
      }
    }
    sum = warp_add(sum);
    const float inv = 1.f / sum;
    if (lane == 0 && p.lse != nullptr) p.lse[static_cast<long long>(bh) * p.Nq + i] = m + __logf(sum);
#pragma unroll
    for (int t = 0; t < kGenMaxKeysPerLane; ++t) {
      const int j = lane + 32 * t;
      if (j < Nk) sp[j] = keep_prob_x(p, bh, i, j) ? s[t] * inv * p.drop.scale : 0.f;
    }
    __syncwarp();
    float o[4];
    weighted_sum(sp, sV, Nk, hd, hdp, lane, o);
    __nv_bfloat16* orow = p.out + b * p.ctx_img + static_cast<long long>(i) * p.ldc + h * hd;
#pragma unroll
    for (int q = 0; q < 4; ++q)
      if (lane + 32 * q < hd) orow[lane + 32 * q] = __float2bfloat16_rn(o[q]);
    __syncwarp();
  }
}

// backward.  blockIdx.z == 0: query rows (K, V resident) -> dQ;  == 1: key rows (Q, dO, lse and
// dO . O resident) -> dK, dV.  Per-warp scratch: two fp32 vectors [hd] and two fp32 arrays of the
// other side's length.
__global__ void __launch_bounds__(kGenThreads)
attn_xgen_bwd_kernel(const XParams p) {
  extern __shared__ __align__(16) uint8_t smem_gen[];
  const int Nq = p.Nq, Nk = p.Nk, hd = p.hd, hdp = p.hdp;
  const int pass = blockIdx.z;
  const int n_res = pass == 0 ? Nk : Nq;   // rows resident in shared memory
  const int n_own = pass == 0 ? Nq : Nk;   // rows distributed over the warps
  if (blockIdx.x * kGenRowsPerBlock >= n_own) return;
  __nv_bfloat16* sA = reinterpret_cast<__nv_bfloat16*>(smem_gen);
  __nv_bfloat16* sB = sA + n_res * hdp;
  float* s_lse = reinterpret_cast<float*>(sB + n_res * hdp);
  float* s_drow = s_lse + n_res;
  float* sw = s_drow + n_res;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* v0 = sw + warp * (2 * hd + 2 * n_res);
  float* v1 = v0 + hd;
  float* w0 = v1 + hd;
  float* w1 = w0 + n_res;
  const int bh = blockIdx.y, b = bh / p.H, h = bh - b * p.H;
  const __nv_bfloat16* q = p.q + b * p.q_img + h * hd;
  const __nv_bfloat16* k = p.k + b * p.kv_img + h * hd;
  const __nv_bfloat16* v = p.v + b * p.kv_img + h * hd;
  const __nv_bfloat16* ctx = p.ctx + b * p.ctx_img + h * hd;
  const __nv_bfloat16* dctx = p.dctx + b * p.ctx_img + h * hd;
  const float* lse = p.lse + static_cast<long long>(bh) * Nq;
  if (pass == 0) {
    stage_rows(sA, k, p.ldkv, Nk, hd, hdp);
    stage_rows(sB, v, p.ldkv, Nk, hd, hdp);
  } else {
    stage_rows(sA, q, p.ldq, Nq, hd, hdp);
    stage_rows(sB, dctx, p.ldc, Nq, hd, hdp);
    for (int i = threadIdx.x; i < Nq; i += blockDim.x) s_lse[i] = lse[i];
  }
  __syncthreads();
  if (pass == 1) {
    for (int i = warp; i < Nq; i += kGenWarps) {
      float acc = 0.f;
      for (int d = lane; d < hd; d += 32)
        acc = fmaf(__bfloat162float(sB[i * hdp + d]),
                   __bfloat162float(ctx[static_cast<long long>(i) * p.ldc + d]), acc);
      acc = warp_add(acc);
      if (lane == 0) s_drow[i] = acc;
    }
    __syncthreads();
  }
  const int r_end = min(n_own, (blockIdx.x + 1) * kGenRowsPerBlock);
  for (int r = blockIdx.x * kGenRowsPerBlock + warp; r < r_end; r += kGenWarps) {
    if (pass == 0) {
      const int i = r;
      float dr = 0.f;
      for (int d = lane; d < hd; d += 32) {
        const float go = __bfloat162float(dctx[static_cast<long long>(i) * p.ldc + d]);
        v0[d] = __bfloat162float(q[static_cast<long long>(i) * p.ldq + d]);
        v1[d] = go;
        dr = fmaf(go, __bfloat162float(ctx[static_cast<long long>(i) * p.ldc + d]), dr);
      }
      dr = warp_add(dr);
      const float lse_i = lse[i];
      __syncwarp();
      for (int j = lane; j < Nk; j += 32) {
        const float pij = __expf(dot_row(v0, sA + j * hdp, hd) * p.scale - lse_i);
        float dp = dot_row(v1, sB + j * hdp, hd);
        dp = keep_prob_x(p, bh, i, j) ? dp * p.drop.scale : 0.f;
        w0[j] = pij * (dp - dr) * p.scale;
      }
      __syncwarp();
      float o[4];
      weighted_sum(w0, sA, Nk, hd, hdp, lane, o);
      __nv_bfloat16* out = p.dq + b * p.dq_img + static_cast<long long>(i) * p.lddq + h * hd;
#pragma unroll
      for (int t = 0; t < 4; ++t)
        if (lane + 32 * t < hd) out[lane + 32 * t] = __float2bfloat16_rn(o[t]);
    } else {
      const int j = r;
      for (int d = lane; d < hd; d += 32) {
        v0[d] = __bfloat162float(k[static_cast<long long>(j) * p.ldkv + d]);
        v1[d] = __bfloat162float(v[static_cast<long long>(j) * p.ldkv + d]);
      }
      __syncwarp();
      for (int i = lane; i < Nq; i += 32) {
        const float pij = __expf(dot_row(v0, sA + i * hdp, hd) * p.scale - s_lse[i]);
        float dp = dot_row(v1, sB + i * hdp, hd);
        const bool keep = keep_prob_x(p, bh, i, j);
        dp = keep ? dp * p.drop.scale : 0.f;
        w0[i] = pij * (dp - s_drow[i]) * p.scale;
        w1[i] = keep ? pij * p.drop.scale : 0.f;
      }
      __syncwarp();
      float dk[4], dv[4];
      weighted_sum(w0, sA, Nq, hd, hdp, lane, dk);
      weighted_sum(w1, sB, Nq, hd, hdp, lane, dv);
      const long long off = b * p.dkv_img + static_cast<long long>(j) * p.lddkv + h * hd;
#pragma unroll
      for (int t = 0; t < 4; ++t)
        if (lane + 32 * t < hd) {
          p.dk[off + lane + 32 * t] = __float2bfloat16_rn(dk[t]);
          p.dv[off + lane + 32 * t] = __float2bfloat16_rn(dv[t]);
        }
    }
    __syncwarp();
  }
}

int check_shape(int B, int N, int H, int hd, const DropParams* drop) {
  VITK_REQUIRE(B > 0 && N > 0 && H > 0, "attention (generic): bad shape B=%d N=%d H=%d", B, N, H);
  VITK_REQUIRE(hd >= 8 && hd <= 128 && hd % 8 == 0,
               "attention (generic): head_dim %d unsupported (8 .. 128 in steps of 8)", hd);
  VITK_REQUIRE(N <= 32 * kGenMaxKeysPerLane, "attention (generic): at most %d tokens (got %d)",
               32 * kGenMaxKeysPerLane, N);
  const int Nk = (N + 15) & ~15;
  VITK_REQUIRE(drop == nullptr || drop->thresh == 0u ||
                   static_cast<long long>(B) * H * N * Nk < (1ll << 32),
               "attention dropout: batch * heads * tokens^2 must stay below 2^32");
  return VITK_OK;
}

}  // namespace

bool attention_gen_fits(int N, int hd) {
  if (hd < 8 || hd > 128 || hd % 8 != 0 || N <= 0 || N > 32 * kGenMaxKeysPerLane) return false;
  const size_t bwd = 2 * static_cast<size_t>(N) * (hd + 8) * 2 + 2 * static_cast<size_t>(N) * 4 +
                     kGenWarps * (2 * static_cast<size_t>(hd) + 2 * N) * 4;
  return bwd <= 232448;
}

int attention_gen_fwd(const void* qkv, void* ctx, float* lse, int B, int N, int H, int hd,
                      cudaStream_t stream, const DropParams* drop) {
  VITK_REQUIRE(qkv && ctx, "attention (generic): null operand");
  VITK_TRY(check_shape(B, N, H, hd, drop));
  GenParams p{};
  p.qkv = static_cast<const __nv_bfloat16*>(qkv);
  p.out = static_cast<__nv_bfloat16*>(ctx);
  p.lse = lse;
  p.N = N;
  p.H = H;
  p.hd = hd;
  p.hdp = hd + 8;
  p.Nk = (N + 15) & ~15;
  p.scale = 1.0f / sqrtf(static_cast<float>(hd));
  if (drop != nullptr) p.drop = *drop;
  const size_t smem = 2 * static_cast<size_t>(N) * p.hdp * 2 + kGenWarps * (static_cast<size_t>(hd) + N) * 4;
  VITK_REQUIRE(smem <= 232448, "attention (generic): %d tokens x head_dim %d do not fit in shared "
               "memory", N, hd);
  if (smem > 48 * 1024) VITK_TRY(opt_in_smem<attn_gen_fwd_kernel>(232448, "attn_gen_fwd_kernel"));
  ProfileScope prof(PROF_ATTN, attention_flops(B, H, N, N, hd), stream);
  const dim3 grid((N + kGenRowsPerBlock - 1) / kGenRowsPerBlock, B * H);
  attn_gen_fwd_kernel<<<grid, kGenThreads, smem, stream>>>(p);
  VITK_CHECK_LAUNCH("attn_gen_fwd_kernel");
  return VITK_OK;
}

int attention_gen_bwd(const void* qkv, const void* ctx, const void* dctx, const float* lse,
                      void* dqkv, int B, int N, int H, int hd, cudaStream_t stream,
                      const DropParams* drop, float* dbias) {
  VITK_REQUIRE(qkv && ctx && dctx && lse && dqkv, "attention_bwd (generic): null operand");
  VITK_TRY(check_shape(B, N, H, hd, drop));
  VITK_REQUIRE(attention_gen_fits(N, hd), "attention_bwd (generic): %d tokens x head_dim %d do not "
               "fit in shared memory", N, hd);
  GenParams p{};
  p.qkv = static_cast<const __nv_bfloat16*>(qkv);
  p.ctx = static_cast<const __nv_bfloat16*>(ctx);
  p.dctx = static_cast<const __nv_bfloat16*>(dctx);
  p.out = static_cast<__nv_bfloat16*>(dqkv);
  p.lse = const_cast<float*>(lse);
  p.N = N;
  p.H = H;
  p.hd = hd;
  p.hdp = hd + 8;
  p.Nk = (N + 15) & ~15;
  p.scale = 1.0f / sqrtf(static_cast<float>(hd));
  if (drop != nullptr) p.drop = *drop;
  const size_t smem = 2 * static_cast<size_t>(N) * p.hdp * 2 + 2 * static_cast<size_t>(N) * 4 +
                      kGenWarps * (2 * static_cast<size_t>(hd) + 2 * N) * 4;
  if (smem > 48 * 1024) VITK_TRY(opt_in_smem<attn_gen_bwd_kernel>(232448, "attn_gen_bwd_kernel"));
  ProfileScope prof(PROF_ATTN, attention_flops(B, H, N, N, hd, true), stream);
  const dim3 grid((N + kGenRowsPerBlock - 1) / kGenRowsPerBlock, B * H, 2);
  attn_gen_bwd_kernel<<<grid, kGenThreads, smem, stream>>>(p);
  VITK_CHECK_LAUNCH("attn_gen_bwd_kernel");
  if (dbias != nullptr)   // bias gradient of the qkv Linear: column sums of dqkv
    return colsum_bf16(dqkv, 3ll * H * hd, B * N, 3 * H * hd, dbias, stream);
  return VITK_OK;
}

namespace {
int xgen_check(const AttnXSrc& s, int B, int Nq, int Nk, int H, int hd, const DropParams* drop) {
  VITK_REQUIRE(drop == nullptr || drop->thresh == 0u ||
                   static_cast<long long>(B) * H * Nq * ((Nk + 15) & ~15) < (1ll << 32),
               "attention dropout: batch * heads * queries * keys must stay below 2^32");
  VITK_REQUIRE(s.q && s.k && s.v, "attention (generic sources): null operand");
  VITK_REQUIRE(B > 0 && Nq > 0 && Nk > 0 && H > 0, "attention (generic sources): bad shape");
  VITK_REQUIRE(hd >= 8 && hd <= 128 && hd % 8 == 0,
               "attention (generic sources): head_dim %d unsupported (8 .. 128 in steps of 8)", hd);
  VITK_REQUIRE(Nq <= 32 * kGenMaxKeysPerLane && Nk <= 32 * kGenMaxKeysPerLane,
               "attention (generic sources): at most %d queries / keys", 32 * kGenMaxKeysPerLane);
  VITK_REQUIRE(s.ldq % 8 == 0 && s.ldkv % 8 == 0 && s.q_img % 8 == 0 && s.kv_img % 8 == 0,
               "attention (generic sources): pitches must be multiples of 8 elements");
  return VITK_OK;
}
}  // namespace

int attention_xgen_fwd(const AttnXSrc& s, void* ctx, long long ctx_img, int ldc, float* lse, int B,
                       int Nq, int Nk, int H, int hd, cudaStream_t stream, const DropParams* drop) {
  VITK_TRY(xgen_check(s, B, Nq, Nk, H, hd, drop));
  VITK_REQUIRE(ctx != nullptr, "attention (generic sources): null output");
  XParams p{};
  p.q = static_cast<const __nv_bfloat16*>(s.q);
  p.k = static_cast<const __nv_bfloat16*>(s.k);
  p.v = static_cast<const __nv_bfloat16*>(s.v);
  p.out = static_cast<__nv_bfloat16*>(ctx);
  p.lse = lse;
  p.q_img = s.q_img; p.kv_img = s.kv_img; p.ctx_img = ctx_img;
  p.ldq = s.ldq; p.ldkv = s.ldkv; p.ldc = ldc;
  p.Nq = Nq; p.Nk = Nk; p.H = H; p.hd = hd; p.hdp = hd + 8;
  p.Nkp = (Nk + 15) & ~15;
  p.scale = 1.0f / sqrtf(static_cast<float>(hd));
  if (drop != nullptr) p.drop = *drop;
  const size_t smem = 2 * static_cast<size_t>(Nk) * p.hdp * 2 + kGenWarps * (static_cast<size_t>(hd) + Nk) * 4;
  VITK_REQUIRE(smem <= 232448, "attention (generic sources): %d keys x head_dim %d do not fit in "
               "shared memory", Nk, hd);
  if (smem > 48 * 1024) VITK_TRY(opt_in_smem<attn_xgen_fwd_kernel>(232448, "attn_xgen_fwd_kernel"));
  ProfileScope prof(PROF_ATTN, attention_flops(B, H, Nq, Nk, hd), stream);
  const dim3 grid((Nq + kGenRowsPerBlock - 1) / kGenRowsPerBlock, B * H);
  attn_xgen_fwd_kernel<<<grid, kGenThreads, smem, stream>>>(p);
  VITK_CHECK_LAUNCH("attn_xgen_fwd_kernel");
  return VITK_OK;
}

int attention_xgen_bwd(const AttnXSrc& s, const void* ctx, const void* dctx, long long ctx_img,
                       int ldc, const float* lse, void* dq, long long dq_img, int lddq, void* dk,
                       void* dv, long long dkv_img, int lddkv, int B, int Nq, int Nk, int H, int hd,
                       cudaStream_t stream, const DropParams* drop) {
  VITK_TRY(xgen_check(s, B, Nq, Nk, H, hd, drop));
  VITK_REQUIRE(ctx && dctx && lse && dq && dk && dv, "attention_bwd (generic sources): null operand");
  XParams p{};
  p.q = static_cast<const __nv_bfloat16*>(s.q);
  p.k = static_cast<const __nv_bfloat16*>(s.k);
  p.v = static_cast<const __nv_bfloat16*>(s.v);
  p.ctx = static_cast<const __nv_bfloat16*>(ctx);
  p.dctx = static_cast<const __nv_bfloat16*>(dctx);
  p.dq = static_cast<__nv_bfloat16*>(dq);
  p.dk = static_cast<__nv_bfloat16*>(dk);
  p.dv = static_cast<__nv_bfloat16*>(dv);
  p.lse = const_cast<float*>(lse);
  p.q_img = s.q_img; p.kv_img = s.kv_img; p.ctx_img = ctx_img; p.dq_img = dq_img; p.dkv_img = dkv_img;
  p.ldq = s.ldq; p.ldkv = s.ldkv; p.ldc = ldc; p.lddq = lddq; p.lddkv = lddkv;
  p.Nq = Nq; p.Nk = Nk; p.H = H; p.hd = hd; p.hdp = hd + 8;
  p.Nkp = (Nk + 15) & ~15;
  p.scale = 1.0f / sqrtf(static_cast<float>(hd));
  if (drop != nullptr) p.drop = *drop;
  const size_t nmax = static_cast<size_t>(Nq > Nk ? Nq : Nk);
  const size_t smem = 2 * nmax * p.hdp * 2 + 2 * nmax * 4 + kGenWarps * (2 * static_cast<size_t>(hd) + 2 * nmax) * 4;
  VITK_REQUIRE(smem <= 232448, "attention_bwd (generic sources): %d x head_dim %d do not fit in "
               "shared memory", static_cast<int>(nmax), hd);
  if (smem > 48 * 1024) VITK_TRY(opt_in_smem<attn_xgen_bwd_kernel>(232448, "attn_xgen_bwd_kernel"));
  ProfileScope prof(PROF_ATTN, attention_flops(B, H, Nq, Nk, hd, true), stream);
  const int rows = Nq > Nk ? Nq : Nk;
  const dim3 grid((rows + kGenRowsPerBlock - 1) / kGenRowsPerBlock, B * H, 2);
  attn_xgen_bwd_kernel<<<grid, kGenThreads, smem, stream>>>(p);
  VITK_CHECK_LAUNCH("attn_xgen_bwd_kernel");
  return VITK_OK;
}

}  // namespace vitk
