// Tensor-core (mma.sync) attention with separate query and key / value sources, backward and a
// training forward (log-sum-exp output, dropout on the probabilities) - the decoder
// layers of the detection head under training (nn.MultiheadAttention inside
// nn.TransformerDecoderLayer, train.py:701-707, differentiated at train.py:1455): 100 object
// queries against 100 (self-attention) or 196 (cross-attention onto the patch tokens) keys, 8 heads
// of dimension 96 - and the encoder's own attention under training when head_dim != 64 (the
// reference's shipped Config: 25 heads of 16, train.py:1345-1356).  head_dim 16 .. 128 in steps of
// 16; any number of queries and keys that fits shared memory.
//
//   P  = exp(q k^T * scale - lse)           dP = d_ctx v^T           Drow = rowsum(d_ctx * ctx)
//   dS = P * (dropmask(dP) - Drow) * scale  dq = dS k     dk = dS^T q     dv = dropmask(P)^T d_ctx
//
// One CTA per (image, head): q, d_ctx, k, v of the head are staged once by cp.async into rows
// padded by 16 bytes (conflict-free ldmatrix for every head size).  Two passes, as in
// attention_flash.cu, so that no sum ever crosses a warp: a warp owns 16 query rows (dq) or 16 key
// rows (dk, dv) and walks the other side in chunks of 32, recomputing its score blocks with bf16
// m16n8k16 MMAs (fp32 accumulate) from the saved log-sum-exp; the probabilities and dS go straight
// from the accumulator registers into the A fragments of the second product.
// (Replaces the CUDA-core attn_xgen_bwd_kernel for these shapes: 1.2 ms -> see DESIGN.md 3.7.)
#include <cuda_bf16.h>

#include "attention_kernels.cuh"
#include "common.h"
#include "dropout.cuh"
#include "ptx.cuh"

namespace vitk {
using namespace ptx;

namespace {

constexpr int kWarps = 8;
constexpr int kThreads = kWarps * 32;
constexpr int kCW = 32;  // columns of a score block

struct XmParams {
  const __nv_bfloat16 *q, *k, *v, *ctx, *dctx;
  __nv_bfloat16 *dq, *dk, *dv;
  const float* lse;
  long long q_img, kv_img, ctx_img, dq_img, dkv_img;
  int ldq, ldkv, ldc, lddq, lddkv;
  int Nq, Nk, Nq16, Nk16, H, Nkp;
  float scale;
  DropParams drop;
};

template <int HD>
struct Tile {
  static constexpr int kPitch = HD * 2 + 16;  // bytes per staged row
  static constexpr int kKS = HD / 16;         // k-steps over the head dimension
  static __device__ __forceinline__ uint32_t at(uint32_t base, int row, int ch) {
    return base + static_cast<uint32_t>(row) * kPitch + static_cast<uint32_t>(ch) * 16u;
  }
  // rows [0, rows16) x HD of one head: `rows` valid, the rest zero-filled
  static __device__ __forceinline__ void stage(uint32_t dst, const __nv_bfloat16* src, int ld,
                                               int rows, int rows16) {
    for (int idx = threadIdx.x; idx < rows16 * (HD / 8); idx += kThreads) {
      const int row = idx / (HD / 8), ch = idx - row * (HD / 8);
      const bool valid = row < rows;
      cp_async_16(at(dst, row, ch), src + static_cast<long long>(valid ? row : 0) * ld + ch * 8, valid);
    }
  }
  // A fragments (m16 x HD) of rows [row0, row0 + 16)
  static __device__ __forceinline__ void load_a(uint32_t base, int row0, int lane,
                                                uint32_t (&a)[kKS][4]) {
    const int r = row0 + (lane & 7) + ((lane >> 3) & 1) * 8;
#pragma unroll
    for (int kk = 0; kk < kKS; ++kk)
      ldmatrix_x4(at(base, r, kk * 2 + (lane >> 4)), a[kk][0], a[kk][1], a[kk][2], a[kk][3]);
  }
  // acc[16 x 32] = A[16 x HD] * Brows[row0 .. row0 + 32)[HD]^T; 8-row groups at or beyond `rem`
  // are skipped (acc = 0)
  static __device__ __forceinline__ void mma_nt(float (&acc)[kCW / 8][4], const uint32_t (&a)[kKS][4],
                                                uint32_t sB, int row0, int rem, int lane) {
#pragma unroll
    for (int j = 0; j < kCW / 8; ++j) {
      acc[j][0] = acc[j][1] = acc[j][2] = acc[j][3] = 0.f;
      if (j * 8 < rem) {
        const int row = row0 + j * 8 + (lane & 7);
#pragma unroll
        for (int q4 = 0; q4 < HD / 32; ++q4) {
          uint32_t b0, b1, b2, b3;
          ldmatrix_x4(at(sB, row, (lane >> 3) + 4 * q4), b0, b1, b2, b3);
          mma_m16n8k16(acc[j], a[2 * q4], b0, b1);
          mma_m16n8k16(acc[j], a[2 * q4 + 1], b2, b3);
        }
        if constexpr (HD % 32 != 0) {   // odd number of k-steps: the last one alone
          uint32_t b0, b1;
          ldmatrix_x2(at(sB, row, ((lane >> 3) & 1) + 4 * (HD / 32)), b0, b1);
          mma_m16n8k16(acc[j], a[kKS - 1], b0, b1);
        }
      }
    }
  }
  // out[16 x HD] += W[16 x 32] * Brows[row0 .. row0 + 32)[HD]; W given as fp32 C fragments
  static __device__ __forceinline__ void mma_wv(float (&out)[HD / 8][4], const float (&w)[kCW / 8][4],
                                                uint32_t sB, int row0, int rem, int lane) {
#pragma unroll
    for (int kk = 0; kk < kCW / 16; ++kk) {
      if (kk * 16 < rem) {
        uint32_t wa[4];
        wa[0] = pack_bf16x2(w[2 * kk][0], w[2 * kk][1]);
        wa[1] = pack_bf16x2(w[2 * kk][2], w[2 * kk][3]);
        wa[2] = pack_bf16x2(w[2 * kk + 1][0], w[2 * kk + 1][1]);
        wa[3] = pack_bf16x2(w[2 * kk + 1][2], w[2 * kk + 1][3]);
        const int mi = lane >> 3;
        const int row = row0 + kk * 16 + (mi & 1) * 8 + (lane & 7);
#pragma unroll
        for (int jj = 0; jj < kKS; ++jj) {
          uint32_t v0, v1, v2, v3;
          ldmatrix_x4_trans(at(sB, row, 2 * jj + (mi >> 1)), v0, v1, v2, v3);
          mma_m16n8k16(out[2 * jj], wa, v0, v1);
          mma_m16n8k16(out[2 * jj + 1], wa, v2, v3);
        }
      }
    }
  }
  // 16 x HD fp32 accumulators -> bf16 rows of dst (row pitch ld elements)
  static __device__ __forceinline__ void store(const float (&o)[HD / 8][4], int lane,
                                               __nv_bfloat16* dst, long long ld, int row0,
                                               int row_limit) {
    const int g = lane >> 2, t = lane & 3;
    const int r0 = row0 + g, r1 = row0 + g + 8;
#pragma unroll
    for (int j = 0; j < HD / 8; ++j) {
      if (r0 < row_limit)
        *reinterpret_cast<uint32_t*>(dst + r0 * ld + j * 8 + t * 2) = pack_bf16x2(o[j][0], o[j][1]);
      if (r1 < row_limit)
        *reinterpret_cast<uint32_t*>(dst + r1 * ld + j * 8 + t * 2) = pack_bf16x2(o[j][2], o[j][3]);
    }
  }
};

__device__ __forceinline__ bool keep_x(const XmParams& p, int bh, int i, int j) {
  const uint32_t idx = (static_cast<uint32_t>(bh) * static_cast<uint32_t>(p.Nq) +
                        static_cast<uint32_t>(i)) * static_cast<uint32_t>(p.Nkp) +
                       static_cast<uint32_t>(j);
  return drop_keep(idx, p.drop.key, p.drop.thresh);
}

template <int HD>
__global__ void __launch_bounds__(kThreads, 1)
attn_xmma_bwd_kernel(const XmParams p) {
  using T = Tile<HD>;
  extern __shared__ __align__(128) uint8_t smem[];
  const int Nq = p.Nq, Nk = p.Nk;
  const uint32_t sQ = smem_u32(smem);
  const uint32_t sdO = sQ + p.Nq16 * T::kPitch;
  const uint32_t sK = sdO + p.Nq16 * T::kPitch;
  const uint32_t sV = sK + p.Nk16 * T::kPitch;
  // +32 floats: the column loops read up to a whole 32-query chunk past Nq16 - 16
  float* sLse = reinterpret_cast<float*>(smem + static_cast<size_t>(2 * p.Nq16 + 2 * p.Nk16) * T::kPitch);
  float* sD = sLse + p.Nq16 + 32;

  const int bh = blockIdx.x, b = bh / p.H, h = bh - b * p.H;
  const __nv_bfloat16* qb = p.q + b * p.q_img + h * HD;
  const __nv_bfloat16* kb = p.k + b * p.kv_img + h * HD;
  const __nv_bfloat16* vb = p.v + b * p.kv_img + h * HD;
  const __nv_bfloat16* ob = p.ctx + b * p.ctx_img + h * HD;
  const __nv_bfloat16* dob = p.dctx + b * p.ctx_img + h * HD;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int g = lane >> 2, t = lane & 3;
  const bool dropping = p.drop.thresh != 0u;

  T::stage(sQ, qb, p.ldq, Nq, p.Nq16);
  T::stage(sdO, dob, p.ldc, Nq, p.Nq16);
  T::stage(sK, kb, p.ldkv, Nk, p.Nk16);
  T::stage(sV, vb, p.ldkv, Nk, p.Nk16);
  asm volatile("cp.async.commit_group;" ::: "memory");
  // Drow = rowsum(d_ctx * ctx) and the saved log-sum-exp in base-2 units, one query per thread
  for (int r = tid; r < p.Nq16 + 32; r += kThreads) {
    float dsum = 0.f, l2 = INFINITY;  // queries >= Nq: P = 2^(-inf) = 0
    if (r < Nq) {
      const uint4* po = reinterpret_cast<const uint4*>(ob + static_cast<long long>(r) * p.ldc);
      const uint4* pd = reinterpret_cast<const uint4*>(dob + static_cast<long long>(r) * p.ldc);
#pragma unroll
      for (int c8 = 0; c8 < HD / 8; ++c8) {
        const uint4 a = __ldg(po + c8), d = __ldg(pd + c8);
        dsum += bf16lo_to_f32(a.x) * bf16lo_to_f32(d.x) + bf16hi_to_f32(a.x) * bf16hi_to_f32(d.x);
        dsum += bf16lo_to_f32(a.y) * bf16lo_to_f32(d.y) + bf16hi_to_f32(a.y) * bf16hi_to_f32(d.y);
        dsum += bf16lo_to_f32(a.z) * bf16lo_to_f32(d.z) + bf16hi_to_f32(a.z) * bf16hi_to_f32(d.z);
        dsum += bf16lo_to_f32(a.w) * bf16lo_to_f32(d.w) + bf16hi_to_f32(a.w) * bf16hi_to_f32(d.w);
      }
      l2 = p.lse[static_cast<long long>(bh) * Nq + r] * kLog2e;
    }
    sLse[r] = l2;
    sD[r] = dsum;
  }
  asm volatile("cp.async.wait_group 0;" ::: "memory");
  __syncthreads();

  const float c = p.scale * kLog2e;

  // ================= pass 1: query tiles -> dq =================
  for (int qt = warp; qt * 16 < Nq; qt += kWarps) {
    const int q0 = qt * 16;
    uint32_t qa[T::kKS][4], doa[T::kKS][4];
    T::load_a(sQ, q0, lane, qa);
    T::load_a(sdO, q0, lane, doa);
    const float l0 = sLse[q0 + g], l1 = sLse[q0 + g + 8];
    const float d0 = sD[q0 + g], d1 = sD[q0 + g + 8];
    float dq[HD / 8][4];
#pragma unroll
    for (int j = 0; j < HD / 8; ++j) dq[j][0] = dq[j][1] = dq[j][2] = dq[j][3] = 0.f;
    for (int kc = 0; kc * kCW < Nk; ++kc) {
      const int rem = Nk - kc * kCW;
      float s[kCW / 8][4], dp[kCW / 8][4];
      T::mma_nt(s, qa, sK, kc * kCW, rem, lane);
      T::mma_nt(dp, doa, sV, kc * kCW, rem, lane);
#pragma unroll
      for (int j = 0; j < kCW / 8; ++j) {
        const int k0 = j * 8 + t * 2;          // key within the chunk of this thread's column pair
        const int key = kc * kCW + k0;
        const float p00 = (k0 < rem) ? ex2_approx(fmaf(s[j][0], c, -l0)) : 0.f;
        const float p01 = (k0 + 1 < rem) ? ex2_approx(fmaf(s[j][1], c, -l0)) : 0.f;
        const float p10 = (k0 < rem) ? ex2_approx(fmaf(s[j][2], c, -l1)) : 0.f;
        const float p11 = (k0 + 1 < rem) ? ex2_approx(fmaf(s[j][3], c, -l1)) : 0.f;
        if (dropping) {
          dp[j][0] = keep_x(p, bh, q0 + g, key) ? dp[j][0] * p.drop.scale : 0.f;
          dp[j][1] = keep_x(p, bh, q0 + g, key + 1) ? dp[j][1] * p.drop.scale : 0.f;
          dp[j][2] = keep_x(p, bh, q0 + g + 8, key) ? dp[j][2] * p.drop.scale : 0.f;
          dp[j][3] = keep_x(p, bh, q0 + g + 8, key + 1) ? dp[j][3] * p.drop.scale : 0.f;
        }
        s[j][0] = p00 * (dp[j][0] - d0) * p.scale;
        s[j][1] = p01 * (dp[j][1] - d0) * p.scale;
        s[j][2] = p10 * (dp[j][2] - d1) * p.scale;
        s[j][3] = p11 * (dp[j][3] - d1) * p.scale;
      }
      T::mma_wv(dq, s, sK, kc * kCW, rem, lane);
    }
    T::store(dq, lane, p.dq + b * p.dq_img + h * HD, p.lddq, q0, Nq);
  }

  // ================= pass 2: key tiles -> dk, dv =================
  for (int kt = warp; kt * 16 < Nk; kt += kWarps) {
    const int k0 = kt * 16;
    uint32_t ka[T::kKS][4], va[T::kKS][4];
    T::load_a(sK, k0, lane, ka);
    T::load_a(sV, k0, lane, va);
    const bool row0_ok = (k0 + g) < Nk, row1_ok = (k0 + g + 8) < Nk;
    float dk[HD / 8][4], dv[HD / 8][4];
#pragma unroll
    for (int j = 0; j < HD / 8; ++j) {
      dk[j][0] = dk[j][1] = dk[j][2] = dk[j][3] = 0.f;
      dv[j][0] = dv[j][1] = dv[j][2] = dv[j][3] = 0.f;
    }
    for (int qc = 0; qc * kCW < Nq; ++qc) {
      const int rem = Nq - qc * kCW;
      float st[kCW / 8][4], dpt[kCW / 8][4];
      T::mma_nt(st, ka, sQ, qc * kCW, rem, lane);    // S^T  = k q^T
      T::mma_nt(dpt, va, sdO, qc * kCW, rem, lane);  // dP^T = v d_ctx^T
#pragma unroll
      for (int j = 0; j < kCW / 8; ++j) {
        const int qi = qc * kCW + j * 8 + t * 2;     // query of this thread's column pair
        const float la = sLse[qi], lb = sLse[qi + 1];  // +inf beyond Nq -> P = 0
        const float da = sD[qi], db = sD[qi + 1];
        float p00 = row0_ok ? ex2_approx(fmaf(st[j][0], c, -la)) : 0.f;
        float p01 = row0_ok ? ex2_approx(fmaf(st[j][1], c, -lb)) : 0.f;
        float p10 = row1_ok ? ex2_approx(fmaf(st[j][2], c, -la)) : 0.f;
        float p11 = row1_ok ? ex2_approx(fmaf(st[j][3], c, -lb)) : 0.f;
        float g00 = dpt[j][0], g01 = dpt[j][1], g10 = dpt[j][2], g11 = dpt[j][3];
        float pd00 = p00, pd01 = p01, pd10 = p10, pd11 = p11;
        if (dropping) {
          const bool m00 = keep_x(p, bh, qi, k0 + g), m01 = keep_x(p, bh, qi + 1, k0 + g);
          const bool m10 = keep_x(p, bh, qi, k0 + g + 8), m11 = keep_x(p, bh, qi + 1, k0 + g + 8);
          g00 = m00 ? g00 * p.drop.scale : 0.f;
          g01 = m01 ? g01 * p.drop.scale : 0.f;
          g10 = m10 ? g10 * p.drop.scale : 0.f;
          g11 = m11 ? g11 * p.drop.scale : 0.f;
          pd00 = m00 ? p00 * p.drop.scale : 0.f;
          pd01 = m01 ? p01 * p.drop.scale : 0.f;
          pd10 = m10 ? p10 * p.drop.scale : 0.f;
          pd11 = m11 ? p11 * p.drop.scale : 0.f;
        }
        st[j][0] = pd00;   // the dv product uses the dropped probabilities
        st[j][1] = pd01;
        st[j][2] = pd10;
        st[j][3] = pd11;
        dpt[j][0] = p00 * (g00 - da) * p.scale;
        dpt[j][1] = p01 * (g01 - db) * p.scale;
        dpt[j][2] = p10 * (g10 - da) * p.scale;
        dpt[j][3] = p11 * (g11 - db) * p.scale;
      }
      T::mma_wv(dv, st, sdO, qc * kCW, rem, lane);  // dv += P~^T d_ctx
      T::mma_wv(dk, dpt, sQ, qc * kCW, rem, lane);  // dk += dS^T q
    }
    T::store(dk, lane, p.dk + b * p.dkv_img + h * HD, p.lddkv, k0, Nk);
    T::store(dv, lane, p.dv + b * p.dkv_img + h * HD, p.lddkv, k0, Nk);
  }
}

// Forward with the log-sum-exp output and dropout on the probabilities (training when the tcgen05
// kernel does not apply: dropout, more than 128 queries or 256 keys): flash-style, one pass over
// the keys in chunks of 32 with a running row maximum; a warp owns 16 query rows.
template <int HD>
__global__ void __launch_bounds__(kThreads, 1)
attn_xmma_fwd_kernel(const XmParams p, __nv_bfloat16* __restrict__ out, float* __restrict__ lse_out) {
  using T = Tile<HD>;
  extern __shared__ __align__(128) uint8_t smem[];
  const int Nq = p.Nq, Nk = p.Nk;
  const uint32_t sQ = smem_u32(smem);
  const uint32_t sK = sQ + p.Nq16 * T::kPitch;
  const uint32_t sV = sK + p.Nk16 * T::kPitch;
  const int bh = blockIdx.x, b = bh / p.H, h = bh - b * p.H;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = lane >> 2, t = lane & 3;
  const bool dropping = p.drop.thresh != 0u;
  T::stage(sQ, p.q + b * p.q_img + h * HD, p.ldq, Nq, p.Nq16);
  T::stage(sK, p.k + b * p.kv_img + h * HD, p.ldkv, Nk, p.Nk16);
  T::stage(sV, p.v + b * p.kv_img + h * HD, p.ldkv, Nk, p.Nk16);
  asm volatile("cp.async.commit_group;" ::: "memory");
  asm volatile("cp.async.wait_group 0;" ::: "memory");
  __syncthreads();
  const float c = p.scale * kLog2e;
  for (int qt = warp; qt * 16 < Nq; qt += kWarps) {
    const int q0 = qt * 16;
    uint32_t qa[T::kKS][4];
    T::load_a(sQ, q0, lane, qa);
    float m0 = -INFINITY, m1 = -INFINITY, l0 = 0.f, l1 = 0.f;   // base-2 units
    float o[HD / 8][4];
#pragma unroll
    for (int j = 0; j < HD / 8; ++j) o[j][0] = o[j][1] = o[j][2] = o[j][3] = 0.f;
    for (int kc = 0; kc * kCW < Nk; ++kc) {
      const int rem = Nk - kc * kCW;
      float s[kCW / 8][4];
      T::mma_nt(s, qa, sK, kc * kCW, rem, lane);
      float cm0 = -INFINITY, cm1 = -INFINITY;
#pragma unroll
      for (int j = 0; j < kCW / 8; ++j) {
        const int k0 = j * 8 + t * 2;
        s[j][0] = (k0 < rem) ? s[j][0] * c : -INFINITY;
        s[j][1] = (k0 + 1 < rem) ? s[j][1] * c : -INFINITY;
        s[j][2] = (k0 < rem) ? s[j][2] * c : -INFINITY;
        s[j][3] = (k0 + 1 < rem) ? s[j][3] * c : -INFINITY;
        cm0 = fmaxf(cm0, fmaxf(s[j][0], s[j][1]));
        cm1 = fmaxf(cm1, fmaxf(s[j][2], s[j][3]));
      }
      cm0 = fmaxf(cm0, __shfl_xor_sync(0xffffffffu, cm0, 1));
      cm0 = fmaxf(cm0, __shfl_xor_sync(0xffffffffu, cm0, 2));
      cm1 = fmaxf(cm1, __shfl_xor_sync(0xffffffffu, cm1, 1));
      cm1 = fmaxf(cm1, __shfl_xor_sync(0xffffffffu, cm1, 2));
      const float n0 = fmaxf(m0, cm0), n1 = fmaxf(m1, cm1);   // finite: a chunk has a valid key
      const float a0 = ex2_approx(m0 - n0), a1 = ex2_approx(m1 - n1);
      m0 = n0;
      m1 = n1;
      float ps0 = 0.f, ps1 = 0.f;
#pragma unroll
      for (int j = 0; j < kCW / 8; ++j) {
        const int key = kc * kCW + j * 8 + t * 2;
        float p00 = ex2_approx(s[j][0] - n0), p01 = ex2_approx(s[j][1] - n0);
        float p10 = ex2_approx(s[j][2] - n1), p11 = ex2_approx(s[j][3] - n1);
        ps0 += p00 + p01;
        ps1 += p10 + p11;
        if (dropping) {   // dropout follows the softmax normalisation: the row sum keeps every term
          p00 = keep_x(p, bh, q0 + g, key) ? p00 * p.drop.scale : 0.f;
          p01 = keep_x(p, bh, q0 + g, key + 1) ? p01 * p.drop.scale : 0.f;
          p10 = keep_x(p, bh, q0 + g + 8, key) ? p10 * p.drop.scale : 0.f;
          p11 = keep_x(p, bh, q0 + g + 8, key + 1) ? p11 * p.drop.scale : 0.f;
        }
        s[j][0] = p00;
        s[j][1] = p01;
        s[j][2] = p10;
        s[j][3] = p11;
      }
      l0 = l0 * a0 + ps0;
      l1 = l1 * a1 + ps1;
#pragma unroll
      for (int j = 0; j < HD / 8; ++j) {
        o[j][0] *= a0;
        o[j][1] *= a0;
        o[j][2] *= a1;
        o[j][3] *= a1;
      }
      T::mma_wv(o, s, sV, kc * kCW, rem, lane);
    }
    l0 += __shfl_xor_sync(0xffffffffu, l0, 1);
    l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
    l1 += __shfl_xor_sync(0xffffffffu, l1, 1);
    l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
    const float i0 = 1.f / l0, i1 = 1.f / l1;
#pragma unroll
    for (int j = 0; j < HD / 8; ++j) {
      o[j][0] *= i0;
      o[j][1] *= i0;
      o[j][2] *= i1;
      o[j][3] *= i1;
    }
    T::store(o, lane, out + b * p.ctx_img + h * HD, p.ldc, q0, Nq);
    if (lse_out != nullptr && t == 0) {
      constexpr float kLn2 = 0.69314718055994530942f;
      if (q0 + g < Nq) lse_out[static_cast<long long>(bh) * Nq + q0 + g] = (m0 + log2f(l0)) * kLn2;
      if (q0 + g + 8 < Nq) lse_out[static_cast<long long>(bh) * Nq + q0 + g + 8] = (m1 + log2f(l1)) * kLn2;
    }
  }
}

template <int HD>
int launch_xmma_fwd(const XmParams& p, int B, void* out, float* lse, cudaStream_t stream) {
  const size_t smem = static_cast<size_t>(p.Nq16 + 2 * p.Nk16) * Tile<HD>::kPitch;
  VITK_TRY(opt_in_smem<attn_xmma_fwd_kernel<HD>>(232448, "attn_xmma_fwd_kernel"));
  attn_xmma_fwd_kernel<HD><<<B * p.H, kThreads, smem, stream>>>(p, static_cast<__nv_bfloat16*>(out), lse);
  VITK_CHECK_LAUNCH("attn_xmma_fwd_kernel");
  return VITK_OK;
}

template <int HD>
size_t xmma_smem(int Nq16, int Nk16) {
  return static_cast<size_t>(2 * Nq16 + 2 * Nk16) * Tile<HD>::kPitch + 2 * static_cast<size_t>(Nq16 + 32) * 4;
}

template <int HD>
int launch_xmma(const XmParams& p, int B, cudaStream_t stream) {
  const size_t smem = xmma_smem<HD>(p.Nq16, p.Nk16);
  VITK_TRY(opt_in_smem<attn_xmma_bwd_kernel<HD>>(232448, "attn_xmma_bwd_kernel"));
  attn_xmma_bwd_kernel<HD><<<B * p.H, kThreads, smem, stream>>>(p);
  VITK_CHECK_LAUNCH("attn_xmma_bwd_kernel");
  return VITK_OK;
}

}  // namespace

bool attention_xmma_fits(int Nq, int Nk, int hd) {
  if (hd < 16 || hd > 128 || hd % 16 != 0) return false;
  if (Nq <= 0 || Nk <= 0) return false;
  const int Nq16 = (Nq + 15) & ~15, Nk16 = (Nk + 15) & ~15;
  const size_t smem = static_cast<size_t>(2 * Nq16 + 2 * Nk16) * (hd * 2 + 16) +
                      2 * static_cast<size_t>(Nq16 + 32) * 4;
  return smem <= 232448;
}

int attention_xmma_bwd(const AttnXSrc& s, const void* ctx, const void* dctx, long long ctx_img,
                       int ldc, const float* lse, void* dq, long long dq_img, int lddq, void* dk,
                       void* dv, long long dkv_img, int lddkv, int B, int Nq, int Nk, int H, int hd,
                       cudaStream_t stream, const DropParams* drop) {
  VITK_REQUIRE(s.q && s.k && s.v && ctx && dctx && lse && dq && dk && dv,
               "attention_bwd (tensor-core, generic sources): null operand");
  VITK_REQUIRE(B > 0 && H > 0 && attention_xmma_fits(Nq, Nk, hd),
               "attention_bwd (tensor-core, generic sources): head_dim a multiple of 16 up to 128 and queries + "
               "keys within shared memory (got %d x %d, head_dim %d)", Nq, Nk, hd);
  // 16-byte cp.async / uint4 reads and 4-byte paired stores
  VITK_REQUIRE(s.ldq % 8 == 0 && s.ldkv % 8 == 0 && ldc % 8 == 0 && lddq % 2 == 0 && lddkv % 2 == 0 &&
                   s.q_img % 8 == 0 && s.kv_img % 8 == 0 && ctx_img % 8 == 0 && dq_img % 2 == 0 &&
                   dkv_img % 2 == 0,
               "attention_bwd (tensor-core, generic sources): pitches must be multiples of 8 elements");
  VITK_REQUIRE(drop == nullptr || drop->thresh == 0u ||
                   static_cast<long long>(B) * H * Nq * ((Nk + 15) & ~15) < (1ll << 32),
               "attention dropout: batch * heads * queries * keys must stay below 2^32");
  XmParams p{};
  p.q = static_cast<const __nv_bfloat16*>(s.q);
  p.k = static_cast<const __nv_bfloat16*>(s.k);
  p.v = static_cast<const __nv_bfloat16*>(s.v);
  p.ctx = static_cast<const __nv_bfloat16*>(ctx);
  p.dctx = static_cast<const __nv_bfloat16*>(dctx);
  p.dq = static_cast<__nv_bfloat16*>(dq);
  p.dk = static_cast<__nv_bfloat16*>(dk);
  p.dv = static_cast<__nv_bfloat16*>(dv);
  p.lse = lse;
  p.q_img = s.q_img; p.kv_img = s.kv_img; p.ctx_img = ctx_img; p.dq_img = dq_img; p.dkv_img = dkv_img;
  p.ldq = s.ldq; p.ldkv = s.ldkv; p.ldc = ldc; p.lddq = lddq; p.lddkv = lddkv;
  p.Nq = Nq; p.Nk = Nk; p.Nq16 = (Nq + 15) & ~15; p.Nk16 = (Nk + 15) & ~15; p.H = H;
  p.Nkp = (Nk + 15) & ~15;
  p.scale = 1.0f / sqrtf(static_cast<float>(hd));
  if (drop != nullptr) p.drop = *drop;
  ProfileScope prof(PROF_ATTN, attention_flops(B, H, Nq, Nk, hd, true), stream);
  switch (hd) {
    case 16: return launch_xmma<16>(p, B, stream);
    case 32: return launch_xmma<32>(p, B, stream);
    case 48: return launch_xmma<48>(p, B, stream);
    case 64: return launch_xmma<64>(p, B, stream);
    case 80: return launch_xmma<80>(p, B, stream);
    case 96: return launch_xmma<96>(p, B, stream);
    case 112: return launch_xmma<112>(p, B, stream);
    default: return launch_xmma<128>(p, B, stream);
  }
}

int attention_xmma_fwd(const AttnXSrc& s, void* ctx, long long ctx_img, int ldc, float* lse, int B,
                       int Nq, int Nk, int H, int hd, cudaStream_t stream, const DropParams* drop) {
  VITK_REQUIRE(s.q && s.k && s.v && ctx, "attention (tensor-core, generic sources): null operand");
  VITK_REQUIRE(B > 0 && H > 0 && attention_xmma_fits(Nq, Nk, hd),
               "attention (tensor-core, generic sources): head_dim a multiple of 16 up to 128 and queries + keys "
               "within shared memory (got %d x %d, head_dim %d)", Nq, Nk, hd);
  VITK_REQUIRE(s.ldq % 8 == 0 && s.ldkv % 8 == 0 && ldc % 2 == 0 && s.q_img % 8 == 0 &&
                   s.kv_img % 8 == 0 && ctx_img % 2 == 0,
               "attention (tensor-core, generic sources): pitches must be multiples of 8 elements");
  VITK_REQUIRE(drop == nullptr || drop->thresh == 0u ||
                   static_cast<long long>(B) * H * Nq * ((Nk + 15) & ~15) < (1ll << 32),
               "attention dropout: batch * heads * queries * keys must stay below 2^32");
  XmParams p{};
  p.q = static_cast<const __nv_bfloat16*>(s.q);
  p.k = static_cast<const __nv_bfloat16*>(s.k);
  p.v = static_cast<const __nv_bfloat16*>(s.v);
  p.q_img = s.q_img; p.kv_img = s.kv_img; p.ctx_img = ctx_img;
  p.ldq = s.ldq; p.ldkv = s.ldkv; p.ldc = ldc;
  p.Nq = Nq; p.Nk = Nk; p.Nq16 = (Nq + 15) & ~15; p.Nk16 = (Nk + 15) & ~15; p.H = H;
  p.Nkp = (Nk + 15) & ~15;
  p.scale = 1.0f / sqrtf(static_cast<float>(hd));
  if (drop != nullptr) p.drop = *drop;
  ProfileScope prof(PROF_ATTN, attention_flops(B, H, Nq, Nk, hd), stream);
  switch (hd) {
    case 16: return launch_xmma_fwd<16>(p, B, ctx, lse, stream);
    case 32: return launch_xmma_fwd<32>(p, B, ctx, lse, stream);
    case 48: return launch_xmma_fwd<48>(p, B, ctx, lse, stream);
    case 64: return launch_xmma_fwd<64>(p, B, ctx, lse, stream);
    case 80: return launch_xmma_fwd<80>(p, B, ctx, lse, stream);
    case 96: return launch_xmma_fwd<96>(p, B, ctx, lse, stream);
    case 112: return launch_xmma_fwd<112>(p, B, ctx, lse, stream);
    default: return launch_xmma_fwd<128>(p, B, ctx, lse, stream);
  }
}

}  // namespace vitk
