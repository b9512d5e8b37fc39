// The two head_dim-64 flash kernels on the packed qkv activation: bf16 mma.sync m16n8k16 MMAs
// (fp32 accumulate), one CTA per (image, head), the whole head staged once in shared memory
// (cp.async, XOR-swizzled 128-byte rows).  vitk_attention_set_impl(1) selects them; attention.cu
// also falls back to them where the tcgen05 kernels do not apply.
//
// Forward, ctx = softmax(q k^T / sqrt(hd)) v without materialising the [B,H,N,N] score tensor
// (reference train.py:543-549 materialises it; evaluation.py:66-72): each warp owns 16-query
// tiles and sweeps the keys in blocks of 64 with a warp-level online softmax (running max / sum in
// registers, quad shuffles).  Reads qkv in place (no permute copies) and writes ctx already in
// [B, N, H*hd] order (the reference's transpose(1,2).reshape is free).
//
// Backward (autograd of train.py:543-549 triggered at train.py:1455): given d_ctx, qkv, ctx and
// the saved log-sum-exp, produce d_qkv.
//   P  = exp(q k^T * scale - lse)           dP = d_ctx v^T           Drow = rowsum(d_ctx * ctx)
//   dS = P * (dP - Drow) * scale            dq = dS k     dk = dS^T q     dv = P^T d_ctx
// q, k, v, d_ctx of the head live in shared memory.  Two passes avoid cross-warp reductions: a
// query-tile pass (dq) and a key-tile pass (dk, dv), each recomputing its 16 x 64 score blocks.
// N <= 256 tokens.
#include <cuda_bf16.h>

#include "attention_kernels.cuh"
#include "common.h"
#include "ptx.cuh"

namespace vitk {
using namespace ptx;

namespace {

constexpr int kAttnWarps = 7;
constexpr int kAttnThreads = kAttnWarps * 32;

// hd == 64 only: one K/V row is exactly one 128-byte swizzle row.
__global__ void __launch_bounds__(kAttnThreads, 2)
attn_fwd_hd64_kernel(const __nv_bfloat16* __restrict__ qkv, __nv_bfloat16* __restrict__ ctx,
                     float* __restrict__ lse, int N, int H, float scale) {
  extern __shared__ __align__(128) uint8_t smem[];
  constexpr int HD = 64;
  const int Nkv = (N + 15) & ~15;
  const uint32_t sK = smem_u32(smem);
  const uint32_t sV = sK + Nkv * 128;
  const uint32_t sO = sV + Nkv * 128;  // kAttnWarps * 2048 bytes of output staging

  const int b = blockIdx.x / H;
  const int h = blockIdx.x - b * H;
  const int D = H * HD;
  const int D3 = 3 * D;
  const __nv_bfloat16* base = qkv + static_cast<size_t>(b) * N * D3 + h * HD;

  const int tid = threadIdx.x;
  const int warp = tid >> 5;
  const int lane = tid & 31;
  const int g = lane >> 2;  // fragment row
  const int t = lane & 3;   // fragment column pair

  // ---- stage K and V (all keys of this head) into swizzled shared memory
  for (int idx = tid; idx < Nkv * 8; idx += kAttnThreads) {
    const int row = idx >> 3;
    const int ch = idx & 7;
    const bool valid = row < N;
    const __nv_bfloat16* src = base + static_cast<size_t>(valid ? row : 0) * D3 + ch * 8;
    const uint32_t off = row * 128 + ((ch ^ (row & 7)) << 4);
    cp_async_16(sK + off, src + D, valid);
    cp_async_16(sV + off, src + 2 * D, valid);
  }
  asm volatile("cp.async.commit_group;" ::: "memory");
  asm volatile("cp.async.wait_group 0;" ::: "memory");
  __syncthreads();

  const float c = scale * kLog2e;  // softmax in base 2
  const uint32_t sOw = sO + warp * 2048;

  for (int qt = warp; qt * 16 < N; qt += kAttnWarps) {
    const int q0 = qt * 16;
    const int r0 = q0 + g, r1 = r0 + 8;
    // ---- Q fragments straight from global (each 128-byte query row is consumed whole)
    uint32_t qa[4][4];
    {
      const uint32_t* p0 = reinterpret_cast<const uint32_t*>(base + static_cast<size_t>(r0) * D3);
      const uint32_t* p1 = reinterpret_cast<const uint32_t*>(base + static_cast<size_t>(r1) * D3);
#pragma unroll
      for (int kk = 0; kk < 4; ++kk) {
        const int w = kk * 8 + t;  // 32-bit word index of d = kk*16 + 2t
        qa[kk][0] = (r0 < N) ? __ldg(p0 + w) : 0u;
        qa[kk][1] = (r1 < N) ? __ldg(p1 + w) : 0u;
        qa[kk][2] = (r0 < N) ? __ldg(p0 + w + 4) : 0u;
        qa[kk][3] = (r1 < N) ? __ldg(p1 + w + 4) : 0u;
      }
    }
    float o[8][4];
#pragma unroll
    for (int j = 0; j < 8; ++j) o[j][0] = o[j][1] = o[j][2] = o[j][3] = 0.f;
    float m0 = -INFINITY, m1 = -INFINITY, l0 = 0.f, l1 = 0.f;

    for (int kb = 0; kb * 64 < N; ++kb) {
      const int rem = N - kb * 64;  // valid keys from the start of this block
      float s[8][4];
      // ---- S = Q K^T for 64 keys
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        if (j * 8 < rem) {
          s[j][0] = s[j][1] = s[j][2] = s[j][3] = 0.f;
          const int key = kb * 64 + j * 8 + (lane & 7);
#pragma unroll
          for (int half = 0; half < 2; ++half) {
            const int ch = (lane >> 3) + 4 * half;
            uint32_t k0, k1, k2, k3;
            ldmatrix_x4(sK + key * 128 + ((ch ^ (key & 7)) << 4), k0, k1, k2, k3);
            mma_m16n8k16(s[j], qa[2 * half], k0, k1);
            mma_m16n8k16(s[j], qa[2 * half + 1], k2, k3);
          }
        } else {
          s[j][0] = s[j][1] = s[j][2] = s[j][3] = -INFINITY;
        }
      }
      if (rem < 64) {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const int k0 = j * 8 + t * 2;
          if (k0 >= rem) s[j][0] = s[j][2] = -INFINITY;
          if (k0 + 1 >= rem) s[j][1] = s[j][3] = -INFINITY;
        }
      }
      // ---- online softmax update
      float mx0 = -INFINITY, mx1 = -INFINITY;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        mx0 = fmaxf(mx0, fmaxf(s[j][0], s[j][1]));
        mx1 = fmaxf(mx1, fmaxf(s[j][2], s[j][3]));
      }
      mx0 = quad_max(mx0);
      mx1 = quad_max(mx1);
      const float mn0 = fmaxf(m0, mx0), mn1 = fmaxf(m1, mx1);
      const float a0 = exp2f((m0 - mn0) * c), a1 = exp2f((m1 - mn1) * c);
      m0 = mn0;
      m1 = mn1;
      const float mc0 = mn0 * c, mc1 = mn1 * c;
      float ps0 = 0.f, ps1 = 0.f;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        s[j][0] = exp2f(fmaf(s[j][0], c, -mc0));
        s[j][1] = exp2f(fmaf(s[j][1], c, -mc0));
        s[j][2] = exp2f(fmaf(s[j][2], c, -mc1));
        s[j][3] = exp2f(fmaf(s[j][3], c, -mc1));
        ps0 += s[j][0] + s[j][1];
        ps1 += s[j][2] + s[j][3];
      }
      l0 = l0 * a0 + ps0;
      l1 = l1 * a1 + ps1;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        o[j][0] *= a0;
        o[j][1] *= a0;
        o[j][2] *= a1;
        o[j][3] *= a1;
      }
      // ---- O += P V
#pragma unroll
      for (int kk = 0; kk < 4; ++kk) {
        if (kk * 16 < rem) {
          uint32_t pa[4];
          pa[0] = pack_bf16x2(s[2 * kk][0], s[2 * kk][1]);
          pa[1] = pack_bf16x2(s[2 * kk][2], s[2 * kk][3]);
          pa[2] = pack_bf16x2(s[2 * kk + 1][0], s[2 * kk + 1][1]);
          pa[3] = pack_bf16x2(s[2 * kk + 1][2], s[2 * kk + 1][3]);
          const int mi = lane >> 3;
          const int key = kb * 64 + kk * 16 + (mi & 1) * 8 + (lane & 7);
#pragma unroll
          for (int jj = 0; jj < 4; ++jj) {
            const int ch = 2 * jj + (mi >> 1);
            uint32_t v0, v1, v2, v3;
            ldmatrix_x4_trans(sV + key * 128 + ((ch ^ (key & 7)) << 4), v0, v1, v2, v3);
            mma_m16n8k16(o[2 * jj], pa, v0, v1);
            mma_m16n8k16(o[2 * jj + 1], pa, v2, v3);
          }
        }
      }
    }

    // ---- finalise: divide by the row sum, stage through smem, 16-byte coalesced stores
    l0 = quad_sum(l0);
    l1 = quad_sum(l1);
    const float inv0 = 1.f / l0, inv1 = 1.f / l1;
    __syncwarp();
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const uint32_t w0 = pack_bf16x2(o[j][0] * inv0, o[j][1] * inv0);
      const uint32_t w1 = pack_bf16x2(o[j][2] * inv1, o[j][3] * inv1);
      const uint32_t a_lo = sOw + g * 128 + ((j ^ (g & 7)) << 4) + t * 4;
      const uint32_t a_hi = sOw + (g + 8) * 128 + ((j ^ ((g + 8) & 7)) << 4) + t * 4;
      asm volatile("st.shared.b32 [%0], %1;" ::"r"(a_lo), "r"(w0) : "memory");
      asm volatile("st.shared.b32 [%0], %1;" ::"r"(a_hi), "r"(w1) : "memory");
    }
    __syncwarp();
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int idx = lane + 32 * i;
      const int row = idx >> 3, ch = idx & 7;
      if (q0 + row < N) {
        uint4 val;
        const uint32_t a = sOw + row * 128 + ((ch ^ (row & 7)) << 4);
        asm volatile("ld.shared.v4.b32 {%0,%1,%2,%3}, [%4];"
                     : "=r"(val.x), "=r"(val.y), "=r"(val.z), "=r"(val.w)
                     : "r"(a)
                     : "memory");
        *reinterpret_cast<uint4*>(ctx + (static_cast<size_t>(b) * N + q0 + row) * D + h * HD +
                                  ch * 8) = val;
      }
    }
    if (lse != nullptr && t == 0) {
      float* lrow = lse + (static_cast<size_t>(b) * H + h) * N;
      if (r0 < N) lrow[r0] = m0 * scale + logf(l0);
      if (r1 < N) lrow[r1] = m1 * scale + logf(l1);
    }
  }
}

constexpr int kWarps = 8;
constexpr int kThreads = kWarps * 32;

// swizzled address of 16-byte chunk `ch` of 128-byte row `row`
__device__ __forceinline__ uint32_t swz(uint32_t base, int row, int ch) {
  return base + row * 128 + ((ch ^ (row & 7)) << 4);
}

// A fragments (m16 x k64) of rows [row0, row0+16) of a swizzled [rows x 64] bf16 tile.
__device__ __forceinline__ void load_a_frags(uint32_t base, int row0, int lane, uint32_t (&a)[4][4]) {
  const int r = row0 + (lane & 7) + ((lane >> 3) & 1) * 8;
#pragma unroll
  for (int kk = 0; kk < 4; ++kk) ldmatrix_x4(swz(base, r, kk * 2 + (lane >> 4)), a[kk][0], a[kk][1], a[kk][2], a[kk][3]);
}

// acc[16 x 64] = A[16 x 64(d)] * Brows[row0 .. row0+64)[64(d)]^T   ("score-like" product);
// only the first `rem` B rows are valid, 8-row groups beyond them are skipped (acc = 0).
__device__ __forceinline__ void mma_nt(float (&acc)[8][4], const uint32_t (&a)[4][4], uint32_t sB,
                                       int row0, int rem, int lane) {
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    acc[j][0] = acc[j][1] = acc[j][2] = acc[j][3] = 0.f;
    if (j * 8 < rem) {
      const int row = row0 + j * 8 + (lane & 7);
#pragma unroll
      for (int half = 0; half < 2; ++half) {
        uint32_t b0, b1, b2, b3;
        ldmatrix_x4(swz(sB, row, (lane >> 3) + 4 * half), b0, b1, b2, b3);
        mma_m16n8k16(acc[j], a[2 * half], b0, b1);
        mma_m16n8k16(acc[j], a[2 * half + 1], b2, b3);
      }
    }
  }
}

// out[16 x 64(d)] += P[16 x 64(rows)] * Brows[row0 .. row0+64)[64(d)]; P given as fp32 C fragments.
__device__ __forceinline__ void mma_pv(float (&out)[8][4], const float (&p)[8][4], uint32_t sB,
                                       int row0, int rem, int lane) {
#pragma unroll
  for (int kk = 0; kk < 4; ++kk) {
    if (kk * 16 < rem) {
      uint32_t pa[4];
      pa[0] = pack_bf16x2(p[2 * kk][0], p[2 * kk][1]);
      pa[1] = pack_bf16x2(p[2 * kk][2], p[2 * kk][3]);
      pa[2] = pack_bf16x2(p[2 * kk + 1][0], p[2 * kk + 1][1]);
      pa[3] = pack_bf16x2(p[2 * kk + 1][2], p[2 * kk + 1][3]);
      const int mi = lane >> 3;
      const int row = row0 + kk * 16 + (mi & 1) * 8 + (lane & 7);
#pragma unroll
      for (int jj = 0; jj < 4; ++jj) {
        uint32_t v0, v1, v2, v3;
        ldmatrix_x4_trans(swz(sB, row, 2 * jj + (mi >> 1)), v0, v1, v2, v3);
        mma_m16n8k16(out[2 * jj], pa, v0, v1);
        mma_m16n8k16(out[2 * jj + 1], pa, v2, v3);
      }
    }
  }
}

// 16 x 64 fp32 tile -> bf16 rows of `dst` (row pitch ld elements), straight from the MMA
// accumulator layout: every lane writes bf16 pairs, 16 contiguous bytes per row and instruction.
// (d_qkv is ~1 % of this kernel's traffic; not staging it frees 16 KB of shared memory so that two
// CTAs are resident per SM.)
__device__ __forceinline__ void store_tile(const float (&o)[8][4], int lane, __nv_bfloat16* dst,
                                           long long ld, int row0, int row_limit) {
  const int g = lane >> 2, t = lane & 3;
  const int r0 = row0 + g, r1 = row0 + g + 8;
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    if (r0 < row_limit)
      *reinterpret_cast<uint32_t*>(dst + r0 * ld + j * 8 + t * 2) = pack_bf16x2(o[j][0], o[j][1]);
    if (r1 < row_limit)
      *reinterpret_cast<uint32_t*>(dst + r1 * ld + j * 8 + t * 2) = pack_bf16x2(o[j][2], o[j][3]);
  }
}

__global__ void __launch_bounds__(kThreads, 1)
attn_bwd_hd64_kernel(const __nv_bfloat16* __restrict__ qkv, const __nv_bfloat16* __restrict__ ctx,
                     const __nv_bfloat16* __restrict__ dctx, const float* __restrict__ lse,
                     __nv_bfloat16* __restrict__ dqkv, int N, int H, float scale) {
  extern __shared__ __align__(128) uint8_t smem[];
  const int Nkv = (N + 15) & ~15;
  const uint32_t sQ = smem_u32(smem);
  const uint32_t sK = sQ + Nkv * 128;
  const uint32_t sV = sK + Nkv * 128;
  const uint32_t sdO = sV + Nkv * 128;
  float* sLse = reinterpret_cast<float*>(smem + 4 * Nkv * 128);
  float* sD = sLse + 256;

  const int b = blockIdx.x / H;
  const int h = blockIdx.x - b * H;
  const int D = H * 64;
  const long long D3 = 3ll * D;
  const __nv_bfloat16* qbase = qkv + static_cast<long long>(b) * N * D3 + h * 64;
  const __nv_bfloat16* obase = ctx + static_cast<long long>(b) * N * D + h * 64;
  const __nv_bfloat16* dobase = dctx + static_cast<long long>(b) * N * D + h * 64;
  __nv_bfloat16* dqbase = dqkv + static_cast<long long>(b) * N * D3 + h * 64;

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int g = lane >> 2, t = lane & 3;

  for (int idx = tid; idx < Nkv * 8; idx += kThreads) {
    const int row = idx >> 3, ch = idx & 7;
    const bool valid = row < N;
    const long long r = valid ? row : 0;
    const uint32_t off = row * 128 + ((ch ^ (row & 7)) << 4);
    cp_async_16(sQ + off, qbase + r * D3 + ch * 8, valid);
    cp_async_16(sK + off, qbase + r * D3 + D + ch * 8, valid);
    cp_async_16(sV + off, qbase + r * D3 + 2 * D + ch * 8, valid);
    cp_async_16(sdO + off, dobase + r * D + ch * 8, valid);
  }
  asm volatile("cp.async.commit_group;" ::: "memory");
  // Drow = rowsum(d_ctx * ctx) and the saved log-sum-exp (base-2 scaled), one row per thread
  for (int r = tid; r < 256; r += kThreads) {
    float dsum = 0.f, l2 = INFINITY;  // rows >= N: P = 2^(-inf) = 0
    if (r < N) {
      const uint4* po = reinterpret_cast<const uint4*>(obase + static_cast<long long>(r) * D);
      const uint4* pd = reinterpret_cast<const uint4*>(dobase + static_cast<long long>(r) * D);
#pragma unroll
      for (int c8 = 0; c8 < 8; ++c8) {
        const uint4 a = __ldg(po + c8), d = __ldg(pd + c8);
        dsum += bf16lo_to_f32(a.x) * bf16lo_to_f32(d.x) + bf16hi_to_f32(a.x) * bf16hi_to_f32(d.x);
        dsum += bf16lo_to_f32(a.y) * bf16lo_to_f32(d.y) + bf16hi_to_f32(a.y) * bf16hi_to_f32(d.y);
        dsum += bf16lo_to_f32(a.z) * bf16lo_to_f32(d.z) + bf16hi_to_f32(a.z) * bf16hi_to_f32(d.z);
        dsum += bf16lo_to_f32(a.w) * bf16lo_to_f32(d.w) + bf16hi_to_f32(a.w) * bf16hi_to_f32(d.w);
      }
      l2 = lse[(static_cast<long long>(b) * H + h) * N + r] * kLog2e;
    }
    sLse[r] = l2;
    sD[r] = dsum;
  }
  asm volatile("cp.async.wait_group 0;" ::: "memory");
  __syncthreads();

  const float c = scale * kLog2e;

  // ================= pass 1: query tiles -> dq =================
  for (int qt = warp; qt * 16 < N; qt += kWarps) {
    const int q0 = qt * 16;
    uint32_t qa[4][4], doa[4][4];
    load_a_frags(sQ, q0, lane, qa);
    load_a_frags(sdO, q0, lane, doa);
    const float l0 = sLse[q0 + g], l1 = sLse[q0 + g + 8];
    const float d0 = sD[q0 + g], d1 = sD[q0 + g + 8];
    float dq[8][4];
#pragma unroll
    for (int j = 0; j < 8; ++j) dq[j][0] = dq[j][1] = dq[j][2] = dq[j][3] = 0.f;
    for (int kb = 0; kb * 64 < N; ++kb) {
      const int rem = N - kb * 64;
      float s[8][4], dp[8][4];
      mma_nt(s, qa, sK, kb * 64, rem, lane);
      mma_nt(dp, doa, sV, kb * 64, rem, lane);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const int k0 = j * 8 + t * 2;
        const float p00 = (k0 < rem) ? ex2_approx(fmaf(s[j][0], c, -l0)) : 0.f;
        const float p01 = (k0 + 1 < rem) ? ex2_approx(fmaf(s[j][1], c, -l0)) : 0.f;
        const float p10 = (k0 < rem) ? ex2_approx(fmaf(s[j][2], c, -l1)) : 0.f;
        const float p11 = (k0 + 1 < rem) ? ex2_approx(fmaf(s[j][3], c, -l1)) : 0.f;
        s[j][0] = p00 * (dp[j][0] - d0) * scale;
        s[j][1] = p01 * (dp[j][1] - d0) * scale;
        s[j][2] = p10 * (dp[j][2] - d1) * scale;
        s[j][3] = p11 * (dp[j][3] - d1) * scale;
      }
      mma_pv(dq, s, sK, kb * 64, rem, lane);
    }
    store_tile(dq, lane, dqbase, D3, q0, N);
  }

  // ================= pass 2: key tiles -> dk, dv =================
  for (int kt = warp; kt * 16 < N; kt += kWarps) {
    const int k0 = kt * 16;
    uint32_t ka[4][4], va[4][4];
    load_a_frags(sK, k0, lane, ka);
    load_a_frags(sV, k0, lane, va);
    const bool row0_ok = (k0 + g) < N, row1_ok = (k0 + g + 8) < N;
    float dk[8][4], dv[8][4];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      dk[j][0] = dk[j][1] = dk[j][2] = dk[j][3] = 0.f;
      dv[j][0] = dv[j][1] = dv[j][2] = dv[j][3] = 0.f;
    }
    for (int qb = 0; qb * 64 < N; ++qb) {
      const int rem = N - qb * 64;
      float st[8][4], dpt[8][4];
      mma_nt(st, ka, sQ, qb * 64, rem, lane);    // S^T  = k q^T
      mma_nt(dpt, va, sdO, qb * 64, rem, lane);  // dP^T = v d_ctx^T
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const int qc = qb * 64 + j * 8 + t * 2;  // query index of this thread's column pair
        const float la = sLse[qc], lb = sLse[qc + 1];  // +inf beyond N -> P = 0
        const float da = sD[qc], db = sD[qc + 1];
        const float p00 = row0_ok ? ex2_approx(fmaf(st[j][0], c, -la)) : 0.f;
        const float p01 = row0_ok ? ex2_approx(fmaf(st[j][1], c, -lb)) : 0.f;
        const float p10 = row1_ok ? ex2_approx(fmaf(st[j][2], c, -la)) : 0.f;
        const float p11 = row1_ok ? ex2_approx(fmaf(st[j][3], c, -lb)) : 0.f;
        st[j][0] = p00;
        st[j][1] = p01;
        st[j][2] = p10;
        st[j][3] = p11;
        dpt[j][0] = p00 * (dpt[j][0] - da) * scale;
        dpt[j][1] = p01 * (dpt[j][1] - db) * scale;
        dpt[j][2] = p10 * (dpt[j][2] - da) * scale;
        dpt[j][3] = p11 * (dpt[j][3] - db) * scale;
      }
      mma_pv(dv, st, sdO, qb * 64, rem, lane);  // dv += P^T d_ctx
      mma_pv(dk, dpt, sQ, qb * 64, rem, lane);  // dk += dS^T q
    }
    store_tile(dk, lane, dqbase + D, D3, k0, N);
    store_tile(dv, lane, dqbase + 2 * D, D3, k0, N);
  }
}

}  // namespace

int attention_fwd_hd64(const void* qkv, void* ctx, float* lse, int B, int N, int H, int hd,
                       cudaStream_t stream) {
  VITK_REQUIRE(B > 0 && N > 0 && H > 0, "attention: bad shape B=%d N=%d H=%d", B, N, H);
  VITK_REQUIRE(hd == 64, "attention: head_dim %d unsupported by the bf16 kernel (needs 64)", hd);
  const int Nkv = (N + 15) & ~15;
  const size_t smem = static_cast<size_t>(Nkv) * 256 + kAttnWarps * 2048;
  VITK_REQUIRE(smem <= 232448, "attention: N=%d keys do not fit in shared memory", N);
  VITK_TRY(opt_in_smem<attn_fwd_hd64_kernel>(232448, "attn_fwd_hd64_kernel"));
  const float scale = 1.0f / sqrtf(static_cast<float>(hd));
  ProfileScope prof(PROF_ATTN, attention_flops(B, H, N, N, hd), stream);
  attn_fwd_hd64_kernel<<<B * H, kAttnThreads, smem, stream>>>(
      static_cast<const __nv_bfloat16*>(qkv), static_cast<__nv_bfloat16*>(ctx), lse, N, H, scale);
  VITK_CHECK_LAUNCH("attn_fwd_hd64_kernel");
  return VITK_OK;
}

int attention_bwd_hd64(const void* qkv, const void* ctx, const void* dctx, const float* lse,
                       void* dqkv, int B, int N, int H, int hd, cudaStream_t stream) {
  VITK_REQUIRE(B > 0 && H > 0 && N > 0, "attention_bwd: bad shape");
  const int Nkv = (N + 15) & ~15;
  const size_t smem = 4 * static_cast<size_t>(Nkv) * 128 + 2 * 256 * sizeof(float);
  VITK_TRY(opt_in_smem<attn_bwd_hd64_kernel>(232448, "attn_bwd_hd64_kernel"));
  const float scale = 1.0f / sqrtf(static_cast<float>(hd));
  ProfileScope prof(PROF_ATTN, attention_flops(B, H, N, N, hd, true), stream);
  attn_bwd_hd64_kernel<<<B * H, kThreads, smem, stream>>>(
      static_cast<const __nv_bfloat16*>(qkv), static_cast<const __nv_bfloat16*>(ctx),
      static_cast<const __nv_bfloat16*>(dctx), lse, static_cast<__nv_bfloat16*>(dqkv), N, H, scale);
  VITK_CHECK_LAUNCH("attn_bwd_hd64_kernel");
  return VITK_OK;
}

}  // namespace vitk
