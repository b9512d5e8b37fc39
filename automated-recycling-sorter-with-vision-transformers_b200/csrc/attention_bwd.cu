// Backward of the attention core (autograd of train.py:543-549 triggered at train.py:1455):
// given d_ctx, the packed qkv activation, ctx and the saved log-sum-exp, produce d_qkv.
//   P  = exp(q k^T * scale - lse)           dP = d_ctx v^T           Drow = rowsum(d_ctx * ctx)
//   dS = P * (dP - Drow) * scale            dq = dS k     dk = dS^T q     dv = P^T d_ctx
// One CTA per (image, head); q, k, v, d_ctx of the head live in swizzled shared memory.  Two
// passes avoid cross-warp reductions: a query-tile pass (dq) and a key-tile pass (dk, dv), each
// recomputing its 16 x 64 score blocks with bf16 m16n8k16 tensor-core MMAs (fp32 accumulate).
// N <= 256 tokens, head_dim 64.
#include <cuda_bf16.h>

#include <mutex>

#include "common.h"
#include "ptx.cuh"
#include "rowops.cuh"
#include "train_ops.cuh"

namespace vitk {
using namespace ptx;

namespace {

constexpr int kWarps = 8;
constexpr int kThreads = kWarps * 32;
constexpr float kLog2e = 1.44269504088896340736f;

__device__ __forceinline__ void mma16816(float (&c)[4], const uint32_t (&a)[4], uint32_t b0,
                                         uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, "
      "{%0,%1,%2,%3};"
      : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ void ldsm4(uint32_t addr, uint32_t& r0, uint32_t& r1, uint32_t& r2,
                                      uint32_t& r3) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3)
               : "r"(addr));
}
__device__ __forceinline__ void ldsm4t(uint32_t addr, uint32_t& r0, uint32_t& r1, uint32_t& r2,
                                       uint32_t& r3) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3)
               : "r"(addr));
}
__device__ __forceinline__ void cp16(uint32_t dst, const void* src, bool valid) {
  const int sz = valid ? 16 : 0;
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(sz)
               : "memory");
}
// swizzled address of 16-byte chunk `ch` of 128-byte row `row`
__device__ __forceinline__ uint32_t swz(uint32_t base, int row, int ch) {
  return base + row * 128 + ((ch ^ (row & 7)) << 4);
}

// A fragments (m16 x k64) of rows [row0, row0+16) of a swizzled [rows x 64] bf16 tile.
__device__ __forceinline__ void load_a_frags(uint32_t base, int row0, int lane, uint32_t (&a)[4][4]) {
  const int r = row0 + (lane & 7) + ((lane >> 3) & 1) * 8;
#pragma unroll
  for (int kk = 0; kk < 4; ++kk) ldsm4(swz(base, r, kk * 2 + (lane >> 4)), a[kk][0], a[kk][1], a[kk][2], a[kk][3]);
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
        ldsm4(swz(sB, row, (lane >> 3) + 4 * half), b0, b1, b2, b3);
        mma16816(acc[j], a[2 * half], b0, b1);
        mma16816(acc[j], a[2 * half + 1], b2, b3);
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
        ldsm4t(swz(sB, row, 2 * jj + (mi >> 1)), v0, v1, v2, v3);
        mma16816(out[2 * jj], pa, v0, v1);
        mma16816(out[2 * jj + 1], pa, v2, v3);
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
    cp16(sQ + off, qbase + r * D3 + ch * 8, valid);
    cp16(sK + off, qbase + r * D3 + D + ch * 8, valid);
    cp16(sV + off, qbase + r * D3 + 2 * D + ch * 8, valid);
    cp16(sdO + off, dobase + r * D + ch * 8, valid);
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

int attention_impl();  // attention.cu: 0 auto, 1 mma.sync kernels, 2 tcgen05 kernels

int attention_bwd(const void* qkv, const void* ctx, const void* dctx, const float* lse, void* dqkv,
                  int B, int N, int H, int hd, cudaStream_t stream, const DropParams* drop,
                  float* dbias) {
  VITK_REQUIRE(qkv && ctx && dctx && lse && dqkv, "attention_bwd: null operand");
  const bool dropping = drop != nullptr && drop->thresh != 0u;
  if ((attention_impl() != 1 || dropping) && hd == 64 && N <= 256 && device_cc() >= 100) {
    if (attention_bwd_tc2_fits(N, H, dbias != nullptr))
      return attention_bwd_tc2(qkv, ctx, dctx, lse, dqkv, B, N, H, hd, stream, drop, dbias);
    return attention_bwd_tc(qkv, ctx, dctx, lse, dqkv, B, N, H, hd, stream, drop, dbias);
  }
  // other head sizes, longer sequences, dropout without the tcgen05 kernel: CUDA-core kernel
  if (hd != 64 || N > 256 || dropping) {
    if (attention_impl() != 1 && attention_xmma_bwd_applicable(N, N, hd)) {
      // tensor cores (mma.sync) on the packed activation: q, k, v are column blocks of qkv
      const __nv_bfloat16* p = static_cast<const __nv_bfloat16*>(qkv);
      __nv_bfloat16* dp = static_cast<__nv_bfloat16*>(dqkv);
      const int D = H * hd;
      const long long img = static_cast<long long>(N) * 3 * D, cimg = static_cast<long long>(N) * D;
      const AttnXSrc src{p, img, 3 * D, p + D, p + 2 * D, img, 3 * D};
      VITK_TRY(attention_xmma_bwd(src, ctx, dctx, cimg, D, lse, dp, img, 3 * D, dp + D, dp + 2 * D, img,
                                  3 * D, B, N, N, H, hd, stream, drop));
      if (dbias != nullptr) return colsum_bf16(dqkv, 3ll * D, B * N, 3 * D, dbias, stream);
      return VITK_OK;
    }
    return attention_gen_bwd(qkv, ctx, dctx, lse, dqkv, B, N, H, hd, stream, drop, dbias);
  }
  VITK_REQUIRE(B > 0 && H > 0 && N > 0, "attention_bwd: bad shape");
  const int Nkv = (N + 15) & ~15;
  const size_t smem = 4 * static_cast<size_t>(Nkv) * 128 + 2 * 256 * sizeof(float);
  static std::once_flag once;
  static cudaError_t attr_err = cudaSuccess;
  std::call_once(once, [&] {
    attr_err = cudaFuncSetAttribute(attn_bwd_hd64_kernel,
                                    cudaFuncAttributeMaxDynamicSharedMemorySize, 232448);
  });
  if (attr_err != cudaSuccess)
    return set_error(VITK_ERR_CUDA, "cudaFuncSetAttribute(attention_bwd) failed: %s",
                     cudaGetErrorString(attr_err));
  const float scale = 1.0f / sqrtf(static_cast<float>(hd));
  ProfileScope prof(PROF_ATTN, 10.0 * B * H * static_cast<double>(N) * N * hd, stream);
  attn_bwd_hd64_kernel<<<B * H, kThreads, smem, stream>>>(
      static_cast<const __nv_bfloat16*>(qkv), static_cast<const __nv_bfloat16*>(ctx),
      static_cast<const __nv_bfloat16*>(dctx), lse, static_cast<__nv_bfloat16*>(dqkv), N, H, scale);
  VITK_CHECK_LAUNCH("attn_bwd_hd64_kernel");
  if (dbias != nullptr)   // this kernel does not accumulate the bias gradient itself
    return colsum_bf16(dqkv, 3ll * H * hd, B * N, 3 * H * hd, dbias, stream);
  return VITK_OK;
}

}  // namespace vitk
