// softmax(q k^T / sqrt(hd)) v with separate query and key/value sources and head_dim 32 / 64 / 96 /
// 128: the attention of the detection head's decoder layers (self-attention over the object
// queries and cross-attention onto the encoder tokens, nn.MultiheadAttention with 8 heads of
// D / 8 = 96, evaluation.py:170-177) and the encoder's own attention (train.py:543-549) when
// head_dim is not 64.  Scores are never materialised.
#include <cuda_bf16.h>

#include "attention_kernels.cuh"
#include "common.h"
#include "ptx.cuh"

namespace vitk {
using namespace ptx;

namespace {

// ---------------------------------------------------------------------------------------------
// softmax(q k^T / sqrt(hd)) v with separate query and key/value sources (self- and
// cross-attention), head_dim 32 / 64 / 96 / 128.  One CTA per (image, head, group of 112
// queries); K and V of the head are staged in shared memory in segments of up to kSegKeys keys
// (rows padded by 16 bytes: conflict-free ldmatrix for every head_dim); each warp owns one
// 16-query tile and keeps its running max / sum / output in registers across key blocks and
// segments (online softmax); bf16 mma.sync m16n8k16 with fp32 accumulation.
// ---------------------------------------------------------------------------------------------
constexpr int kXWarps = 7;
constexpr int kXThreads = kXWarps * 32;
constexpr int kSegKeys = 208;

struct AttnXArgs {
  const __nv_bfloat16* q;  // row r of image b, head h: q + b*q_img + r*ldq + h*HD
  const __nv_bfloat16* k;
  const __nv_bfloat16* v;
  __nv_bfloat16* ctx;
  long long q_img, kv_img, ctx_img;  // elements between consecutive images
  int ldq, ldkv, ldc;                // row pitches, elements
  int Nq, Nk, H;
  float scale;
};

// One block of 64 keys for one 16-query tile: S = Q K^T, online-softmax update, O += P V.
// FULL (all 64 keys valid) is branch-free, so the eight score accumulators and the HD/8 output
// accumulators form independent MMA chains the scheduler can interleave; the ragged last block
// of a segment takes the predicated path.
template <int HD, bool FULL>
__device__ __forceinline__ void attn_x_block(uint32_t sK, uint32_t sV, int key0, int rem, int lane,
                                             const uint32_t (&qa)[HD / 16][4], float (&o)[HD / 8][4],
                                             float& m0, float& m1, float& l0, float& l1, float c) {
  constexpr int PITCH = HD * 2 + 16;
  constexpr int NT = HD / 8;
  const int t = lane & 3;
  float s[8][4];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    if (FULL || j * 8 < rem) s[j][0] = s[j][1] = s[j][2] = s[j][3] = 0.f;
    else s[j][0] = s[j][1] = s[j][2] = s[j][3] = -INFINITY;
  }
#pragma unroll
  for (int half = 0; half < HD / 32; ++half) {
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      if (FULL || j * 8 < rem) {
        const int key = key0 + j * 8 + (lane & 7);
        const int ch = (lane >> 3) + 4 * half;
        uint32_t k0, k1, k2, k3;
        ldmatrix_x4(sK + key * PITCH + ch * 16, k0, k1, k2, k3);
        mma_m16n8k16(s[j], qa[2 * half], k0, k1);
        mma_m16n8k16(s[j], qa[2 * half + 1], k2, k3);
      }
    }
  }
  if (!FULL) {
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int k0 = j * 8 + t * 2;
      if (k0 >= rem) s[j][0] = s[j][2] = -INFINITY;
      if (k0 + 1 >= rem) s[j][1] = s[j][3] = -INFINITY;
    }
  }
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
  for (int j = 0; j < NT; ++j) {
    o[j][0] *= a0;
    o[j][1] *= a0;
    o[j][2] *= a1;
    o[j][3] *= a1;
  }
#pragma unroll
  for (int kk = 0; kk < 4; ++kk) {
    if (FULL || kk * 16 < rem) {
      uint32_t pa[4];
      pa[0] = pack_bf16x2(s[2 * kk][0], s[2 * kk][1]);
      pa[1] = pack_bf16x2(s[2 * kk][2], s[2 * kk][3]);
      pa[2] = pack_bf16x2(s[2 * kk + 1][0], s[2 * kk + 1][1]);
      pa[3] = pack_bf16x2(s[2 * kk + 1][2], s[2 * kk + 1][3]);
      const int mi = lane >> 3;
      const int key = key0 + kk * 16 + (mi & 1) * 8 + (lane & 7);
#pragma unroll
      for (int jj = 0; jj < HD / 16; ++jj) {
        const int ch = 2 * jj + (mi >> 1);
        uint32_t v0, v1, v2, v3;
        ldmatrix_x4_trans(sV + key * PITCH + ch * 16, v0, v1, v2, v3);
        mma_m16n8k16(o[2 * jj], pa, v0, v1);
        mma_m16n8k16(o[2 * jj + 1], pa, v2, v3);
      }
    }
  }
}

template <int HD>
__global__ void __launch_bounds__(kXThreads, HD > 96 ? 1 : 2) attn_x_kernel(const AttnXArgs a) {
  extern __shared__ __align__(128) uint8_t smem[];
  constexpr int PITCH = HD * 2 + 16;  // bytes
  constexpr int CH = HD / 8;          // 16-byte chunks per row
  constexpr int KS = HD / 16;         // k-steps of q k^T
  constexpr int NT = HD / 8;          // output n-tiles
  const uint32_t sK = smem_u32(smem);
  const uint32_t sV = sK + kSegKeys * PITCH;
  const uint32_t sO = sV + kSegKeys * PITCH;

  const int b = blockIdx.x / a.H;
  const int h = blockIdx.x - b * a.H;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int g = lane >> 2, t = lane & 3;
  const __nv_bfloat16* qbase = a.q + b * a.q_img + h * HD;
  const __nv_bfloat16* kbase = a.k + b * a.kv_img + h * HD;
  const __nv_bfloat16* vbase = a.v + b * a.kv_img + h * HD;

  const int q0 = (blockIdx.y * kXWarps + warp) * 16;
  const bool active = q0 < a.Nq;
  const int r0 = q0 + g, r1 = r0 + 8;
  uint32_t qa[KS][4];
  if (active) {
    const uint32_t* p0 = reinterpret_cast<const uint32_t*>(qbase + static_cast<size_t>(r0) * a.ldq);
    const uint32_t* p1 = reinterpret_cast<const uint32_t*>(qbase + static_cast<size_t>(r1) * a.ldq);
#pragma unroll
    for (int kk = 0; kk < KS; ++kk) {
      const int w = kk * 8 + t;
      qa[kk][0] = (r0 < a.Nq) ? __ldg(p0 + w) : 0u;
      qa[kk][1] = (r1 < a.Nq) ? __ldg(p1 + w) : 0u;
      qa[kk][2] = (r0 < a.Nq) ? __ldg(p0 + w + 4) : 0u;
      qa[kk][3] = (r1 < a.Nq) ? __ldg(p1 + w + 4) : 0u;
    }
  }
  float o[NT][4];
#pragma unroll
  for (int j = 0; j < NT; ++j) o[j][0] = o[j][1] = o[j][2] = o[j][3] = 0.f;
  float m0 = -INFINITY, m1 = -INFINITY, l0 = 0.f, l1 = 0.f;
  const float c = a.scale * kLog2e;  // softmax in base 2

  for (int seg0 = 0; seg0 < a.Nk; seg0 += kSegKeys) {
    const int nseg = min(kSegKeys, a.Nk - seg0);
    const int nrows = (nseg + 15) & ~15;
    if (seg0 > 0) __syncthreads();  // everyone is done with the previous segment
    for (int idx = tid; idx < nrows * CH; idx += kXThreads) {
      const int row = idx / CH, ch = idx - row * CH;
      const bool valid = row < nseg;
      const size_t off = static_cast<size_t>(seg0 + (valid ? row : 0)) * a.ldkv + ch * 8;
      cp_async_16(sK + row * PITCH + ch * 16, kbase + off, valid);
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
    for (int idx = tid; idx < nrows * CH; idx += kXThreads) {
      const int row = idx / CH, ch = idx - row * CH;
      const bool valid = row < nseg;
      const size_t off = static_cast<size_t>(seg0 + (valid ? row : 0)) * a.ldkv + ch * 8;
      cp_async_16(sV + row * PITCH + ch * 16, vbase + off, valid);
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
    // K first: the score MMAs of the first key block start while V is still in flight
    asm volatile("cp.async.wait_group 1;" ::: "memory");
    __syncthreads();
    if (!active) {  // warps without a query tile only help staging; match the V barrier below
      asm volatile("cp.async.wait_group 0;" ::: "memory");
      __syncthreads();
      continue;
    }
    bool v_ready = false;

    for (int kb = 0; kb * 64 < nseg; ++kb) {
      const int rem = nseg - kb * 64;
      if (!v_ready) {  // uniform across the CTA: every warp with a tile passes here once
        // (the score MMAs below do not need V, but keeping the barrier ahead of the block body
        // lets the full-block path stay branch-free)
        asm volatile("cp.async.wait_group 0;" ::: "memory");
        __syncthreads();
        v_ready = true;
      }
      if (rem >= 64)
        attn_x_block<HD, true>(sK, sV, kb * 64, 64, lane, qa, o, m0, m1, l0, l1, c);
      else
        attn_x_block<HD, false>(sK, sV, kb * 64, rem, lane, qa, o, m0, m1, l0, l1, c);
    }
  }
  if (!active) return;

  // ---- divide by the row sum, stage the 16 x HD tile through shared memory, 16-byte stores
  l0 = quad_sum(l0);
  l1 = quad_sum(l1);
  const float inv0 = 1.f / l0, inv1 = 1.f / l1;
  const uint32_t sOw = sO + warp * 16 * PITCH;
#pragma unroll
  for (int j = 0; j < NT; ++j) {
    const uint32_t w0 = pack_bf16x2(o[j][0] * inv0, o[j][1] * inv0);
    const uint32_t w1 = pack_bf16x2(o[j][2] * inv1, o[j][3] * inv1);
    asm volatile("st.shared.b32 [%0], %1;" ::"r"(sOw + g * PITCH + j * 16 + t * 4), "r"(w0)
                 : "memory");
    asm volatile("st.shared.b32 [%0], %1;" ::"r"(sOw + (g + 8) * PITCH + j * 16 + t * 4), "r"(w1)
                 : "memory");
  }
  __syncwarp();
  __nv_bfloat16* cbase = a.ctx + b * a.ctx_img + h * HD;
  for (int idx = lane; idx < 16 * CH; idx += 32) {
    const int row = idx / CH, ch = idx - row * CH;
    if (q0 + row < a.Nq) {
      uint4 val;
      asm volatile("ld.shared.v4.b32 {%0,%1,%2,%3}, [%4];"
                   : "=r"(val.x), "=r"(val.y), "=r"(val.z), "=r"(val.w)
                   : "r"(sOw + row * PITCH + ch * 16)
                   : "memory");
      *reinterpret_cast<uint4*>(cbase + static_cast<size_t>(q0 + row) * a.ldc + ch * 8) = val;
    }
  }
}

template <int HD>
int launch_attn_x(const AttnXArgs& a, int B, cudaStream_t stream) {
  constexpr int PITCH = HD * 2 + 16;
  constexpr size_t smem = static_cast<size_t>(2 * kSegKeys + kXWarps * 16) * PITCH;
  VITK_TRY(opt_in_smem<attn_x_kernel<HD>>(static_cast<int>(smem), "attn_x_kernel"));
  const dim3 grid(B * a.H, (a.Nq + kXWarps * 16 - 1) / (kXWarps * 16));
  attn_x_kernel<HD><<<grid, kXThreads, smem, stream>>>(a);
  VITK_CHECK_LAUNCH("attn_x_kernel");
  return VITK_OK;
}

}  // namespace

int attention_x(const void* q, long long q_img, int ldq, const void* k, const void* v,
                long long kv_img, int ldkv, void* ctx, long long ctx_img, int ldc, int B, int Nq,
                int Nk, int H, int hd, cudaStream_t stream) {
  VITK_REQUIRE(q && k && v && ctx, "attention: null operand");
  VITK_REQUIRE(B > 0 && Nq > 0 && Nk > 0 && H > 0, "attention: bad shape B=%d Nq=%d Nk=%d H=%d", B, Nq,
               Nk, H);
  VITK_REQUIRE(hd == 32 || hd == 64 || hd == 96 || hd == 128,
               "attention: head_dim %d unsupported (32, 64, 96 or 128)", hd);
  VITK_REQUIRE(ldq % 8 == 0 && ldkv % 8 == 0 && ldc % 8 == 0 && q_img % 8 == 0 && kv_img % 8 == 0 &&
                   ctx_img % 8 == 0,
               "attention: row pitches and image strides must be multiples of 8 elements");
  VITK_REQUIRE(((reinterpret_cast<uintptr_t>(q) | reinterpret_cast<uintptr_t>(k) |
                 reinterpret_cast<uintptr_t>(v) | reinterpret_cast<uintptr_t>(ctx)) & 15) == 0,
               "attention: operands must be 16-byte aligned");
  AttnXArgs a;
  a.q = static_cast<const __nv_bfloat16*>(q);
  a.k = static_cast<const __nv_bfloat16*>(k);
  a.v = static_cast<const __nv_bfloat16*>(v);
  a.ctx = static_cast<__nv_bfloat16*>(ctx);
  a.q_img = q_img;
  a.kv_img = kv_img;
  a.ctx_img = ctx_img;
  a.ldq = ldq;
  a.ldkv = ldkv;
  a.ldc = ldc;
  a.Nq = Nq;
  a.Nk = Nk;
  a.H = H;
  a.scale = 1.0f / sqrtf(static_cast<float>(hd));
  ProfileScope prof(PROF_ATTN, attention_flops(B, H, Nq, Nk, hd), stream);
  switch (hd) {
    case 32: return launch_attn_x<32>(a, B, stream);
    case 64: return launch_attn_x<64>(a, B, stream);
    case 96: return launch_attn_x<96>(a, B, stream);
    default: return launch_attn_x<128>(a, B, stream);
  }
}

}  // namespace vitk
