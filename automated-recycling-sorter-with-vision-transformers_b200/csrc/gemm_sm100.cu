// C[M,N] = A[M,K] * B[N,K]^T with a fused epilogue — the dense-contraction kernel behind every
// nn.Linear / the patch-embedding Conv2d of the reference encoder
// (reference train.py:505-515 patch conv, :527-553 qkv/projection, :561-572 linear1/GELU/linear2).
//
// sm_100a design:
//   * persistent kernel, one CTA per SM, static round-robin over 128 x BLOCK_N output tiles
//   * warp 0 lane 0 : TMA producer  (cp.async.bulk.tensor, 128B swizzle, kStages-deep mbarrier ring)
//   * warp 1 lane 0 : tcgen05.mma issuer (bf16 x bf16 -> fp32 in TMEM, 128 x BLOCK_N x 16 per MMA)
//   * warp 2        : TMEM allocator (2 accumulator stages so tile i's epilogue overlaps tile
//                     i+1's main loop)
//   * warps 4..11   : epilogue — tcgen05.ld (thread == accumulator row), bias / GELU in registers,
//                     then 32-row x 128-byte slabs staged in swizzled shared memory and written
//                     by TMA (bulk tensor store; the fp32 residual update x += acc + bias is a
//                     TMA reduce-add, so the residual stream is never read by the SM).  A direct
//                     register->global path remains for the token-row remap of the patch embed.
//
// After gemm_bf16_tn, at the end of the file: the host-side GEMM calls that the encoder, training
// and detection-head drivers share (linear_fwd, linear_dgrad, linear_wgrad, ...).
#include "gemm_sm100.cuh"

#include "common.h"
#include "ptx.cuh"
#include "rowops.cuh"
#include "train_ops.cuh"

namespace vitk {
using namespace ptx;

// Debug aid (build with VITK_NVCC_EXTRA=-DVITK_GEMM_TRACE): the MMA-issuing warp of every pair
// leader accumulates the SM clocks it spends waiting for operands (full barriers), for a free
// accumulator stage (the epilogue), and its total run time; tests/trace_gemm.py reads them back.
#ifdef VITK_GEMM_TRACE
__device__ long long g_gemm_trace[160][8];
#define GT_BEGIN(v) const long long v = clock64()
#define GT_ADD(acc, v) acc += clock64() - v
#else
#define GT_BEGIN(v) do { } while (0)
#define GT_ADD(acc, v) do { } while (0)
#endif

namespace {

constexpr int kBlockM = 128;
constexpr int kBlockK = 64;  // 64 bf16 = 128 bytes = one swizzle row
constexpr int kUmmaK = 16;
constexpr int kNumEpiWarps = 8;
constexpr int kFirstEpiWarp = 4;
constexpr int kNumThreads = (kFirstEpiWarp + kNumEpiWarps) * 32;  // 384
constexpr int kAccStages = 2;

// CTAS == 1: one CTA computes a 128 x BLOCK_N tile (tcgen05.mma.cta_group::1, M = 128).
// CTAS == 2: a CTA pair (cluster of 2, same TPC) computes a 256 x BLOCK_N tile with
//            tcgen05.mma.cta_group::2 (M = 256): each CTA stages its own 128 A rows and HALF of
//            the B rows, so per-SM L2->SMEM traffic and SMEM read bandwidth per flop drop by 1/3.
// Epilogue staging: per warp SLABS 32-row x 128-byte slabs (two alternate for TMA stores; the
// gelu'-epilogue adds one that receives the pre-activation tile by TMA load).
template <int BLOCK_N, int CTAS, int SLABS = 2>
struct Cfg {
  static constexpr int kStagingPerWarp = SLABS * 4096;
  static constexpr int kStagingBytes = kNumEpiWarps * kStagingPerWarp;
  static constexpr int kABytes = kBlockM * kBlockK * 2;
  static constexpr int kBRows = BLOCK_N / CTAS;  // B rows staged by this CTA
  static constexpr int kBBytes = kBRows * kBlockK * 2;
  static constexpr int kStageBytes = kABytes + kBBytes;
  static constexpr int kBarBytes = 1024;
  static constexpr int kBudget = 232448 - 1024 - kBarBytes - kStagingBytes;
  static constexpr int kStages = kBudget / kStageBytes > 8 ? 8 : kBudget / kStageBytes;
  static constexpr int kTmemCols = kAccStages * BLOCK_N;  // 512 or 256 (power of two)
  static constexpr int kSmemBytes =
      kStages * kStageBytes + kStagingBytes + kBarBytes + 1024;
  static_assert(kStages >= 3, "pipeline too shallow");
  static_assert(kSmemBytes <= 232448, "exceeds 227 KB of shared memory");
  // barriers: operand ring, accumulator stages, TMEM slot, two aux slabs per epilogue warp
  static constexpr int kNumBars = 2 * kStages + 2 * kAccStages + 1 + 2 * kNumEpiWarps;
  static_assert(8 * kNumBars <= kBarBytes, "barrier block too small");
};

__device__ __forceinline__ float gelu_erf(float x) {
  return 0.5f * x * (1.f + erff(x * 0.70710678118654752440f));
}
// erf-GELU for the bf16 epilogue: x * Phi(x) with the normal CDF written as a logistic of an odd
// polynomial, Phi(x) = 1 / (1 + 2^(-x (c0 + c1 x^2 + c2 x^4))), coefficients fitted to
// 0.5 (1 + erf(x / sqrt 2)) (max |Phi error| 4.5e-5, max |gelu error| 8.6e-5 over all x - far
// below bf16 resolution).  6 FMA-pipe ops + 2 MUFU per element instead of ~25 for erff, which
// made the fc1 epilogue the bottleneck of the GEMM.  x^2 is clamped so the polynomial stays
// monotone; the logistic then saturates to exactly 0 / 1.
__device__ __forceinline__ float gelu_fast(float x) {
  const float x2 = fminf(x * x, 100.f);
  // -log2(e) * {1.595603281, 0.07344414456, -0.000640974726}
  const float p = fmaf(x2, fmaf(x2, 9.2473074e-4f, -0.10595751f), -2.3019681f);
  float e, r;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(x * p));
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(1.f + e));
  return x * r;
}
// Same CDF through the hardware tanh: Phi(x) = 0.5 + 0.5 tanh(x (a0 + a1 x^2 + a2 x^4)).
__device__ __forceinline__ float gelu_fast_tanh(float x) {
  const float x2 = fminf(x * x, 64.f);
  const float p = fmaf(x2, fmaf(x2, -3.5651449e-4f, 0.037011533f), 0.79753114f);
  float t;
  asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(x * p));
  return x * fmaf(0.5f, t, 0.5f);
}
// d/dx [x Phi(x)] with the same logistic CDF: Phi + x Phi (1 - Phi) g'(x), g(x) = x (a0 + a1 x^2 +
// a2 x^4); no extra MUFU beyond the two of Phi.  max |error| 1.8e-4 vs the exact erf derivative.
__device__ __forceinline__ float gelu_grad_fast(float x) {
  const float x2 = fminf(x * x, 100.f);
  const float p = fmaf(x2, fmaf(x2, 9.2473074e-4f, -0.10595751f), -2.3019681f);
  float e, phi;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(x * p));
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(phi) : "f"(1.f + e));
  const float gp = fmaf(x2, fmaf(x2, -3.20487363e-3f, 0.22033243f), 1.5956033f);
  return fmaf(x * phi, (1.f - phi) * gp, phi);
}
// The tanh form on a pair of values with packed fp32 arithmetic (one issue slot per two lanes for
// the polynomial): 6 packed + 2 clamp + 2 MUFU instructions per pair instead of 2 x 9.
__device__ __forceinline__ void gelu_fast_tanh_pair(float& a, float& b) {
  const uint64_t x = pack2f(a, b);
  float q0, q1;
  unpack2(fmul2(x, x), q0, q1);
  const uint64_t x2 = pack2f(fminf(q0, 64.f), fminf(q1, 64.f));
  const uint64_t c2 = pack2f(-3.5651449e-4f, -3.5651449e-4f);
  const uint64_t c1 = pack2f(0.037011533f, 0.037011533f);
  const uint64_t c0 = pack2f(0.79753114f, 0.79753114f);
  float u0, u1;
  unpack2(fmul2(x, ffma2(x2, ffma2(x2, c2, c1), c0)), u0, u1);
  float t0, t1;
  asm("tanh.approx.f32 %0, %1;" : "=f"(t0) : "f"(u0));
  asm("tanh.approx.f32 %0, %1;" : "=f"(t1) : "f"(u1));
  const uint64_t hx = fmul2(x, pack2f(0.5f, 0.5f));
  unpack2(ffma2(hx, pack2f(t0, t1), hx), a, b);
}
// d/dx [x Phi(x)] for a pair with Phi(x) = 0.5 + 0.5 tanh(u), u = x (a0 + a1 x^2 + a2 x^4):
// Phi + 0.5 x (1 - tanh(u)^2) u'(x), u' = a0 + 3 a1 x^2 + 5 a2 x^4.  One MUFU per value, packed fp32
// arithmetic; matches the forward epilogue's CDF.  Returns g (the incoming gradient pair) * gelu'.
__device__ __forceinline__ void dgelu_tanh_pair(float& g0, float& g1, float xa, float xb) {
  const uint64_t x = pack2f(xa, xb);
  float q0, q1;
  unpack2(fmul2(x, x), q0, q1);
  const uint64_t x2 = pack2f(fminf(q0, 64.f), fminf(q1, 64.f));
  const uint64_t poly = ffma2(x2, ffma2(x2, pack2f(-3.5651449e-4f, -3.5651449e-4f),
                                        pack2f(0.037011533f, 0.037011533f)),
                              pack2f(0.79753114f, 0.79753114f));
  const uint64_t dpoly = ffma2(x2, ffma2(x2, pack2f(-1.78257245e-3f, -1.78257245e-3f),
                                         pack2f(0.111034599f, 0.111034599f)),
                               pack2f(0.79753114f, 0.79753114f));
  float u0, u1, t0, t1;
  unpack2(fmul2(x, poly), u0, u1);
  asm("tanh.approx.f32 %0, %1;" : "=f"(t0) : "f"(u0));
  asm("tanh.approx.f32 %0, %1;" : "=f"(t1) : "f"(u1));
  const uint64_t t = pack2f(t0, t1);
  const uint64_t half = pack2f(0.5f, 0.5f);
  const uint64_t phi = ffma2(t, half, half);
  const uint64_t sech2 = ffma2(fmul2(t, pack2f(-1.f, -1.f)), t, pack2f(1.f, 1.f));  // 1 - t^2
  const uint64_t d = ffma2(fmul2(fmul2(x, half), sech2), dpoly, phi);
  unpack2(fmul2(pack2f(g0, g1), d), g0, g1);
}
// The logistic (erf-fitted) form on a pair: 6 packed + 2 clamp + 4 MUFU instructions per pair.
__device__ __forceinline__ void gelu_fast_pair(float& a, float& b) {
  const uint64_t x = pack2f(a, b);
  float q0, q1;
  unpack2(fmul2(x, x), q0, q1);
  const uint64_t x2 = pack2f(fminf(q0, 100.f), fminf(q1, 100.f));
  const uint64_t c2 = pack2f(9.2473074e-4f, 9.2473074e-4f);
  const uint64_t c1 = pack2f(-0.10595751f, -0.10595751f);
  const uint64_t c0 = pack2f(-2.3019681f, -2.3019681f);
  float u0, u1;
  unpack2(fmul2(x, ffma2(x2, ffma2(x2, c2, c1), c0)), u0, u1);
  float e0, e1, r0, r1;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e0) : "f"(u0));
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e1) : "f"(u1));
  float d0, d1;
  unpack2(fadd2(pack2f(e0, e1), pack2f(1.f, 1.f)), d0, d1);
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r0) : "f"(d0));
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r1) : "f"(d1));
  unpack2(fmul2(x, pack2f(r0, r1)), a, b);
}
template <int EPI>
__device__ __forceinline__ float gelu_for(float x) {
  if constexpr (EPI == EPI_RELU_BF16) return fmaxf(x, 0.f);
  else if constexpr (EPI == EPI_GELU_TANH_BF16) return gelu_fast_tanh(x);
  else return gelu_fast(x);
}
template <int EPI>
constexpr bool is_gelu_epi() {  // bias + activation -> bf16 (the ReLU of the decoder FFN included)
  return EPI == EPI_GELU_BF16 || EPI == EPI_GELU_TANH_BF16 || EPI == EPI_RELU_BF16;
}
__device__ __forceinline__ float gelu_erf_grad(float x) {
  const float cdf = 0.5f * (1.f + erff(x * 0.70710678118654752440f));
  const float pdf = 0.39894228040143267794f * __expf(-0.5f * x * x);
  return cdf + x * pdf;
}

__device__ __forceinline__ bool aligned16(const void* p) {
  return (reinterpret_cast<uintptr_t>(p) & 15u) == 0;
}

// Processes one 32-column chunk of one accumulator row held in v[] (raw fp32 bits).
template <int EPI>
__device__ __forceinline__ void epilogue_chunk(const uint32_t (&v)[32], int m, int n0, int N,
                                               const GemmEpilogue& e) {
  // The 16-byte accesses below need 16-byte aligned rows.  ldo is a multiple of 8 elements and n0
  // of 32, so that comes down to the base pointers: this path is also the fallback for an output
  // (and out2 / aux, which share its pitch) at a 2- or 4-byte aligned column offset.
  bool vec_ok = aligned16(e.out);
  if constexpr (is_gelu_epi<EPI>()) vec_ok = vec_ok && aligned16(e.out2);
  if constexpr (EPI == EPI_DGELU_BF16) vec_ok = vec_ok && aligned16(e.aux);
  const bool full = (n0 + 32 <= N) && vec_ok;
  float x[32];
  // ---- alpha * accumulator (+ bias); alpha is only honoured by EPI_F32
  float acc_scale = 1.f;
  if constexpr (EPI == EPI_F32) acc_scale = e.alpha;
  if (full) {
    if (e.bias != nullptr) {
      const float4* b4 = reinterpret_cast<const float4*>(e.bias + n0);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float4 b = __ldg(b4 + j);
        x[4 * j + 0] = fmaf(acc_scale, __uint_as_float(v[4 * j + 0]), b.x);
        x[4 * j + 1] = fmaf(acc_scale, __uint_as_float(v[4 * j + 1]), b.y);
        x[4 * j + 2] = fmaf(acc_scale, __uint_as_float(v[4 * j + 2]), b.z);
        x[4 * j + 3] = fmaf(acc_scale, __uint_as_float(v[4 * j + 3]), b.w);
      }
    } else {
#pragma unroll
      for (int j = 0; j < 32; ++j) x[j] = acc_scale * __uint_as_float(v[j]);
    }
  } else {
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      const float b = (e.bias != nullptr && n0 + j < N) ? __ldg(e.bias + n0 + j) : 0.f;
      x[j] = fmaf(acc_scale, __uint_as_float(v[j]), b);
    }
  }

  const uint32_t drop_idx0 = static_cast<uint32_t>(m) * static_cast<uint32_t>(N) +
                             static_cast<uint32_t>(n0);
  if constexpr (EPI == EPI_RESID_F32 || EPI == EPI_DGELU_BF16) {
    if (e.drop.thresh != 0u) drop_apply_run<32>(x, drop_idx0, e.drop);
  }
  if constexpr (EPI == EPI_BF16 || is_gelu_epi<EPI>() || EPI == EPI_DGELU_BF16) {
    const size_t off = static_cast<size_t>(m) * e.ldo + n0;
    __nv_bfloat16* out = reinterpret_cast<__nv_bfloat16*>(e.out) + off;
    if constexpr (is_gelu_epi<EPI>()) {
      if (e.out2 != nullptr) {
        __nv_bfloat16* out2 = reinterpret_cast<__nv_bfloat16*>(e.out2) + off;
        if (full) {
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            uint4 pk;
            pk.x = pack_bf16x2(x[8 * j + 0], x[8 * j + 1]);
            pk.y = pack_bf16x2(x[8 * j + 2], x[8 * j + 3]);
            pk.z = pack_bf16x2(x[8 * j + 4], x[8 * j + 5]);
            pk.w = pack_bf16x2(x[8 * j + 6], x[8 * j + 7]);
            reinterpret_cast<uint4*>(out2)[j] = pk;
          }
        } else {
          _Pragma("unroll") for (int j = 0; j < 32; ++j)
            if (n0 + j < N) out2[j] = __float2bfloat16_rn(x[j]);
        }
      }
#pragma unroll
      for (int j = 0; j < 32; ++j) x[j] = gelu_for<EPI>(x[j]);
      if (e.drop.thresh != 0u) drop_apply_run<32>(x, drop_idx0, e.drop);
    }
    if constexpr (EPI == EPI_DGELU_BF16) {
      const __nv_bfloat16* aux = reinterpret_cast<const __nv_bfloat16*>(e.aux) + off;
      if (full) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const uint4 a = __ldg(reinterpret_cast<const uint4*>(aux) + j);
          x[8 * j + 0] *= gelu_erf_grad(bf16lo_to_f32(a.x));
          x[8 * j + 1] *= gelu_erf_grad(bf16hi_to_f32(a.x));
          x[8 * j + 2] *= gelu_erf_grad(bf16lo_to_f32(a.y));
          x[8 * j + 3] *= gelu_erf_grad(bf16hi_to_f32(a.y));
          x[8 * j + 4] *= gelu_erf_grad(bf16lo_to_f32(a.z));
          x[8 * j + 5] *= gelu_erf_grad(bf16hi_to_f32(a.z));
          x[8 * j + 6] *= gelu_erf_grad(bf16lo_to_f32(a.w));
          x[8 * j + 7] *= gelu_erf_grad(bf16hi_to_f32(a.w));
        }
      } else {
        _Pragma("unroll") for (int j = 0; j < 32; ++j)
          if (n0 + j < N) x[j] *= gelu_erf_grad(__bfloat162float(aux[j]));
      }
    }
    if (full) {
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        uint4 pk;
        pk.x = pack_bf16x2(x[8 * j + 0], x[8 * j + 1]);
        pk.y = pack_bf16x2(x[8 * j + 2], x[8 * j + 3]);
        pk.z = pack_bf16x2(x[8 * j + 4], x[8 * j + 5]);
        pk.w = pack_bf16x2(x[8 * j + 6], x[8 * j + 7]);
        reinterpret_cast<uint4*>(out)[j] = pk;
      }
    } else {
      _Pragma("unroll") for (int j = 0; j < 32; ++j)
        if (n0 + j < N) out[j] = __float2bfloat16_rn(x[j]);
    }
  } else if constexpr (EPI == EPI_RESID_F32) {
    int out_row = m, res_row = m;
    if (e.rows_per_group > 0) {
      const int g = m / e.rows_per_group;
      const int r = m - g * e.rows_per_group;
      out_row = g * e.group_stride + e.group_offset + r;
      res_row = e.group_offset + r;
    }
    float* out = reinterpret_cast<float*>(e.out) + static_cast<size_t>(out_row) * e.ldo + n0;
    const float* res = e.resid + static_cast<size_t>(res_row) * e.ldr + n0;
    if (full) {
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float4 r = *(reinterpret_cast<const float4*>(res) + j);
        float4 o;
        o.x = x[4 * j + 0] + r.x;
        o.y = x[4 * j + 1] + r.y;
        o.z = x[4 * j + 2] + r.z;
        o.w = x[4 * j + 3] + r.w;
        reinterpret_cast<float4*>(out)[j] = o;
      }
    } else {
      _Pragma("unroll") for (int j = 0; j < 32; ++j)
        if (n0 + j < N) out[j] = x[j] + res[j];
    }
  } else if constexpr (EPI == EPI_F32) {
    float* out = reinterpret_cast<float*>(e.out) + static_cast<size_t>(m) * e.ldo + n0;
    const float beta = e.beta;
    if (full) {
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        float4 o = make_float4(x[4 * j + 0], x[4 * j + 1], x[4 * j + 2], x[4 * j + 3]);
        if (beta != 0.f) {
          const float4 p = reinterpret_cast<const float4*>(out)[j];
          o.x = fmaf(beta, p.x, o.x);
          o.y = fmaf(beta, p.y, o.y);
          o.z = fmaf(beta, p.z, o.z);
          o.w = fmaf(beta, p.w, o.w);
        }
        reinterpret_cast<float4*>(out)[j] = o;
      }
    } else {
      _Pragma("unroll") for (int j = 0; j < 32; ++j)
        if (n0 + j < N) out[j] = (beta != 0.f) ? fmaf(beta, out[j], x[j]) : x[j];
    }
  }
}

// alpha * acc + bias for one 32-column chunk (alpha only for EPI_F32).
template <int EPI>
__device__ __forceinline__ void acc_plus_bias(const uint32_t (&v)[32], int n0, int N,
                                              const GemmEpilogue& e, float (&x)[32]) {
  float acc_scale = 1.f;
  if constexpr (EPI == EPI_F32) acc_scale = e.alpha;
  if (n0 + 32 <= N) {
    if (e.bias != nullptr) {
      const float4* b4 = reinterpret_cast<const float4*>(e.bias + n0);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float4 b = __ldg(b4 + j);
#ifdef VITK_SCALAR_BIAS   // A/B build: the scalar form for every epilogue
        if constexpr (true) {
#else
        if constexpr (EPI == EPI_F32) {
#endif
          x[4 * j + 0] = fmaf(acc_scale, __uint_as_float(v[4 * j + 0]), b.x);
          x[4 * j + 1] = fmaf(acc_scale, __uint_as_float(v[4 * j + 1]), b.y);
          x[4 * j + 2] = fmaf(acc_scale, __uint_as_float(v[4 * j + 2]), b.z);
          x[4 * j + 3] = fmaf(acc_scale, __uint_as_float(v[4 * j + 3]), b.w);
        } else {  // packed fp32: one FADD2 per two columns
          unpack2(fadd2(pack2(v[4 * j + 0], v[4 * j + 1]), pack2f(b.x, b.y)), x[4 * j + 0],
                  x[4 * j + 1]);
          unpack2(fadd2(pack2(v[4 * j + 2], v[4 * j + 3]), pack2f(b.z, b.w)), x[4 * j + 2],
                  x[4 * j + 3]);
        }
      }
    } else {
#pragma unroll
      for (int j = 0; j < 32; ++j) x[j] = acc_scale * __uint_as_float(v[j]);
    }
  } else {
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      const float b = (e.bias != nullptr && n0 + j < N) ? __ldg(e.bias + n0 + j) : 0.f;
      x[j] = fmaf(acc_scale, __uint_as_float(v[j]), b);
    }
  }
}

// LayerNorm folded into the GEMM (GemmEpilogue::ln_part): rstd * acc + bias[n] for one 32-column
// chunk (the weight rows are centred, so the contraction has already removed the row mean);
// packed fp32 arithmetic: one FFMA2 per two columns.
__device__ __forceinline__ void acc_scale_bias(const uint32_t (&v)[32], int n0, int N,
                                               const GemmEpilogue& e, float rstd, float (&x)[32]) {
  if (n0 + 32 <= N) {
    const float4* b4 = reinterpret_cast<const float4*>(e.bias + n0);
    const uint64_t r2 = pack2f(rstd, rstd);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float4 b = __ldg(b4 + j);
      unpack2(ffma2(r2, pack2(v[4 * j + 0], v[4 * j + 1]), pack2f(b.x, b.y)), x[4 * j + 0],
              x[4 * j + 1]);
      unpack2(ffma2(r2, pack2(v[4 * j + 2], v[4 * j + 3]), pack2f(b.z, b.w)), x[4 * j + 2],
              x[4 * j + 3]);
    }
  } else {
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      const float b = (n0 + j < N) ? __ldg(e.bias + n0 + j) : 0.f;
      x[j] = fmaf(rstd, __uint_as_float(v[j]), b);
    }
  }
}

// Residual epilogue without TMA (row remap of the patch embedding: patch row -> token slot, and
// the position-embedding row as the residual; or out != resid): the warp stages its 32 x 32 fp32
// tile in its slab (thread == row), then writes it out cooperatively - eight lanes per row, each
// 16 bytes, so every row segment is one coalesced 128-byte access for the residual read and for
// the store, whatever row the remap sends it to.  (Per-thread stores of whole rows, as in
// epilogue_chunk, touch 32 lines with 16 bytes each per instruction: the patch-embedding GEMM ran
// at 162 us against 71 us for the same contraction with the TMA epilogue.)
__device__ __forceinline__ void resid_chunk_staged(const uint32_t (&v)[32], int row0, int n0, int M,
                                                   int N, const GemmEpilogue& e, uint32_t slab,
                                                   int lane) {
  float x[32];
  acc_plus_bias<EPI_RESID_F32>(v, n0, N, e, x);
  if (e.drop.thresh != 0u)
    drop_apply_run<32>(x, static_cast<uint32_t>(row0 + lane) * static_cast<uint32_t>(N) +
                              static_cast<uint32_t>(n0), e.drop);
  const uint32_t row = slab + static_cast<uint32_t>(lane) * 128u;
#pragma unroll
  for (int j = 0; j < 8; ++j)
    st_shared_v4(row + (static_cast<uint32_t>(j ^ (lane & 7)) << 4), __float_as_uint(x[4 * j]),
                 __float_as_uint(x[4 * j + 1]), __float_as_uint(x[4 * j + 2]),
                 __float_as_uint(x[4 * j + 3]));
  __syncwarp();
  const int piece = lane & 7;
  const bool col_ok = n0 + 4 * piece < N;   // N is a multiple of 8
  // ldo and ldr are multiples of 4: 16-byte accesses unless a base pointer sits at a column offset
  const bool vec_ok = aligned16(e.out) && aligned16(e.resid);
#pragma unroll
  for (int it = 0; it < 8; ++it) {
    const int r = it * 4 + (lane >> 3);
    const int m = row0 + r;
    if (m < M && col_ok) {
      int out_row = m, res_row = m;
      if (e.rows_per_group > 0) {
        const int g = m / e.rows_per_group;
        const int rr = m - g * e.rows_per_group;
        out_row = g * e.group_stride + e.group_offset + rr;
        res_row = e.group_offset + rr;
      }
      float a0, a1, a2, a3;
      asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];"
                   : "=f"(a0), "=f"(a1), "=f"(a2), "=f"(a3)
                   : "r"(slab + static_cast<uint32_t>(r) * 128u +
                         (static_cast<uint32_t>(piece ^ (r & 7)) << 4))
                   : "memory");
      const float* rs = e.resid + static_cast<size_t>(res_row) * e.ldr + n0 + 4 * piece;
      float* o = reinterpret_cast<float*>(e.out) + static_cast<size_t>(out_row) * e.ldo + n0 +
                 4 * piece;
      if (vec_ok) {
        const float4 r4 = *reinterpret_cast<const float4*>(rs);
        *reinterpret_cast<float4*>(o) = make_float4(a0 + r4.x, a1 + r4.y, a2 + r4.z, a3 + r4.w);
      } else {
        o[0] = a0 + rs[0];
        o[1] = a1 + rs[1];
        o[2] = a2 + rs[2];
        o[3] = a3 + rs[3];
      }
    }
  }
  __syncwarp();   // the slab is rewritten by the next chunk
}

// One epilogue warp: stage a 32-row x 128-byte slab (row = lane) in swizzled smem and hand it to
// the TMA engine.  `pk` holds the lane's 128 output bytes. Two buffers alternate per warp.
__device__ __forceinline__ void stage_and_store(const uint32_t (&pk)[32], uint32_t stg, int& buf,
                                                int lane, const CUtensorMap* tmap, int c0, int c1,
                                                bool reduce) {
  // the slab stored two steps ago has been read out
  if (lane == 0) tma_store_wait_read<1>();
  __syncwarp();
  const uint32_t slab = stg + static_cast<uint32_t>(buf) * 4096u;
  const uint32_t row = slab + static_cast<uint32_t>(lane) * 128u;
#pragma unroll
  for (int j = 0; j < 8; ++j)
    st_shared_v4(row + (static_cast<uint32_t>(j ^ (lane & 7)) << 4), pk[4 * j], pk[4 * j + 1],
                 pk[4 * j + 2], pk[4 * j + 3]);
  fence_proxy_async_smem();
  __syncwarp();
  if (lane == 0) {
    if (reduce)
      tma_reduce_add_2d(tmap, slab, c0, c1);
    else
      tma_store_2d(tmap, slab, c0, c1);
    tma_store_commit();
  }
  buf ^= 1;
}

// MN == false: A[M,K], B[N,K] with K contiguous (activations x nn.Linear weights).
// MN == true : A[K,M], B[K,N] with M / N contiguous - the weight-gradient contraction
//              dW[out,in] = sum_tokens dY[token,out] * X[token,in] reads both activations in place
//              as MN-major tcgen05 operands (64x64 TMA boxes, LBO = 8 KB between 64-wide chunks).
// The K range can be split across `num_splits` work items per tile (reduce-add epilogue).
// `e` is __grid_constant__: its fields are read from parameter space where they are used, not
// loaded into registers at the kernel's start.
template <int BLOCK_N, int EPI, int CTAS, bool TMA_EPI, bool MN>
__global__ void __launch_bounds__(kNumThreads, 1)
gemm_tn_kernel(const __grid_constant__ CUtensorMap tmap_a,
               const __grid_constant__ CUtensorMap tmap_b,
               const __grid_constant__ CUtensorMap tmap_c,
               const __grid_constant__ CUtensorMap tmap_c2, int M, int N, int K,
               int kb_per_split, int num_splits, int descending,
               const __grid_constant__ GemmEpilogue e) {
  constexpr bool kAuxTma = TMA_EPI && (EPI == EPI_DGELU_BF16);
  constexpr bool kStats = TMA_EPI && (EPI == EPI_RESID_STATS_F32);
  static_assert(EPI != EPI_RESID_STATS_F32 || TMA_EPI, "the statistics epilogue is TMA-only");
  using C = Cfg<BLOCK_N, CTAS, kAuxTma ? 3 : 2>;
  constexpr int kStagingBytes = C::kStagingBytes;
  constexpr int kStagingPerWarp = C::kStagingPerWarp;
  constexpr int kTileM = kBlockM * CTAS;  // rows of C per cluster tile
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = smem_u32(smem_raw);
  const uint32_t base = (raw_addr + 1023u) & ~1023u;  // SWIZZLE_128B atoms need 1024B alignment
  uint8_t* smem = smem_raw + (base - raw_addr);

  const uint32_t staging_base = base + C::kStages * C::kStageBytes;  // 1024-aligned
  const uint32_t bar_base = staging_base + kStagingBytes;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (C::kStages + s); };
  auto tfull_bar = [&](int a) { return bar_base + 8u * (2 * C::kStages + a); };
  auto tempty_bar = [&](int a) { return bar_base + 8u * (2 * C::kStages + kAccStages + a); };
  volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(
      smem + C::kStages * C::kStageBytes + kStagingBytes + 8 * (2 * C::kStages + 2 * kAccStages));
  auto aux_bar = [&](int w) { return bar_base + 8u * (2 * C::kStages + 2 * kAccStages + 1 + w); };
  // second slab barrier of the statistics epilogue (the first is aux_bar)
  [[maybe_unused]] auto aux2_bar = [&](int w) {
    return bar_base + 8u * (2 * C::kStages + 2 * kAccStages + 1 + kNumEpiWarps + w);
  };

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t cta_rank = (CTAS == 2) ? cluster_ctarank() : 0u;  // 0 = MMA leader of the pair
  const bool is_leader = (cta_rank == 0);
  const int cluster_id = blockIdx.x / CTAS;
  const int num_clusters = gridDim.x / CTAS;

  const int num_m_tiles = (M + kTileM - 1) / kTileM;
  const int num_n_tiles = (N + BLOCK_N - 1) / BLOCK_N;
  const int num_out_tiles = num_m_tiles * num_n_tiles;
  const int num_tiles = num_out_tiles * num_splits;  // work items: (output tile, K split)
  const int num_kb_total = (K + kBlockK - 1) / kBlockK;
  // output tile of a work item; `descending` walks the row tiles from the last to the first
  auto tile_of = [&](int work) {
    const int tile = work % num_out_tiles;
    return descending ? num_out_tiles - 1 - tile : tile;
  };
  auto kb_begin = [&](int work) { return (work / num_out_tiles) * kb_per_split; };
  auto kb_end = [&](int work) {
    const int e2 = (work / num_out_tiles + 1) * kb_per_split;
    return e2 < num_kb_total ? e2 : num_kb_total;
  };

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tmap_a);
    prefetch_tmap(&tmap_b);
    if constexpr (TMA_EPI) prefetch_tmap(&tmap_c);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < C::kStages; ++s) {
      mbar_init(full_bar(s), 1);   // leader: one arrive.expect_tx covering both CTAs' bytes
      mbar_init(empty_bar(s), 1);  // one (multicast) tcgen05.commit
    }
    for (int a = 0; a < kAccStages; ++a) {
      mbar_init(tfull_bar(a), 1);
      mbar_init(tempty_bar(a), kNumEpiWarps * CTAS);  // leader collects both CTAs' epilogues
    }
    if constexpr (kAuxTma || kStats)
      for (int w2 = 0; w2 < kNumEpiWarps; ++w2) mbar_init(aux_bar(w2), 1);
    if constexpr (kStats)
      for (int w2 = 0; w2 < kNumEpiWarps; ++w2) mbar_init(aux2_bar(w2), 1);
    fence_mbar_init();
  }
  if (warp == 2) {
    if constexpr (CTAS == 2) {
      tmem_alloc_2sm(smem_u32(const_cast<uint32_t*>(tmem_slot)), C::kTmemCols);
      tmem_relinquish_2sm();
    } else {
      tmem_alloc(smem_u32(const_cast<uint32_t*>(tmem_slot)), C::kTmemCols);
      tmem_relinquish();
    }
  }
  tc_fence_before();
  if constexpr (CTAS == 2) cluster_sync_all(); else __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ======================= TMA producer (every CTA stages its own operand slices) ==========
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int work = cluster_id; work < num_tiles; work += num_clusters) {
        const int tile = tile_of(work);
        const int m_blk = tile / num_n_tiles;
        const int n_blk = tile - m_blk * num_n_tiles;
        const int m0 = m_blk * kTileM + static_cast<int>(cta_rank) * kBlockM;
        const int n0 = n_blk * BLOCK_N + static_cast<int>(cta_rank) * C::kBRows;
        for (int kb = kb_begin(work); kb < kb_end(work); ++kb) {
          mbar_wait(empty_bar(stage), phase ^ 1u);
          const uint32_t sa = base + stage * C::kStageBytes;
          const uint32_t sb = sa + C::kABytes;
          const uint32_t fbar = (CTAS == 2) ? (full_bar(stage) & kPeerBitMask) : full_bar(stage);
          if constexpr (CTAS == 2) {
            if (is_leader) mbar_arrive_expect_tx(full_bar(stage), 2 * C::kStageBytes);
          } else {
            mbar_arrive_expect_tx(full_bar(stage), C::kStageBytes);
          }
          if constexpr (!MN) {
            if constexpr (CTAS == 2) {
              tma_load_2d_2sm(sa, &tmap_a, fbar, kb * kBlockK, m0);
              tma_load_2d_2sm(sb, &tmap_b, fbar, kb * kBlockK, n0);
            } else {
              tma_load_2d(sa, &tmap_a, fbar, kb * kBlockK, m0);
              tma_load_2d(sb, &tmap_b, fbar, kb * kBlockK, n0);
            }
          } else {
            // 64 (M or N, contiguous) x 64 (K) boxes; chunk j of the tile sits 8 KB after chunk j-1
#pragma unroll
            for (int j = 0; j < kBlockM / 64; ++j) {
              if constexpr (CTAS == 2)
                tma_load_2d_2sm(sa + j * 8192, &tmap_a, fbar, m0 + 64 * j, kb * kBlockK);
              else
                tma_load_2d(sa + j * 8192, &tmap_a, fbar, m0 + 64 * j, kb * kBlockK);
            }
#pragma unroll
            for (int j = 0; j < C::kBRows / 64; ++j) {
              if constexpr (CTAS == 2)
                tma_load_2d_2sm(sb + j * 8192, &tmap_b, fbar, n0 + 64 * j, kb * kBlockK);
              else
                tma_load_2d(sb + j * 8192, &tmap_b, fbar, n0 + 64 * j, kb * kBlockK);
            }
          }
          if (++stage == C::kStages) {
            stage = 0;
            phase ^= 1u;
          }
        }
      }
      if constexpr (CTAS == 2) {
        // tail: every slot this CTA filled has been consumed, i.e. all multicast commits aimed at
        // this CTA's barriers have landed before it may reach the final cluster barrier and exit
        for (int s = 0; s < C::kStages; ++s) {
          mbar_wait(empty_bar(stage), phase ^ 1u);
          if (++stage == C::kStages) {
            stage = 0;
            phase ^= 1u;
          }
        }
      }
    }
  } else if (warp == 1) {
    // ======================= MMA issuer (pair leader only) =======================
    // The whole warp stays converged and one elected lane issues: the uniform-datapath
    // instructions (UTCHMMA, UTCBAR) are then emitted without a per-active-lane election loop
    // and register->uniform-register broadcasts around each of them.
    if (is_leader) {
      constexpr uint32_t idesc = make_idesc_bf16(kTileM, BLOCK_N, MN ? 1 : 0, MN ? 1 : 0);
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      [[maybe_unused]] long long gt_full = 0, gt_empty = 0;
      GT_BEGIN(gt_start);
      for (int work = cluster_id; work < num_tiles; work += num_clusters) {
        GT_BEGIN(gt_e);
        mbar_wait(tempty_bar(acc), acc_phase ^ 1u);
        GT_ADD(gt_empty, gt_e);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + static_cast<uint32_t>(acc * BLOCK_N);
        const int kb0 = kb_begin(work);
        for (int kb = kb0; kb < kb_end(work); ++kb) {
          GT_BEGIN(gt_f);
          mbar_wait(full_bar(stage), phase);
          GT_ADD(gt_full, gt_f);
          tc_fence_after();
          const uint32_t sa = base + stage * C::kStageBytes;
          const uint32_t sb = sa + C::kABytes;
          // K-major: LBO unused, 8-row groups 1024 B apart, +32 B per 16-element K step.
          // MN-major: 64-wide M/N chunks 8192 B apart (LBO), 8-row K groups 1024 B apart (SBO),
          //           +2048 B (16 K rows of 128 B) per K step.
          const uint64_t a_desc = make_desc_sw128(sa, MN ? 8192 : 16, 1024);
          const uint64_t b_desc = make_desc_sw128(sb, MN ? 8192 : 16, 1024);
          constexpr uint32_t kstep = MN ? 128u : 2u;  // descriptor start-address units of 16 B
          if (elect_one_sync()) {
#pragma unroll
            for (int k = 0; k < kBlockK / kUmmaK; ++k) {
              const uint32_t accum = (kb > kb0 || k > 0) ? 1u : 0u;
              if constexpr (CTAS == 2)
                mma_bf16_ss_2sm(d_tmem, a_desc + kstep * k, b_desc + kstep * k, idesc, accum);
              else
                mma_bf16_ss(d_tmem, a_desc + kstep * k, b_desc + kstep * k, idesc, accum);
            }
            // frees the smem slot (in both CTAs) when these MMAs retire
            if constexpr (CTAS == 2) mma_commit_2sm_mc(empty_bar(stage), 3);
            else mma_commit(empty_bar(stage));
          }
          __syncwarp();
          if (++stage == C::kStages) {
            stage = 0;
            phase ^= 1u;
          }
        }
        // accumulator complete -> epilogue warps of both CTAs
        if (elect_one_sync()) {
          if constexpr (CTAS == 2) mma_commit_2sm_mc(tfull_bar(acc), 3);
          else mma_commit(tfull_bar(acc));
        }
        __syncwarp();
        if (++acc == kAccStages) {
          acc = 0;
          acc_phase ^= 1u;
        }
      }
#ifdef VITK_GEMM_TRACE
      if (lane == 0 && cluster_id < 160) {
        g_gemm_trace[cluster_id][0] = clock64() - gt_start;
        g_gemm_trace[cluster_id][1] = gt_full;
        g_gemm_trace[cluster_id][2] = gt_empty;
        g_gemm_trace[cluster_id][3] = (num_tiles - cluster_id + num_clusters - 1) / num_clusters;
      }
#endif
    }
  } else if (warp >= kFirstEpiWarp) {
    // ======================= epilogue =======================
    const int q = warp & 3;                        // TMEM lane quarter this warp may access
    const int half = (warp - kFirstEpiWarp) >> 2;  // which half of the tile's columns
    constexpr int kColsPerWarp = BLOCK_N / 2;
    const int slab_row = static_cast<int>(cta_rank) * kBlockM + q * 32;  // first row of this warp
    const uint32_t stg = staging_base + static_cast<uint32_t>(warp - kFirstEpiWarp) * kStagingPerWarp;
    int buf = 0;
    int acc = 0;
    uint32_t acc_phase = 0;
    [[maybe_unused]] uint32_t aux_phase = 0;
    [[maybe_unused]] const uint32_t aux_slab = stg + 2u * 4096u;
    [[maybe_unused]] const uint32_t my_aux_bar = aux_bar(warp - kFirstEpiWarp);
    [[maybe_unused]] const uint32_t my_aux2_bar = aux2_bar(warp - kFirstEpiWarp);
    [[maybe_unused]] uint32_t x_phase = 0;  // statistics epilogue: parity bit per slab
    [[maybe_unused]] long long gt_epi_wait = 0, gt_epi_ld = 0, gt_epi_math = 0, gt_epi_store = 0;
    // folded LayerNorm (consumer side): partial sums of the next tile's row, in flight
    [[maybe_unused]] float2 ln_next[8];
    [[maybe_unused]] float ln_rstd_next = 1.f;
    [[maybe_unused]] bool ln_have_next = false;
    [[maybe_unused]] auto ln_load_stats = [&](int m, float2 (&t)[8]) {
#pragma unroll
      for (int p2 = 0; p2 < 8; ++p2) {
        t[p2] = make_float2(0.f, 0.f);
        // volatile: issued HERE (before the wait for the accumulator), not sunk to the use
        if (p2 < e.ln_nparts && m < M)
          asm volatile("ld.global.nc.v2.f32 {%0, %1}, [%2];"
                       : "=f"(t[p2].x), "=f"(t[p2].y)
                       : "l"(e.ln_part + static_cast<size_t>(p2) * M + m));
      }
    };
    [[maybe_unused]] auto ln_finish = [&](float s1, float s2) {
      const float inv_d = 1.f / static_cast<float>(e.ln_dim);
      const float mean = s1 * inv_d;
      const float var = fmaxf(fmaf(-mean, mean, s2 * inv_d), 0.f);
      return rsqrtf(var + e.ln_eps);
    };
    for (int work = cluster_id; work < num_tiles; work += num_clusters) {
      const int tile = tile_of(work);
      const int m_blk = tile / num_n_tiles;
      const int n_blk = tile - m_blk * num_n_tiles;
      if constexpr (kAuxTma) {
        // fetch the first pre-activation slab of this tile while its main loop is still running
        const int r0 = m_blk * kTileM + slab_row;
        const int c0 = n_blk * BLOCK_N + half * kColsPerWarp;
        if (lane == 0 && r0 < M && c0 < N) {
          mbar_arrive_expect_tx(my_aux_bar, 4096);
          tma_load_2d(aux_slab, &tmap_c2, my_aux_bar, c0, r0);
        }
      }
      const int row0 = m_blk * kTileM + slab_row;
      if constexpr (kStats) {
        // fetch this warp's first two 32 x 32 tiles of x while the main loop is still running;
        // both slabs were last the source of the previous tile's stores
        if (lane == 0 && row0 < M) {
          tma_store_wait_read<0>();
#pragma unroll
          for (int c = 0; c < 2; ++c) {
            const int c0 = n_blk * BLOCK_N + half * kColsPerWarp + 32 * c;
            if (c0 < N) {
              const uint32_t xb = c == 0 ? my_aux_bar : my_aux2_bar;
              mbar_arrive_expect_tx(xb, 4096);
              tma_load_2d(stg + static_cast<uint32_t>(c) * 4096u, &tmap_c, xb, c0, row0);
            }
          }
        }
      }
      // LayerNorm folded into this GEMM: mean / rstd of this thread's row from the partial sums
      // the producing residual GEMM left (fixed summation order)
      [[maybe_unused]] float ln_rstd = 1.f;
      if constexpr (TMA_EPI && (EPI == EPI_BF16 || is_gelu_epi<EPI>())) {
        if (e.ln_part != nullptr) {
          // rstd of this thread's row of THIS tile: reduced at the end of the previous tile's
          // epilogue from loads issued at its start (below), so the round trip to L2 is hidden;
          // only the first tile of a CTA pays it
          if (ln_have_next) {
            ln_rstd = ln_rstd_next;
          } else {
            float s1 = 0.f, s2 = 0.f;
            ln_load_stats(row0 + lane, ln_next);
#pragma unroll
            for (int p2 = 0; p2 < 8; ++p2) {
              s1 += ln_next[p2].x;
              s2 += ln_next[p2].y;
            }
            ln_rstd = ln_finish(s1, s2);
          }
          // the next tile's partial sums: up to 8 independent loads in flight under this epilogue
          const int work_nx = work + num_clusters;
          ln_have_next = work_nx < num_tiles;
          if (ln_have_next)
            ln_load_stats((tile_of(work_nx) / num_n_tiles) * kTileM + slab_row + lane, ln_next);
        }
      }
      GT_BEGIN(gt_w);
      mbar_wait(tfull_bar(acc), acc_phase);
      GT_ADD(gt_epi_wait, gt_w);
      tc_fence_after();
      const uint32_t t_row = tmem_base + (static_cast<uint32_t>(q * 32) << 16) +
                             static_cast<uint32_t>(acc * BLOCK_N + half * kColsPerWarp);
      const int n_base = n_blk * BLOCK_N + half * kColsPerWarp;
      // The accumulator stage goes back to the MMA warp as soon as this warp's last TMEM read has
      // landed in registers - the arithmetic and the stores of the last chunk then run under the
      // next-but-one tile's MMAs instead of in front of them.
      auto release_acc = [&]() {
        tc_fence_before();
        __syncwarp();
        if (lane == 0) {
          if (CTAS == 2 && !is_leader)
            mbar_arrive_cluster(mapa_shared(tempty_bar(acc), 0));
          else
            mbar_arrive(tempty_bar(acc));
        }
      };
      if constexpr (kStats) {
        // x (fp32, in place) += acc + bias; bf16 copy; partial row sums.  Thread == row.
        const bool o2_wide =
            ((reinterpret_cast<uintptr_t>(e.out2) | static_cast<uintptr_t>(e.ldo * 2)) & 31u) == 0;
        float sum1 = 0.f, sum2 = 0.f;
        uint32_t v[2][32];
        tmem_ld_32x32b_x32(t_row, v[0]);
#pragma unroll
        for (int c = 0; c < kColsPerWarp / 32; ++c) {
          tmem_ld_wait();
          if (c + 1 < kColsPerWarp / 32) tmem_ld_32x32b_x32(t_row + (c + 1) * 32, v[(c + 1) & 1]);
          else release_acc();
          const int n0 = n_base + c * 32;
          if (row0 < M && n0 < N) {
            float x[32];
            acc_plus_bias<EPI>(v[c & 1], n0, N, e, x);
            const uint32_t slab = stg + static_cast<uint32_t>(c & 1) * 4096u;
            const uint32_t row = slab + static_cast<uint32_t>(lane) * 128u;
            mbar_wait((c & 1) ? my_aux2_bar : my_aux_bar, (x_phase >> (c & 1)) & 1u);
            x_phase ^= 1u << (c & 1);
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              float r0, r1, r2, r3;
              asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];"
                           : "=f"(r0), "=f"(r1), "=f"(r2), "=f"(r3)
                           : "r"(row + (static_cast<uint32_t>(j ^ (lane & 7)) << 4))
                           : "memory");
              x[4 * j + 0] += r0;
              x[4 * j + 1] += r1;
              x[4 * j + 2] += r2;
              x[4 * j + 3] += r3;
            }
            // (columns >= N hold zeros: zero-filled operands, no bias, zero-filled x)
#pragma unroll
            for (int j = 0; j < 32; ++j) {
              sum1 += x[j];
              sum2 = fmaf(x[j], x[j], sum2);
            }
#pragma unroll
            for (int j = 0; j < 8; ++j)
              st_shared_v4(row + (static_cast<uint32_t>(j ^ (lane & 7)) << 4),
                           __float_as_uint(x[4 * j]), __float_as_uint(x[4 * j + 1]),
                           __float_as_uint(x[4 * j + 2]), __float_as_uint(x[4 * j + 3]));
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) {
              tma_store_2d(&tmap_c, slab, n0, row0);
              tma_store_commit();
            }
            // bf16 copy of the row segment: 64 contiguous bytes per thread
            if (row0 + lane < M) {
              __nv_bfloat16* o2 = reinterpret_cast<__nv_bfloat16*>(e.out2) +
                                  static_cast<size_t>(row0 + lane) * e.ldo + n0;
              if (n0 + 32 <= N && o2_wide) {
                // two 32-byte stores: whole sectors (four 16-byte stores per row reach the L2 as
                // half-sector writes and count twice against its slice throughput)
#pragma unroll
                for (int j = 0; j < 2; ++j)
                  st_global_v8(o2 + 16 * j, pack_bf16x2(x[16 * j + 0], x[16 * j + 1]),
                               pack_bf16x2(x[16 * j + 2], x[16 * j + 3]),
                               pack_bf16x2(x[16 * j + 4], x[16 * j + 5]),
                               pack_bf16x2(x[16 * j + 6], x[16 * j + 7]),
                               pack_bf16x2(x[16 * j + 8], x[16 * j + 9]),
                               pack_bf16x2(x[16 * j + 10], x[16 * j + 11]),
                               pack_bf16x2(x[16 * j + 12], x[16 * j + 13]),
                               pack_bf16x2(x[16 * j + 14], x[16 * j + 15]));
              } else if (n0 + 32 <= N) {
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                  uint4 pk;
                  pk.x = pack_bf16x2(x[8 * j + 0], x[8 * j + 1]);
                  pk.y = pack_bf16x2(x[8 * j + 2], x[8 * j + 3]);
                  pk.z = pack_bf16x2(x[8 * j + 4], x[8 * j + 5]);
                  pk.w = pack_bf16x2(x[8 * j + 6], x[8 * j + 7]);
                  reinterpret_cast<uint4*>(o2)[j] = pk;
                }
              } else {
                _Pragma("unroll") for (int j = 0; j < 32; ++j)
                  if (n0 + j < N) o2[j] = __float2bfloat16_rn(x[j]);
              }
            }
            // refill this slab with the tile two chunks ahead once the store has read it
            if (lane == 0 && c + 2 < kColsPerWarp / 32 && n0 + 64 < N) {
              tma_store_wait_read<0>();
              const uint32_t xb = (c & 1) ? my_aux2_bar : my_aux_bar;
              mbar_arrive_expect_tx(xb, 4096);
              tma_load_2d(slab, &tmap_c, xb, n0 + 64, row0);
            }
          }
        }
        if (row0 + lane < M && n_base < N)
          e.ln_part_out[static_cast<size_t>(n_base / kColsPerWarp) * M + (row0 + lane)] =
              make_float2(sum1, sum2);
      } else if constexpr (TMA_EPI) {
        constexpr bool kOutF32 = (EPI == EPI_RESID_F32 || EPI == EPI_F32);
        if constexpr (kOutF32) {
          const bool reduce = (EPI == EPI_RESID_F32) || (e.beta != 0.f);
          uint32_t v[2][32];
          tmem_ld_32x32b_x32(t_row, v[0]);
#pragma unroll
          for (int c = 0; c < kColsPerWarp / 32; ++c) {
            tmem_ld_wait();
            if (c + 1 < kColsPerWarp / 32) tmem_ld_32x32b_x32(t_row + (c + 1) * 32, v[(c + 1) & 1]);
            else release_acc();
            const int n0 = n_base + c * 32;
            if (row0 < M && n0 < N) {
              float x[32];
              acc_plus_bias<EPI>(v[c & 1], n0, N, e, x);
              if constexpr (EPI == EPI_RESID_F32) {
                if (e.drop.thresh != 0u)
                  drop_apply_run<32>(x, static_cast<uint32_t>(row0 + lane) * static_cast<uint32_t>(N) +
                                            static_cast<uint32_t>(n0), e.drop);
              }
              uint32_t pk[32];
#pragma unroll
              for (int j = 0; j < 32; ++j) pk[j] = __float_as_uint(x[j]);
              stage_and_store(pk, stg, buf, lane, &tmap_c, n0, row0, reduce);
            }
          }
        } else {
#pragma unroll 1
          for (int g = 0; g < kColsPerWarp / 64; ++g) {
            uint32_t v0[32], v1[32];
            GT_BEGIN(gt_l);
            tmem_ld_32x32b_x32(t_row + g * 64, v0);
            tmem_ld_32x32b_x32(t_row + g * 64 + 32, v1);
            tmem_ld_wait();
            if (g + 1 == kColsPerWarp / 64) release_acc();
            GT_ADD(gt_epi_ld, gt_l);
            GT_BEGIN(gt_m);
            const int n0 = n_base + g * 64;
            if (row0 < M && n0 < N) {
              float x0[32], x1[32];
              if (e.ln_part != nullptr) {
                acc_scale_bias(v0, n0, N, e, ln_rstd, x0);
                acc_scale_bias(v1, n0 + 32, N, e, ln_rstd, x1);
              } else {
                acc_plus_bias<EPI>(v0, n0, N, e, x0);
                acc_plus_bias<EPI>(v1, n0 + 32, N, e, x1);
              }
              uint32_t pk[32];
              [[maybe_unused]] const uint32_t drop_idx0 =
                  static_cast<uint32_t>(row0 + lane) * static_cast<uint32_t>(N) +
                  static_cast<uint32_t>(n0);
              if constexpr (EPI == EPI_DGELU_BF16) {
                if (e.drop.thresh != 0u) {
                  drop_apply_run<32>(x0, drop_idx0, e.drop);
                  drop_apply_run<32>(x1, drop_idx0 + 32u, e.drop);
                }
              }
              if constexpr (kAuxTma) {
                // this lane's row of the pre-activation slab (64 bf16), then refill the slab with
                // the next group's tile while the math below runs
                mbar_wait(my_aux_bar, aux_phase);
                aux_phase ^= 1u;
                uint32_t a[32];
                const uint32_t arow = aux_slab + static_cast<uint32_t>(lane) * 128u;
#pragma unroll
                for (int j = 0; j < 8; ++j)
                  asm volatile("ld.shared.v4.b32 {%0,%1,%2,%3}, [%4];"
                               : "=r"(a[4 * j]), "=r"(a[4 * j + 1]), "=r"(a[4 * j + 2]),
                                 "=r"(a[4 * j + 3])
                               : "r"(arow + (static_cast<uint32_t>(j ^ (lane & 7)) << 4))
                               : "memory");
                __syncwarp();
                const int n_next = n0 + 64;
                if (lane == 0 && g + 1 < kColsPerWarp / 64 && n_next < N) {
                  mbar_arrive_expect_tx(my_aux_bar, 4096);
                  tma_load_2d(aux_slab, &tmap_c2, my_aux_bar, n_next, row0);
                }
#pragma unroll
                for (int j = 0; j < 16; ++j) {
                  dgelu_tanh_pair(x0[2 * j], x0[2 * j + 1], bf16lo_to_f32(a[j]), bf16hi_to_f32(a[j]));
                  dgelu_tanh_pair(x1[2 * j], x1[2 * j + 1], bf16lo_to_f32(a[16 + j]),
                                  bf16hi_to_f32(a[16 + j]));
                }
              }
              if constexpr (is_gelu_epi<EPI>()) {
                if (e.out2 != nullptr) {
#pragma unroll
                  for (int j = 0; j < 16; ++j) {
                    pk[j] = pack_bf16x2(x0[2 * j], x0[2 * j + 1]);
                    pk[16 + j] = pack_bf16x2(x1[2 * j], x1[2 * j + 1]);
                  }
                  stage_and_store(pk, stg, buf, lane, &tmap_c2, n0, row0, false);
                }
                if constexpr (EPI == EPI_RELU_BF16) {
#pragma unroll
                  for (int j = 0; j < 32; ++j) {
                    x0[j] = fmaxf(x0[j], 0.f);
                    x1[j] = fmaxf(x1[j], 0.f);
                  }
                } else if constexpr (EPI == EPI_GELU_TANH_BF16) {
#pragma unroll
                  for (int j = 0; j < 16; ++j) {
                    gelu_fast_tanh_pair(x0[2 * j], x0[2 * j + 1]);
                    gelu_fast_tanh_pair(x1[2 * j], x1[2 * j + 1]);
                  }
                } else {
#pragma unroll
                  for (int j = 0; j < 16; ++j) {
                    gelu_fast_pair(x0[2 * j], x0[2 * j + 1]);
                    gelu_fast_pair(x1[2 * j], x1[2 * j + 1]);
                  }
                }
                if (e.drop.thresh != 0u) {
                  drop_apply_run<32>(x0, drop_idx0, e.drop);
                  drop_apply_run<32>(x1, drop_idx0 + 32u, e.drop);
                }
              }
#pragma unroll
              for (int j = 0; j < 16; ++j) {
                pk[j] = pack_bf16x2(x0[2 * j], x0[2 * j + 1]);
                pk[16 + j] = pack_bf16x2(x1[2 * j], x1[2 * j + 1]);
              }
              GT_ADD(gt_epi_math, gt_m);
              GT_BEGIN(gt_s);
              stage_and_store(pk, stg, buf, lane, &tmap_c, n0, row0, false);
              GT_ADD(gt_epi_store, gt_s);
            }
          }
        }
      } else {
        const int m = row0 + lane;
        // two 32-column chunks in flight: the TMEM read of chunk c+1 overlaps the math of chunk c
        uint32_t v[2][32];
        tmem_ld_32x32b_x32(t_row, v[0]);
#pragma unroll
        for (int c = 0; c < kColsPerWarp / 32; ++c) {
          tmem_ld_wait();
          if (c + 1 < kColsPerWarp / 32) tmem_ld_32x32b_x32(t_row + (c + 1) * 32, v[(c + 1) & 1]);
          else release_acc();
          const int n0 = n_base + c * 32;
          if constexpr (EPI == EPI_RESID_F32) {
            if (row0 < M && n0 < N) resid_chunk_staged(v[c & 1], row0, n0, M, N, e, stg, lane);
          } else {
            if (m < M && n0 < N) epilogue_chunk<EPI>(v[c & 1], m, n0, N, e);
          }
        }
      }
      if (++acc == kAccStages) {
        acc = 0;
        acc_phase ^= 1u;
      }
      if constexpr (TMA_EPI && (EPI == EPI_BF16 || is_gelu_epi<EPI>())) {
        if (e.ln_part != nullptr && ln_have_next) {
          float s1 = 0.f, s2 = 0.f;
#pragma unroll
          for (int p2 = 0; p2 < 8; ++p2) {
            s1 += ln_next[p2].x;
            s2 += ln_next[p2].y;
          }
          ln_rstd_next = ln_finish(s1, s2);
        }
      }
    }
#ifdef VITK_GEMM_TRACE
    if (lane == 0 && warp == kFirstEpiWarp && is_leader && cluster_id < 160) {
      g_gemm_trace[cluster_id][4] = gt_epi_wait;
      g_gemm_trace[cluster_id][5] = gt_epi_ld;
      g_gemm_trace[cluster_id][6] = gt_epi_math;
      g_gemm_trace[cluster_id][7] = gt_epi_store;
    }
#endif
    if constexpr (TMA_EPI) {
      if (lane == 0) tma_store_wait<0>();  // all bulk stores of this warp have completed
    }
  }

  tc_fence_before();
  if constexpr (CTAS == 2) cluster_sync_all(); else __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    if constexpr (CTAS == 2) tmem_dealloc_2sm(tmem_base, C::kTmemCols);
    else tmem_dealloc(tmem_base, C::kTmemCols);
  }
}

int g_force_ctas = 0;        // 0 = auto, 1 / 2 = forced (tests, A/B timing)
int g_force_direct_epi = 0;  // 1 = never use the TMA-store epilogue (tests, A/B timing)

template <int BLOCK_N, int EPI, int CTAS, bool TMA_EPI, bool MN>
int launch(const GemmProblem& p, cudaStream_t stream) {
  using C = Cfg<BLOCK_N, CTAS, (TMA_EPI && EPI == EPI_DGELU_BF16) ? 3 : 2>;
  auto kernel = gemm_tn_kernel<BLOCK_N, EPI, CTAS, TMA_EPI, MN>;
  VITK_TRY((opt_in_smem<gemm_tn_kernel<BLOCK_N, EPI, CTAS, TMA_EPI, MN>>(C::kSmemBytes,
                                                                       "gemm_tn_kernel")));
  CUtensorMap ta, tb, tc, tc2;
  if constexpr (MN) {
    VITK_TRY(make_tmap_2d(&ta, p.A, 2, (uint64_t)p.M, (uint64_t)p.K, (uint64_t)p.lda * 2, 64, 64));
    VITK_TRY(make_tmap_2d(&tb, p.B, 2, (uint64_t)p.N, (uint64_t)p.K, (uint64_t)p.ldb * 2, 64, 64));
  } else {
    VITK_TRY(make_tmap_2d(&ta, p.A, 2, (uint64_t)p.K, (uint64_t)p.M, (uint64_t)p.lda * 2, kBlockK,
                          kBlockM));
    VITK_TRY(make_tmap_2d(&tb, p.B, 2, (uint64_t)p.K, (uint64_t)p.N, (uint64_t)p.ldb * 2, kBlockK,
                          C::kBRows));
  }
  if constexpr (TMA_EPI) {
    constexpr bool kOutF32 =
        (EPI == EPI_RESID_F32 || EPI == EPI_F32 || EPI == EPI_RESID_STATS_F32);
    constexpr int eb = kOutF32 ? 4 : 2;
    VITK_TRY(make_tmap_2d(&tc, p.e.out, eb, (uint64_t)p.N, (uint64_t)p.M, (uint64_t)p.e.ldo * eb,
                          128 / eb, 32));
    tc2 = tc;
    if (is_gelu_epi<EPI>() && p.e.out2 != nullptr)
      VITK_TRY(make_tmap_2d(&tc2, p.e.out2, eb, (uint64_t)p.N, (uint64_t)p.M,
                            (uint64_t)p.e.ldo * eb, 128 / eb, 32));
    if (EPI == EPI_DGELU_BF16)   // the pre-activation tile is TMA-loaded, same geometry as out
      VITK_TRY(make_tmap_2d(&tc2, p.e.aux, 2, (uint64_t)p.N, (uint64_t)p.M, (uint64_t)p.e.ldo * 2,
                            64, 32));
  } else {
    tc = ta;
    tc2 = ta;
  }
  const int tile_m = kBlockM * CTAS;
  const int num_kb = (p.K + kBlockK - 1) / kBlockK;
  int splits = p.split_k < 1 ? 1 : p.split_k;
  if (splits > num_kb) splits = num_kb;
  const int kb_per_split = (num_kb + splits - 1) / splits;
  splits = (num_kb + kb_per_split - 1) / kb_per_split;  // no empty K ranges
  const int num_tiles = ((p.M + tile_m - 1) / tile_m) * ((p.N + BLOCK_N - 1) / BLOCK_N) * splits;
  int grid = sm_count();
  if (grid <= 0) return set_error(VITK_ERR_NO_DEVICE, "no CUDA device");
  grid = grid / CTAS * CTAS;
  if (num_tiles * CTAS < grid) grid = num_tiles * CTAS;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(kNumThreads);
  cfg.dynamicSmemBytes = C::kSmemBytes;
  cfg.stream = stream;
  cudaLaunchAttribute attr;
  attr.id = cudaLaunchAttributeClusterDimension;
  attr.val.clusterDim.x = CTAS;
  attr.val.clusterDim.y = 1;
  attr.val.clusterDim.z = 1;
  cfg.attrs = &attr;
  cfg.numAttrs = 1;
  ProfileScope prof(PROF_GEMM, 2.0 * p.M * p.N * p.K, stream);
  const int descending = sweep_next();
  cudaError_t le = cudaLaunchKernelEx(&cfg, kernel, ta, tb, tc, tc2, p.M, p.N, p.K, kb_per_split,
                                      splits, descending, p.e);
  if (le != cudaSuccess)
    return set_error(VITK_ERR_CUDA, "launch of gemm_tn_kernel<%d,%d,%d,%d,%d> failed: %s", BLOCK_N,
                     EPI, CTAS, (int)TMA_EPI, (int)MN, cudaGetErrorString(le));
  VITK_CHECK_LAUNCH("gemm_tn_kernel");
  return VITK_OK;
}

template <int EPI, bool TMA_EPI, bool MN>
int dispatch_tile(const GemmProblem& p, cudaStream_t stream) {
  // 256-wide tiles unless they would waste more than a 128-wide tiling does.
  const int waste256 = ((p.N + 255) / 256) * 256 - p.N;
  const int waste128 = ((p.N + 127) / 128) * 128 - p.N;
  const bool n128 = waste128 < waste256;
  // CTA pairs (256-row tiles) whenever there is more than one 128-row tile of work
  int ctas = (p.M > kBlockM) ? 2 : 1;
  if (g_force_ctas == 1 || g_force_ctas == 2) ctas = g_force_ctas;
  if (ctas == 2)
    return n128 ? launch<128, EPI, 2, TMA_EPI, MN>(p, stream)
                : launch<256, EPI, 2, TMA_EPI, MN>(p, stream);
  // single-CTA tiles keep the direct epilogue for the gelu' variant (no room for a third slab)
  constexpr bool kTma1 = TMA_EPI && (EPI != EPI_DGELU_BF16);
  return n128 ? launch<128, EPI, 1, kTma1, MN>(p, stream)
              : launch<256, EPI, 1, kTma1, MN>(p, stream);
}

// The TMA epilogue needs 16-byte aligned output rows and, for the residual form, an in-place
// update without row remapping.
bool tma_epilogue_ok(const GemmProblem& p, bool honour_force = true) {
  if (honour_force && g_force_direct_epi) return false;
  const bool f32 = (p.epi == EPI_RESID_F32 || p.epi == EPI_F32 || p.epi == EPI_RESID_STATS_F32);
  const int eb = f32 ? 4 : 2;
  if ((reinterpret_cast<uintptr_t>(p.e.out) & 15) != 0 || (p.e.ldo * eb) % 16 != 0) return false;
  switch (p.epi) {
    case EPI_BF16: return true;
    case EPI_GELU_BF16:
    case EPI_GELU_TANH_BF16:
    case EPI_RELU_BF16:
      return p.e.out2 == nullptr || (reinterpret_cast<uintptr_t>(p.e.out2) & 15) == 0;
    case EPI_RESID_F32:
      return p.e.rows_per_group == 0 && p.e.resid == p.e.out && p.e.ldr == p.e.ldo;
    case EPI_RESID_STATS_F32:
      return p.e.rows_per_group == 0 && p.e.resid == p.e.out && p.e.ldr == p.e.ldo &&
             p.e.out2 != nullptr && (reinterpret_cast<uintptr_t>(p.e.out2) & 15) == 0;
    case EPI_F32: return p.e.beta == 0.f || p.e.beta == 1.f;
    case EPI_DGELU_BF16: return (reinterpret_cast<uintptr_t>(p.e.aux) & 15) == 0;
    default: return false;
  }
}

template <int EPI>
int dispatch(const GemmProblem& p, cudaStream_t stream) {
  if constexpr (EPI == EPI_DGELU_BF16) {
    if (tma_epilogue_ok(p)) return dispatch_tile<EPI, true, false>(p, stream);
    return dispatch_tile<EPI, false, false>(p, stream);
  } else if constexpr (EPI == EPI_F32) {
    if (p.mn_major) {
      // weight-gradient form: fp32 output through the TMA store / reduce-add epilogue only
      if (!tma_epilogue_ok(p, false) || (p.split_k > 1 && p.e.beta != 1.f))
        return set_error(VITK_ERR_INVALID,
                         "gemm: MN-major operands need beta in {0,1} (beta = 1 when split_k > 1)");
      return dispatch_tile<EPI, true, true>(p, stream);
    }
    if (tma_epilogue_ok(p)) return dispatch_tile<EPI, true, false>(p, stream);
    return dispatch_tile<EPI, false, false>(p, stream);
  } else {
    if (tma_epilogue_ok(p)) return dispatch_tile<EPI, true, false>(p, stream);
    return dispatch_tile<EPI, false, false>(p, stream);
  }
}

}  // namespace

int gemm_debug_trace(long long* out, int n) {
#ifdef VITK_GEMM_TRACE
  if (n > 160 * 8) n = 160 * 8;
  return cudaMemcpyFromSymbol(out, g_gemm_trace, static_cast<size_t>(n) * sizeof(long long)) ==
                 cudaSuccess ? n : -1;
#else
  (void)out;
  (void)n;
  return 0;   // not a trace build
#endif
}
void gemm_force_cta_group(int ctas) { g_force_ctas = ctas; }
void gemm_force_direct_epilogue(int on) { g_force_direct_epi = on; }
int gemm_stats_parts(int N) {
  // as dispatch_tile: 256-wide tiles unless they waste more than 128-wide ones; an epilogue warp
  // owns half a tile's columns
  const int waste256 = ((N + 255) / 256) * 256 - N;
  const int waste128 = ((N + 127) / 128) * 128 - N;
  const int cols = (waste128 < waste256) ? 64 : 128;
  return (N + cols - 1) / cols;
}

int gemm_bf16_tn(const GemmProblem& p, cudaStream_t stream) {
  VITK_REQUIRE(p.A && p.B && p.e.out, "gemm: null operand");
  VITK_REQUIRE(p.M > 0 && p.N > 0 && p.K > 0, "gemm: empty problem %dx%dx%d", p.M, p.N, p.K);
  VITK_REQUIRE(p.lda % 8 == 0 && p.ldb % 8 == 0 && (p.mn_major || p.K % 8 == 0),
               "gemm: K/lda/ldb must be multiples of 8 (got K=%d lda=%d ldb=%d)", p.K, p.lda,
               p.ldb);
  VITK_REQUIRE(!p.mn_major || p.epi == EPI_F32, "gemm: MN-major operands only with EPI_F32");
  VITK_REQUIRE(p.split_k <= 1 || p.epi == EPI_F32, "gemm: split_k only with EPI_F32");
  VITK_REQUIRE(p.split_k <= 1 || (p.e.beta == 1.f && p.e.bias == nullptr),
               "gemm: split_k > 1 accumulates (beta must be 1, no bias)");
  VITK_REQUIRE(p.N % 8 == 0 && p.e.ldo % 8 == 0, "gemm: N and ldo must be multiples of 8");
  VITK_REQUIRE(device_cc() >= 100, "gemm: requires an sm_100 device (found sm_%d)", device_cc());
  VITK_REQUIRE(p.e.drop.thresh == 0u ||
                   ((p.epi == EPI_RESID_F32 || p.epi == EPI_DGELU_BF16 || p.epi == EPI_GELU_BF16 ||
                     p.epi == EPI_GELU_TANH_BF16 || p.epi == EPI_RELU_BF16) &&
                    p.e.rows_per_group == 0 && p.N % 2 == 0 &&
                    static_cast<long long>(p.M) * p.N < (1ll << 32)),
               "gemm: dropout needs a residual / GELU / GELU' epilogue without row remap");
  if (p.e.ln_part != nullptr) {
    VITK_REQUIRE(p.epi == EPI_BF16 || p.epi == EPI_GELU_BF16 || p.epi == EPI_GELU_TANH_BF16 ||
                     p.epi == EPI_RELU_BF16,
                 "gemm: a folded LayerNorm needs a bf16-output epilogue");
    VITK_REQUIRE(p.e.bias && p.e.ln_nparts > 0 && p.e.ln_nparts <= 8 && p.e.ln_dim > 0,
                 "gemm: folded LayerNorm needs the folded bias and the row statistics");
    VITK_REQUIRE(tma_epilogue_ok(p, false), "gemm: folded LayerNorm needs 16-byte aligned outputs");
    switch (p.epi) {
      case EPI_BF16: return dispatch_tile<EPI_BF16, true, false>(p, stream);
      case EPI_GELU_BF16: return dispatch_tile<EPI_GELU_BF16, true, false>(p, stream);
      case EPI_GELU_TANH_BF16: return dispatch_tile<EPI_GELU_TANH_BF16, true, false>(p, stream);
      default: return dispatch_tile<EPI_RELU_BF16, true, false>(p, stream);
    }
  }
  switch (p.epi) {
    case EPI_RESID_STATS_F32:
      VITK_REQUIRE(p.e.resid != nullptr && p.e.ln_part_out != nullptr && p.e.drop.thresh == 0u,
                   "gemm: the statistics epilogue needs resid and ln_part_out (no dropout)");
      VITK_REQUIRE(tma_epilogue_ok(p, false),
                   "gemm: the statistics epilogue updates x in place (resid == out, no row remap) "
                   "and needs 16-byte aligned outputs");
      return dispatch_tile<EPI_RESID_STATS_F32, true, false>(p, stream);
    case EPI_BF16: return dispatch<EPI_BF16>(p, stream);
    case EPI_GELU_BF16: return dispatch<EPI_GELU_BF16>(p, stream);
    case EPI_GELU_TANH_BF16: return dispatch<EPI_GELU_TANH_BF16>(p, stream);
    case EPI_RELU_BF16: return dispatch<EPI_RELU_BF16>(p, stream);
    case EPI_RESID_F32:
      VITK_REQUIRE(p.e.resid != nullptr && p.e.ldr % 4 == 0, "gemm: residual epilogue needs resid");
      return dispatch<EPI_RESID_F32>(p, stream);
    case EPI_F32: return dispatch<EPI_F32>(p, stream);
    case EPI_DGELU_BF16:
      VITK_REQUIRE(p.e.aux != nullptr, "gemm: dgelu epilogue needs aux");
      return dispatch<EPI_DGELU_BF16>(p, stream);
    default: return set_error(VITK_ERR_INVALID, "gemm: unknown epilogue %d", (int)p.epi);
  }
}

int linear_fwd(const void* A, int lda, const void* W, int M, int N, int K, GemmEpi epi,
               const float* bias, const float* resid, int ldr, void* out, void* out2, int ldo,
               cudaStream_t stream, const DropParams& drop) {
  GemmProblem p;
  p.A = A;
  p.lda = lda;
  p.B = W;
  p.ldb = K;
  p.M = M;
  p.N = N;
  p.K = K;
  p.epi = epi;
  p.e.bias = bias;
  p.e.resid = resid;
  p.e.ldr = ldr;
  p.e.out = out;
  p.e.out2 = out2;
  p.e.ldo = ldo;
  p.e.drop = drop;
  return gemm_bf16_tn(p, stream);
}

int linear_dgrad(const void* dY, int out_f, const void* Wt, int M, int in_f, GemmEpi epi,
                 const void* aux, void* dX, float beta, cudaStream_t stream,
                 const DropParams& drop) {
  GemmProblem p;
  p.A = dY;
  p.lda = out_f;
  p.B = Wt;
  p.ldb = out_f;
  p.M = M;
  p.N = in_f;
  p.K = out_f;
  p.epi = epi;
  p.e.aux = aux;
  p.e.out = dX;
  p.e.ldo = in_f;
  p.e.beta = beta;
  p.e.drop = drop;
  return gemm_bf16_tn(p, stream);
}

int gemm_wgrad(const void* A, int lda, const void* B, int ldb, int M, int N, int K, float* out,
               int ldo, float alpha, float beta, int split_k, cudaStream_t stream) {
  GemmProblem p;
  p.A = A;
  p.lda = lda;
  p.B = B;
  p.ldb = ldb;
  p.M = M;
  p.N = N;
  p.K = K;
  p.epi = EPI_F32;
  p.mn_major = true;
  p.split_k = split_k;
  p.e.out = out;
  p.e.ldo = ldo;
  p.e.alpha = alpha;
  p.e.beta = beta;
  return gemm_bf16_tn(p, stream);
}

int linear_wgrad(const void* dY, int out_f, const void* X, int in_f, int rows, float* dW,
                 float* db, cudaStream_t stream) {
  // enough K splits to give every CTA pair about two work items
  const int tiles = ((out_f + 255) / 256) * ((in_f + 255) / 256);
  int split = (sm_count() / 2 * 2) / (tiles > 0 ? tiles : 1);
  if (split < 1) split = 1;
  const int num_kb = (rows + 63) / 64;
  if (split > num_kb / 4) split = num_kb / 4 > 0 ? num_kb / 4 : 1;
  VITK_TRY(gemm_wgrad(dY, out_f, X, in_f, out_f, in_f, rows, dW, in_f, 1.f, 1.f, split, stream));
  if (db != nullptr) VITK_TRY(colsum_bf16(dY, out_f, rows, out_f, db, stream));
  return VITK_OK;
}

int patch_embed(const void* patches, const void* W, int B, int P, int K, int D, int N, int prefix,
                const float* bias, const float* pos_embed, float* x, cudaStream_t stream) {
  GemmProblem p;
  p.A = patches;
  p.lda = K;
  p.B = W;
  p.ldb = K;
  p.M = B * P;
  p.N = D;
  p.K = K;
  p.epi = EPI_RESID_F32;
  p.e.bias = bias;
  p.e.resid = pos_embed;
  p.e.ldr = D;
  p.e.out = x;
  p.e.ldo = D;
  p.e.rows_per_group = P;
  p.e.group_stride = N;
  p.e.group_offset = prefix;
  return gemm_bf16_tn(p, stream);
}

int linear_resid_ln(const void* A, int lda, const void* W, int ldb, int M, int N, int K,
                    const float* bias, float* x, const float* gamma, const float* beta, float eps,
                    void* ln_out, float* mean_out, float* rstd_out, cudaStream_t stream) {
  GemmProblem p;
  p.A = A;
  p.lda = lda;
  p.B = W;
  p.ldb = ldb;
  p.M = M;
  p.N = N;
  p.K = K;
  p.epi = EPI_RESID_F32;
  p.e.bias = bias;
  p.e.resid = x;
  p.e.ldr = N;
  p.e.out = x;
  p.e.ldo = N;
  VITK_TRY(gemm_bf16_tn(p, stream));
  return layernorm_fwd(x, N, gamma, beta, ln_out, 0, N, mean_out, rstd_out, M, N, eps, stream);
}

int linear_resid_stats(const void* A, int lda, const void* W, int ldb, int M, int N, int K,
                       const float* bias, float* x, void* xb, float2* stats, cudaStream_t stream) {
  GemmProblem p;
  p.A = A;
  p.lda = lda;
  p.B = W;
  p.ldb = ldb;
  p.M = M;
  p.N = N;
  p.K = K;
  p.epi = EPI_RESID_STATS_F32;
  p.e.bias = bias;
  p.e.resid = x;
  p.e.ldr = N;
  p.e.out = x;
  p.e.out2 = xb;
  p.e.ldo = N;
  p.e.ln_part_out = stats;
  return gemm_bf16_tn(p, stream);
}

int linear_ln(const void* xb, int lda, const void* w_ln, int ldb, int M, int N, int K, GemmEpi epi,
              const float* b_ln, const float2* stats, int nparts, float eps, void* out, int ldo,
              cudaStream_t stream) {
  GemmProblem p;
  p.A = xb;
  p.lda = lda;
  p.B = w_ln;
  p.ldb = ldb;
  p.M = M;
  p.N = N;
  p.K = K;
  p.epi = epi;
  p.e.bias = b_ln;
  p.e.out = out;
  p.e.ldo = ldo;
  p.e.ln_part = stats;
  p.e.ln_nparts = nparts;
  p.e.ln_dim = K;
  p.e.ln_eps = eps;
  return gemm_bf16_tn(p, stream);
}

}  // namespace vitk
