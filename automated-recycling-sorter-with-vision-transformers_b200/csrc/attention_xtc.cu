// tcgen05 form of the generic-source attention (attention_x.cu) for the detection head's decoder
// layers: softmax(q k^T / sqrt(hd)) v with separate query and key/value sources, head_dim 32 / 64 /
// 96 / 128, at most 128 queries (the 100 object queries are one MMA tile) and at most 256 keys
// (100 queries for self-attention, 196 patch tokens for cross-attention: one key block).
// Reference semantics: nn.MultiheadAttention inside nn.TransformerDecoderLayer, 8 heads,
// evaluation.py:170-177.
//
// Persistent CTAs loop over (image, head) items; two items are in flight, one per TMEM region and
// softmax warpgroup:
//   TMA   Q [128 x hd], K [Nk x hd] (single buffer: free again as soon as S = Q K^T has retired,
//         so the next item's Q/K arrive during this item's softmax) and V [Nk x hd] (two buffers),
//         as 64-column 128B-swizzled boxes (hd 96 = one full box + half of a second one; rows
//         beyond the valid queries / keys and columns beyond the row are zero-filled)
//   MMA   S = Q K^T: hd/16 k-steps, D = 128 x Nk fp32 in TMEM columns [0, Nk) of the region
//   softmax warpgroup (thread == query row): two sweeps over the row in TMEM (max; exp2 / sum),
//         P written back as packed bf16 over the dead S columns [0, Nk/2)
//   MMA   O = P V: A from TMEM, B = V from smem (MN-major), one MMA per 64-column box and
//         16-key step, D in TMEM columns [128, 128 + hd)
//   epilogue: O / rowsum -> bf16 -> 16-byte global stores (each thread owns one contiguous row)
// The issue order S(i+1) before P V(i) lets the tensor pipe compute the next scores while this
// item's softmax runs.
#include <cuda_bf16.h>

#include "attention_kernels.cuh"
#include "common.h"
#include "ptx.cuh"

namespace vitk {
using namespace ptx;

namespace {

constexpr int kThreads = 12 * 32;  // warp 0 TMA, 1 MMA, 2 TMEM alloc, 4-7 / 8-11 softmax groups
constexpr int kRegionCols = 256;   // per item: S [0,Nk) -> P [0,Nk/2), O [128, 128+hd)
constexpr int kOCol = 128;

struct XtcParams {
  __nv_bfloat16* ctx;
  long long ctx_img;  // elements
  int ldc;
  int B, H, Nq, Nkeys, Nk;  // Nk = keys rounded up to 16
  float scale;
  float* lse;  // optional [B, H, Nq]: natural log of the row sums of exp(scaled scores) (training)
};

template <int HD>
__global__ void __launch_bounds__(kThreads, 1)
attn_xtc_kernel(const __grid_constant__ CUtensorMap tm_q, const __grid_constant__ CUtensorMap tm_k,
                const __grid_constant__ CUtensorMap tm_v, const XtcParams p) {
  constexpr int NB = (HD + 63) / 64;        // 64-column boxes per row
  constexpr int LAST = HD - 64 * (NB - 1);  // columns used of the last box (32 or 64)
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = smem_u32(smem_raw);
  const uint32_t base = (raw_addr + 1023u) & ~1023u;
  uint8_t* smem = smem_raw + (base - raw_addr);

  const int Nk = p.Nk;
  const uint32_t box_q = 128u * 128u;                      // bytes of one Q box
  const uint32_t box_kv = static_cast<uint32_t>(Nk) * 128u;  // bytes of one K / V box
  const uint32_t sq = base;
  const uint32_t sk = sq + NB * box_q;
  const uint32_t sv0 = sk + NB * box_kv;                   // two V buffers
  const uint32_t bar_base = sv0 + 2u * NB * box_kv;
  const uint32_t qk_full = bar_base, qk_empty = bar_base + 8u;
  auto v_full = [&](int r) { return bar_base + 8u * (2 + r); };
  auto v_empty = [&](int r) { return bar_base + 8u * (4 + r); };
  auto s_full = [&](int r) { return bar_base + 8u * (6 + r); };
  auto p_full = [&](int r) { return bar_base + 8u * (8 + r); };
  auto o_full = [&](int r) { return bar_base + 8u * (10 + r); };
  auto o_free = [&](int r) { return bar_base + 8u * (12 + r); };
  volatile uint32_t* tmem_slot =
      reinterpret_cast<volatile uint32_t*>(smem + (bar_base - base) + 8 * 14);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int num_items = p.B * p.H;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tm_q);
    prefetch_tmap(&tm_k);
    prefetch_tmap(&tm_v);
  }
  if (warp == 1 && lane == 0) {
    mbar_init(qk_full, 1);
    mbar_init(qk_empty, 1);
    for (int r = 0; r < 2; ++r) {
      mbar_init(v_full(r), 1);
      mbar_init(v_empty(r), 1);
      mbar_init(s_full(r), 1);
      mbar_init(p_full(r), 4);
      mbar_init(o_full(r), 1);
      mbar_init(o_free(r), 4);
    }
    fence_mbar_init();
  }
  if (warp == 2) {
    tmem_alloc(smem_u32(const_cast<uint32_t*>(tmem_slot)), 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ======================= TMA producer =======================
    if (lane == 0) {
      int it = 0;
      for (int item = blockIdx.x; item < num_items; item += gridDim.x, ++it) {
        const int r = it & 1;
        const uint32_t k = (it >> 1) & 1;
        const int b = item / p.H, h = item - b * p.H;
        mbar_wait(qk_empty, (it & 1) ^ 1u);
        mbar_arrive_expect_tx(qk_full, NB * (box_q + box_kv));
#pragma unroll
        for (int x = 0; x < NB; ++x) {
          tma_load_3d(sq + x * box_q, &tm_q, qk_full, h * HD + 64 * x, 0, b);
          tma_load_3d(sk + x * box_kv, &tm_k, qk_full, h * HD + 64 * x, 0, b);
        }
        mbar_wait(v_empty(r), k ^ 1u);
        mbar_arrive_expect_tx(v_full(r), NB * box_kv);
#pragma unroll
        for (int x = 0; x < NB; ++x)
          tma_load_3d(sv0 + (r * NB + x) * box_kv, &tm_v, v_full(r), h * HD + 64 * x, 0, b);
      }
    }
  } else if (warp == 1) {
    // ======================= MMA issuer =======================
    if (lane == 0) {
      const uint32_t idesc_s = make_idesc_bf16(128, Nk);
      const uint32_t idesc_pv64 = make_idesc_bf16(128, 64, 0, 1);   // B (= V) is MN-major
      const uint32_t idesc_pvl = make_idesc_bf16(128, LAST, 0, 1);
      int n_it = 0;
      for (int item = blockIdx.x; item < num_items; item += gridDim.x) ++n_it;
      auto issue_s = [&](int it) {
        const int r = it & 1;
        const uint32_t k = (it >> 1) & 1;
        mbar_wait(qk_full, it & 1);
        mbar_wait(o_free(r), k ^ 1u);  // the region's previous item (it - 2) has been read out
        tc_fence_after();
        const uint32_t d_s = tmem_base + static_cast<uint32_t>(r * kRegionCols);
#pragma unroll
        for (int ks = 0; ks < HD / 16; ++ks) {
          const int x = ks >> 2, kk = ks & 3;  // box, 16-column step inside it (32 bytes)
          const uint64_t q_desc = make_desc_sw128(sq + x * box_q, 16, 1024) + 2u * kk;
          const uint64_t k_desc = make_desc_sw128(sk + x * box_kv, 16, 1024) + 2u * kk;
          mma_bf16_ss(d_s, q_desc, k_desc, idesc_s, ks > 0 ? 1u : 0u);
        }
        mma_commit(s_full(r));
        mma_commit(qk_empty);  // Q / K smem reusable once the MMAs above have retired
      };
      auto issue_pv = [&](int it) {
        const int r = it & 1;
        const uint32_t k = (it >> 1) & 1;
        mbar_wait(p_full(r), k);
        mbar_wait(v_full(r), k);
        tc_fence_after();
        const uint32_t region = tmem_base + static_cast<uint32_t>(r * kRegionCols);
        for (int ks = 0; ks < Nk / 16; ++ks) {
#pragma unroll
          for (int x = 0; x < NB; ++x) {
            // V box: rows = keys (128 B each, 8-row swizzle atoms 1024 B apart); 16 keys per MMA
            const uint64_t v_desc = make_desc_sw128(sv0 + (r * NB + x) * box_kv, box_kv, 1024) +
                                    static_cast<uint64_t>(ks) * 128u;
            mma_bf16_ts(region + kOCol + 64 * x, region + static_cast<uint32_t>(ks * 8), v_desc,
                        (x == NB - 1) ? idesc_pvl : idesc_pv64, ks > 0 ? 1u : 0u);
          }
        }
        mma_commit(o_full(r));
        mma_commit(v_empty(r));
      };
      if (n_it > 0) issue_s(0);
      for (int it = 0; it < n_it; ++it) {
        if (it + 1 < n_it) issue_s(it + 1);  // next scores run under this item's softmax
        issue_pv(it);
      }
    }
  } else if (warp >= 4) {
    // ======================= softmax + output (thread == query row) =======================
    const int r = (warp - 4) >> 2;  // region / item parity of this warpgroup
    const int q = warp & 3;         // TMEM lane quarter
    const float c = p.scale * kLog2e;
    const int N = p.Nkeys;
    const int row = q * 32 + lane;
    const bool warp_rows = q * 32 < p.Nq;
    const uint32_t region = tmem_base + (static_cast<uint32_t>(q * 32) << 16) +
                            static_cast<uint32_t>(r * kRegionCols);
    const int n32 = Nk >> 5;
    const bool tail16 = (Nk & 31) != 0;
    int it = r;
    for (int item = blockIdx.x + r * gridDim.x; item < num_items; item += 2 * gridDim.x, it += 2) {
      const uint32_t ph = (it >> 1) & 1;
      const int b = item / p.H, h = item - b * p.H;
      mbar_wait(s_full(r), ph);
      tc_fence_after();
      float inv_l = 0.f;
      if (warp_rows) {
        // ---- sweep 1: row max
        float m = -INFINITY;
        for (int ch = 0; ch < n32; ++ch) {
          uint32_t v[32];
          tmem_ld_32x32b_x32(region + ch * 32, v);
          tmem_ld_wait();
          const int k0 = ch * 32;
          if (k0 + 32 <= N) {
#pragma unroll
            for (int j = 0; j < 32; ++j) m = fmaxf(m, __uint_as_float(v[j]));
          } else {
#pragma unroll
            for (int j = 0; j < 32; ++j)
              if (k0 + j < N) m = fmaxf(m, __uint_as_float(v[j]));
          }
        }
        if (tail16) {
          uint32_t v[16];
          tmem_ld_32x32b_x16(region + n32 * 32, v);
          tmem_ld_wait();
          const int k0 = n32 * 32;
#pragma unroll
          for (int j = 0; j < 16; ++j)
            if (k0 + j < N) m = fmaxf(m, __uint_as_float(v[j]));
        }
        // ---- sweep 2: p = 2^((s - m) * c), row sum, P -> TMEM (bf16 pairs over dead S columns)
        const float mc = m * c;
        float l = 0.f;
        for (int ch = 0; ch < n32; ++ch) {
          uint32_t v[32];
          tmem_ld_32x32b_x32(region + ch * 32, v);
          tmem_ld_wait();
          const int k0 = ch * 32;
          uint32_t pk[16];
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            float e0 = ex2_approx(fmaf(__uint_as_float(v[2 * j]), c, -mc));
            float e1 = ex2_approx(fmaf(__uint_as_float(v[2 * j + 1]), c, -mc));
            if (k0 + 32 > N) {
              if (k0 + 2 * j >= N) e0 = 0.f;
              if (k0 + 2 * j + 1 >= N) e1 = 0.f;
            }
            l += e0 + e1;
            pk[j] = pack_bf16x2(e0, e1);
          }
          tmem_st_32x32b_x16(region + ch * 16, pk);
        }
        if (tail16) {
          uint32_t v[16];
          tmem_ld_32x32b_x16(region + n32 * 32, v);
          tmem_ld_wait();
          const int k0 = n32 * 32;
          uint32_t pk[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            float e0 = ex2_approx(fmaf(__uint_as_float(v[2 * j]), c, -mc));
            float e1 = ex2_approx(fmaf(__uint_as_float(v[2 * j + 1]), c, -mc));
            if (k0 + 2 * j >= N) e0 = 0.f;
            if (k0 + 2 * j + 1 >= N) e1 = 0.f;
            l += e0 + e1;
            pk[j] = pack_bf16x2(e0, e1);
          }
          tmem_st_32x32b_x8(region + n32 * 16, pk);
        }
        tmem_st_wait();
        inv_l = 1.f / l;
        if (p.lse != nullptr && row < p.Nq)
          p.lse[static_cast<long long>(item) * p.Nq + row] = fmaf(m, p.scale, __logf(l));
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(p_full(r));

      // ---- O = P V is ready: normalise, convert, store this thread's row
      mbar_wait(o_full(r), ph);
      tc_fence_after();
      if (warp_rows) {
        __nv_bfloat16* dst = p.ctx + b * p.ctx_img + static_cast<long long>(row) * p.ldc + h * HD;
#pragma unroll
        for (int ch = 0; ch < HD / 32; ++ch) {
          uint32_t o[32];
          tmem_ld_32x32b_x32(region + kOCol + ch * 32, o);
          tmem_ld_wait();
          if (row < p.Nq) {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              uint4 w;
              w.x = pack_bf16x2(__uint_as_float(o[8 * j + 0]) * inv_l, __uint_as_float(o[8 * j + 1]) * inv_l);
              w.y = pack_bf16x2(__uint_as_float(o[8 * j + 2]) * inv_l, __uint_as_float(o[8 * j + 3]) * inv_l);
              w.z = pack_bf16x2(__uint_as_float(o[8 * j + 4]) * inv_l, __uint_as_float(o[8 * j + 5]) * inv_l);
              w.w = pack_bf16x2(__uint_as_float(o[8 * j + 6]) * inv_l, __uint_as_float(o[8 * j + 7]) * inv_l);
              *reinterpret_cast<uint4*>(dst + ch * 32 + j * 8) = w;
            }
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(o_free(r));
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

template <int HD>
int launch_xtc(const void* q, long long q_img, int ldq, const void* k, const void* v,
               long long kv_img, int ldkv, const XtcParams& prm, cudaStream_t stream) {
  constexpr int NB = (HD + 63) / 64;
  const size_t smem = static_cast<size_t>(NB) * (128 * 128 + 3 * static_cast<size_t>(prm.Nk) * 128) +
                      256 + 1024;
  VITK_REQUIRE(smem <= 232448, "attention(xtc): shared memory budget exceeded");
  VITK_TRY(opt_in_smem<attn_xtc_kernel<HD>>(232448, "attn_xtc_kernel"));
  const int D = prm.H * HD;
  CUtensorMap tq, tk, tv;
  VITK_TRY(make_row_map(&tq, q, prm.B, prm.Nq, D, ldq, 128, q_img));
  VITK_TRY(make_row_map(&tk, k, prm.B, prm.Nkeys, D, ldkv, prm.Nk, kv_img));
  VITK_TRY(make_row_map(&tv, v, prm.B, prm.Nkeys, D, ldkv, prm.Nk, kv_img));
  const int grid = persistent_grid(prm.B * prm.H);
  attn_xtc_kernel<HD><<<grid, kThreads, smem, stream>>>(tq, tk, tv, prm);
  VITK_CHECK_LAUNCH("attn_xtc_kernel");
  return VITK_OK;
}

}  // namespace

bool attention_xtc_applicable(long long q_img, long long kv_img, int B, int Nq, int Nk, int hd) {
  if (device_cc() < 100) return false;
  if (!(hd == 32 || hd == 64 || hd == 96 || hd == 128)) return false;
  if (Nq > 128 || Nk > 256) return false;
  if (B > 1 && (q_img <= 0 || kv_img <= 0)) return false;
  const int nb = (hd + 63) / 64, nk = (Nk + 15) & ~15;
  return static_cast<size_t>(nb) * (128 * 128 + 3 * static_cast<size_t>(nk) * 128) + 1280 <= 232448;
}

int attention_xtc(const void* q, long long q_img, int ldq, const void* k, const void* v,
                  long long kv_img, int ldkv, void* ctx, long long ctx_img, int ldc, int B, int Nq,
                  int Nk, int H, int hd, cudaStream_t stream, float* lse) {
  VITK_REQUIRE(q && k && v && ctx, "attention: null operand");
  VITK_REQUIRE(attention_xtc_applicable(q_img, kv_img, B, Nq, Nk, hd),
               "attention(xtc): needs <= 128 queries, <= 256 keys, head_dim 32/64/96/128");
  VITK_REQUIRE(ldc % 8 == 0 && ctx_img % 8 == 0 && (reinterpret_cast<uintptr_t>(ctx) & 15) == 0,
               "attention(xtc): output must be 16-byte aligned");
  XtcParams prm;
  prm.ctx = static_cast<__nv_bfloat16*>(ctx);
  prm.ctx_img = ctx_img;
  prm.ldc = ldc;
  prm.B = B;
  prm.H = H;
  prm.Nq = Nq;
  prm.Nkeys = Nk;
  prm.Nk = (Nk + 15) & ~15;
  prm.scale = 1.0f / sqrtf(static_cast<float>(hd));
  prm.lse = lse;
  // a single image has no batch stride: any positive pitch describes it
  if (B == 1) {
    if (q_img <= 0) q_img = static_cast<long long>(Nq) * ldq;
    if (kv_img <= 0) kv_img = static_cast<long long>(Nk) * ldkv;
  }
  ProfileScope prof(PROF_ATTN, attention_flops(B, H, Nq, Nk, hd), stream);
  switch (hd) {
    case 32: return launch_xtc<32>(q, q_img, ldq, k, v, kv_img, ldkv, prm, stream);
    case 64: return launch_xtc<64>(q, q_img, ldq, k, v, kv_img, ldkv, prm, stream);
    case 96: return launch_xtc<96>(q, q_img, ldq, k, v, kv_img, ldkv, prm, stream);
    default: return launch_xtc<128>(q, q_img, ldq, k, v, kv_img, ldkv, prm, stream);
  }
}

}  // namespace vitk
