// tcgen05 separate-source attention forward for every head_dim from 16 to 128 ("xr": ragged
// head_dim), with the envelope of attention_xtc.cu: at most 128 queries (one MMA tile) and at
// most 256 keys (one key block).  That covers the detection head's decoder attentions at any
// embed width (train.py's Config: D = 400, 8 heads of 50; 100 or 5 object queries against
// themselves or 196 patch tokens) and the CLS-only tail of the encoder (1 query, head_dim 16).
// Three modes: inference (no log-sum-exp), training (log-sum-exp [B, H, Nq]) and training with
// dropout on the attention probabilities (mask index ((b*H + h)*Nq + i)*round16(Nk) + j, applied
// after normalisation, exactly as attn_xmma_fwd_kernel does).
//
// The pipeline is attention_xtc.cu's (two items in flight, one per TMEM region and softmax
// warpgroup), with the head dimension padded to HDP = round16(hd):
//   load  64-column 128B-swizzled boxes of the head's columns.  hd a multiple of 8: by TMA from
//         element h*hd; columns [hd, HDP) of the Q tile then hold the next head and are zeroed
//         (swizzled addresses) by the MMA warp before S = Q K^T reads them.  Otherwise h*hd is
//         not 16-byte aligned, which a TMA box start must be: warp 0 stages the tiles with
//         thread loads (8, 4 or 2 bytes wide) and writes zeros past column hd itself.  Columns
//         past HDP are never contracted
//   MMA   S = Q K^T over HDP/16 k-steps; O = P V one 64-column N block per box
//   softmax + epilogue: thread == query row; O / rowsum leaves through thread stores of exactly
//         hd columns, as wide as the output's alignment allows (never a 64-column TMA store,
//         which would overwrite the neighbouring head another CTA is writing)
#include <cuda_bf16.h>

#include "attention_kernels.cuh"
#include "attention_xr.cuh"
#include "common.h"
#include "dropout.cuh"
#include "ptx.cuh"

namespace vitk {
using namespace ptx;

namespace {

constexpr int kThreads = 12 * 32;  // warp 0 TMA, 1 MMA, 2 TMEM alloc, 4-7 / 8-11 softmax groups
constexpr int kRegionCols = 256;   // per item: S [0,Nk) -> P [0,Nk/2), O [128, 128 + 64*NB)
constexpr int kOCol = 128;

struct XrParams {
  __nv_bfloat16* ctx;
  long long ctx_img;  // elements
  int ldc;
  int B, H, Nq, Nkeys, Nk;  // Nk = keys rounded up to 16
  int hd, vw;               // true head_dim, store width (elements)
  float scale;
  float* lse;  // optional [B, H, Nq]
  DropParams drop;
  // operands for the thread-staged path (tma == 0: hd not a multiple of 8)
  const __nv_bfloat16 *q, *k, *v;
  long long q_img, kv_img;
  int ldq, ldkv, tma;
};

template <int HDP>
__global__ void __launch_bounds__(kThreads, 1)
attn_xr_fwd_kernel(const __grid_constant__ CUtensorMap tm_q, const __grid_constant__ CUtensorMap tm_k,
                   const __grid_constant__ CUtensorMap tm_v, const XrParams p) {
  constexpr int NB = (HDP + 63) / 64;  // 64-column boxes per row
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = smem_u32(smem_raw);
  const uint32_t base = (raw_addr + 1023u) & ~1023u;
  uint8_t* smem = smem_raw + (base - raw_addr);

  const int Nk = p.Nk;
  const uint32_t box_q = 128u * 128u;
  const uint32_t box_kv = static_cast<uint32_t>(Nk) * 128u;
  const uint32_t sq = base;
  const uint32_t sk = sq + NB * box_q;
  const uint32_t sv0 = sk + NB * box_kv;  // two V buffers
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
  const int hd = p.hd;

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

  if (warp == 0 && !p.tma) {
    // ============ producer, head offset not 16-byte aligned: the warp stages the tiles ============
    int it = 0;
    for (int item = blockIdx.x; item < num_items; item += gridDim.x, ++it) {
      const int r = it & 1;
      const uint32_t k = (it >> 1) & 1;
      const int b = item / p.H, h = item - b * p.H;
      mbar_wait(qk_empty, (it & 1) ^ 1u);
      xr::load_tile(sq, box_q, p.q + b * p.q_img + h * hd, p.ldq, p.Nq, p.Nq, hd, HDP, lane, 32);
      xr::load_tile(sk, box_kv, p.k + b * p.kv_img + h * hd, p.ldkv, Nk, p.Nkeys, hd, HDP, lane, 32);
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) mbar_arrive(qk_full);
      mbar_wait(v_empty(r), k ^ 1u);
      // rows [Nkeys, Nk) zero: P is 0 there, and 0 * (stale value) must stay 0
      xr::load_tile(sv0 + r * NB * box_kv, box_kv, p.v + b * p.kv_img + h * hd, p.ldkv, Nk, p.Nkeys,
                    hd, HDP, lane, 32);
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) mbar_arrive(v_full(r));
    }
  } else if (warp == 0) {
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
          tma_load_3d(sq + x * box_q, &tm_q, qk_full, h * hd + 64 * x, 0, b);
          tma_load_3d(sk + x * box_kv, &tm_k, qk_full, h * hd + 64 * x, 0, b);
        }
        mbar_wait(v_empty(r), k ^ 1u);
        mbar_arrive_expect_tx(v_full(r), NB * box_kv);
#pragma unroll
        for (int x = 0; x < NB; ++x)
          tma_load_3d(sv0 + (r * NB + x) * box_kv, &tm_v, v_full(r), h * hd + 64 * x, 0, b);
      }
    }
  } else if (warp == 1) {
    // ============ MMA issuer (whole warp: it zeroes the Q padding, one lane issues) ============
    const uint32_t idesc_s = make_idesc_bf16(128, Nk);
    const uint32_t idesc_pv = make_idesc_bf16(128, 64, 0, 1);  // B (= V) is MN-major
    int n_it = 0;
    for (int item = blockIdx.x; item < num_items; item += gridDim.x) ++n_it;
    auto issue_s = [&](int it) {
      const int r = it & 1;
      const uint32_t k = (it >> 1) & 1;
      mbar_wait(qk_full, it & 1);
      if (p.tma && hd < HDP) {
        xr::zero_pad_cols(sq, box_q, 128, hd, HDP, lane, 32);
        fence_proxy_async_smem();
      }
      __syncwarp();
      mbar_wait(o_free(r), k ^ 1u);  // the region's previous item (it - 2) has been read out
      tc_fence_after();
      const uint32_t d_s = tmem_base + static_cast<uint32_t>(r * kRegionCols);
      if (lane == 0) {
#pragma unroll
        for (int ks = 0; ks < HDP / 16; ++ks) {
          const int x = ks >> 2, kk = ks & 3;
          const uint64_t q_desc = make_desc_sw128(sq + x * box_q, 16, 1024) + 2u * kk;
          const uint64_t k_desc = make_desc_sw128(sk + x * box_kv, 16, 1024) + 2u * kk;
          mma_bf16_ss(d_s, q_desc, k_desc, idesc_s, ks > 0 ? 1u : 0u);
        }
        mma_commit(s_full(r));
        mma_commit(qk_empty);
      }
      __syncwarp();
    };
    auto issue_pv = [&](int it) {
      const int r = it & 1;
      const uint32_t k = (it >> 1) & 1;
      mbar_wait(p_full(r), k);
      mbar_wait(v_full(r), k);
      tc_fence_after();
      const uint32_t region = tmem_base + static_cast<uint32_t>(r * kRegionCols);
      if (lane == 0) {
        for (int ks = 0; ks < Nk / 16; ++ks) {
#pragma unroll
          for (int x = 0; x < NB; ++x) {
            const uint64_t v_desc = make_desc_sw128(sv0 + (r * NB + x) * box_kv, box_kv, 1024) +
                                    static_cast<uint64_t>(ks) * 128u;
            mma_bf16_ts(region + kOCol + 64 * x, region + static_cast<uint32_t>(ks * 8), v_desc,
                        idesc_pv, ks > 0 ? 1u : 0u);
          }
        }
        mma_commit(o_full(r));
        mma_commit(v_empty(r));
      }
      __syncwarp();
    };
    if (n_it > 0) issue_s(0);
    for (int it = 0; it < n_it; ++it) {
      if (it + 1 < n_it) issue_s(it + 1);  // next scores run under this item's softmax
      issue_pv(it);
    }
  } else if (warp >= 4) {
    // ======================= softmax + output (thread == query row) =======================
    const int r = (warp - 4) >> 2;
    const int q = warp & 3;
    const float c = p.scale * kLog2e;
    const int N = p.Nkeys;
    const int row = q * 32 + lane;
    const bool warp_rows = q * 32 < p.Nq;
    const bool dropping = p.drop.thresh != 0u;
    const uint32_t region = tmem_base + (static_cast<uint32_t>(q * 32) << 16) +
                            static_cast<uint32_t>(r * kRegionCols);
    const int n32 = Nk >> 5;
    const bool tail16 = (Nk & 31) != 0;
    int it = r;
    for (int item = blockIdx.x + r * gridDim.x; item < num_items; item += 2 * gridDim.x, it += 2) {
      const uint32_t ph = (it >> 1) & 1;
      const int b = item / p.H, h = item - b * p.H;
      // element index of (row, key 0) in the dropout mask (pairs start at even keys: Nk is even)
      const uint32_t drop_row = (static_cast<uint32_t>(item) * static_cast<uint32_t>(p.Nq) +
                                 static_cast<uint32_t>(row)) * static_cast<uint32_t>(Nk);
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
        // ---- sweep 2: p = 2^((s - m) * c), row sum over every term, dropped / scaled P -> TMEM
        const float mc = m * c;
        float l = 0.f;
        auto pair = [&](uint32_t s0, uint32_t s1, int key) {
          float e0 = ex2_approx(fmaf(__uint_as_float(s0), c, -mc));
          float e1 = ex2_approx(fmaf(__uint_as_float(s1), c, -mc));
          if (key >= N) e0 = 0.f;
          if (key + 1 >= N) e1 = 0.f;
          l += e0 + e1;
          if (dropping) {
            const uint32_t bits = drop_bits((drop_row + static_cast<uint32_t>(key)) >> 1, p.drop.key);
            e0 = drop_keep_lo(bits, p.drop.thresh) ? e0 * p.drop.scale : 0.f;
            e1 = drop_keep_hi(bits, p.drop.thresh) ? e1 * p.drop.scale : 0.f;
          }
          return pack_bf16x2(e0, e1);
        };
        for (int ch = 0; ch < n32; ++ch) {
          uint32_t v[32];
          tmem_ld_32x32b_x32(region + ch * 32, v);
          tmem_ld_wait();
          uint32_t pk[16];
#pragma unroll
          for (int j = 0; j < 16; ++j) pk[j] = pair(v[2 * j], v[2 * j + 1], ch * 32 + 2 * j);
          tmem_st_32x32b_x16(region + ch * 16, pk);
        }
        if (tail16) {
          uint32_t v[16];
          tmem_ld_32x32b_x16(region + n32 * 32, v);
          tmem_ld_wait();
          uint32_t pk[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) pk[j] = pair(v[2 * j], v[2 * j + 1], n32 * 32 + 2 * j);
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

      // ---- O = P V is ready: normalise, convert, store hd columns of this thread's row
      mbar_wait(o_full(r), ph);
      tc_fence_after();
      if (warp_rows) {
        __nv_bfloat16* dst = p.ctx + b * p.ctx_img + static_cast<long long>(row) * p.ldc + h * hd;
#pragma unroll
        for (int ch = 0; ch < HDP / 16; ++ch) {
          uint32_t o[16];
          tmem_ld_32x32b_x16(region + kOCol + ch * 16, o);
          tmem_ld_wait();
          float f[16];
#pragma unroll
          for (int j = 0; j < 16; ++j) f[j] = __uint_as_float(o[j]) * inv_l;
          if (row < p.Nq) xr::store_cols16(dst, ch * 16, hd, p.vw, f);
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

size_t xr_fwd_smem(int hd, int Nk) {
  const size_t nb = (xr::pad16(hd) + 63) / 64, nk = xr::pad16(Nk);
  return nb * (128 * 128 + 3 * nk * 128) + 256 + 1024;
}

template <int HDP>
int launch_xr_fwd(const CUtensorMap& tq, const CUtensorMap& tk, const CUtensorMap& tv,
                  const XrParams& prm, size_t smem, cudaStream_t stream) {
  VITK_TRY(opt_in_smem<attn_xr_fwd_kernel<HDP>>(232448, "attn_xr_fwd_kernel"));
  const int grid = persistent_grid(static_cast<long long>(prm.B) * prm.H);
  attn_xr_fwd_kernel<HDP><<<grid, kThreads, smem, stream>>>(tq, tk, tv, prm);
  VITK_CHECK_LAUNCH("attn_xr_fwd_kernel");
  return VITK_OK;
}

}  // namespace

bool attention_src_supported(int Nq, int Nk, int hd) {
  return hd >= 16 && hd <= 128 && Nq >= 1 && Nq <= 128 && Nk >= 1 && Nk <= 256;
}

int attention_xr_fwd(const AttnXSrc& s, void* ctx, long long ctx_img, int ldc, float* lse, int B,
                     int Nq, int Nk, int H, int hd, cudaStream_t stream, const DropParams* drop) {
  VITK_REQUIRE(s.q && s.k && s.v && ctx, "attention(xr): null operand");
  VITK_REQUIRE(B > 0 && H > 0 && attention_src_supported(Nq, Nk, hd),
               "attention(xr): needs head_dim 16..128, <= 128 queries and <= 256 keys (got %d x %d, "
               "head_dim %d)", Nq, Nk, hd);
  VITK_REQUIRE(device_cc() >= 100, "attention(xr): needs an sm_100 device");
  long long q_img = s.q_img, kv_img = s.kv_img;
  if (B == 1) {  // a single image has no batch stride: any positive pitch describes it
    if (q_img <= 0) q_img = static_cast<long long>(Nq) * s.ldq;
    if (kv_img <= 0) kv_img = static_cast<long long>(Nk) * s.ldkv;
  }
  // TMA operands: 16-byte aligned bases, pitches and image strides (the box start h*hd is free)
  VITK_REQUIRE((reinterpret_cast<uintptr_t>(s.q) & 15) == 0 && (reinterpret_cast<uintptr_t>(s.k) & 15) == 0 &&
                   (reinterpret_cast<uintptr_t>(s.v) & 15) == 0 && s.ldq % 8 == 0 && s.ldkv % 8 == 0 &&
                   q_img % 8 == 0 && kv_img % 8 == 0 && q_img > 0 && kv_img > 0,
               "attention(xr): q / k / v need 16-byte aligned bases and pitches (multiples of 8 "
               "elements)");
  VITK_REQUIRE((reinterpret_cast<uintptr_t>(ctx) & 1) == 0 && (B == 1 || ctx_img > 0),
               "attention(xr): misaligned output");
  VITK_REQUIRE(drop == nullptr || drop->thresh == 0u ||
                   static_cast<long long>(B) * H * Nq * xr::pad16(Nk) < (1ll << 32),
               "attention dropout: batch * heads * queries * keys must stay below 2^32");
  const size_t smem = xr_fwd_smem(hd, Nk);
  VITK_REQUIRE(smem <= 232448, "attention(xr): shared memory budget exceeded");
  XrParams prm;
  prm.ctx = static_cast<__nv_bfloat16*>(ctx);
  prm.ctx_img = B == 1 ? 0 : ctx_img;
  prm.ldc = ldc;
  prm.B = B;
  prm.H = H;
  prm.Nq = Nq;
  prm.Nkeys = Nk;
  prm.Nk = xr::pad16(Nk);
  prm.hd = hd;
  prm.vw = xr::store_width(ctx, ctx_img, ldc, hd, B);
  prm.scale = 1.0f / sqrtf(static_cast<float>(hd));
  prm.lse = lse;
  // without the log-sum-exp this is the inference forward: no dropout
  if (drop != nullptr && lse != nullptr) prm.drop = *drop;
  prm.q = static_cast<const __nv_bfloat16*>(s.q);
  prm.k = static_cast<const __nv_bfloat16*>(s.k);
  prm.v = static_cast<const __nv_bfloat16*>(s.v);
  prm.q_img = B == 1 ? 0 : q_img;
  prm.kv_img = B == 1 ? 0 : kv_img;
  prm.ldq = s.ldq;
  prm.ldkv = s.ldkv;
  prm.tma = hd % 8 == 0;
  const int D = H * hd;
  CUtensorMap tq, tk, tv;
  VITK_TRY(make_row_map(&tq, s.q, B, Nq, D, s.ldq, 128, q_img));
  VITK_TRY(make_row_map(&tk, s.k, B, Nk, D, s.ldkv, prm.Nk, kv_img));
  VITK_TRY(make_row_map(&tv, s.v, B, Nk, D, s.ldkv, prm.Nk, kv_img));
  ProfileScope prof(PROF_ATTN, attention_flops(B, H, Nq, Nk, hd), stream);
  switch (xr::pad16(hd)) {
    case 16: return launch_xr_fwd<16>(tq, tk, tv, prm, smem, stream);
    case 32: return launch_xr_fwd<32>(tq, tk, tv, prm, smem, stream);
    case 48: return launch_xr_fwd<48>(tq, tk, tv, prm, smem, stream);
    case 64: return launch_xr_fwd<64>(tq, tk, tv, prm, smem, stream);
    case 80: return launch_xr_fwd<80>(tq, tk, tv, prm, smem, stream);
    case 96: return launch_xr_fwd<96>(tq, tk, tv, prm, smem, stream);
    case 112: return launch_xr_fwd<112>(tq, tk, tv, prm, smem, stream);
    default: return launch_xr_fwd<128>(tq, tk, tv, prm, smem, stream);
  }
}

}  // namespace vitk
