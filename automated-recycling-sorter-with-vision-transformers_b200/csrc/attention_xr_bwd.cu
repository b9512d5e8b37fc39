// tcgen05 backward of the separate-source attention for every head_dim from 16 to 128 ("xr"), at
// most 128 queries and 256 keys: the training counterpart of attention_xr.cu for the detection
// head's decoder attentions at any embed width (train.py's D = 400: 8 heads of 50, 5 queries).
//
// The S-transposed formulation of attention_bwd_tc.cu (M = 128 keys, N = queries padded to 16,
// which suits 5 queries), one (image, head) per work item, persistent CTAs; HDP = round16(hd):
//
//   for key tile kt (128 keys; at most two):
//     S^T  = K_kt Q^T       A, B from smem (K-major)                 -> TMEM [0, 128)
//     dP^T = V_kt dO^T      A, B from smem (K-major)                 -> TMEM [128, 256)
//     warps 4-11 (thread = key row x half of the query chunks): P^T = exp2(S^T c - lse_q),
//           dS^T = P^T (drop(dP^T) - D_q) scale; P^T (dropped) and dS^T -> TMEM as bf16 in place,
//           dS^T also -> smem tile kt
//     dV_kt = P^T dO        A from TMEM, B = dO (MN-major), one 64-column N block per box -> [256, 384)
//     dK_kt = dS^T Q        A from TMEM, B = Q  (MN-major)                               -> [384, 512)
//   after the key tiles: dQ = sum_kt dS_kt K_kt (A = dS^T tiles read as MN-major, B = K) into
//   the columns S^T and dP^T have freed, [0, 128).
//
// Shared memory: Q, dO, every K tile, one V tile (the next one streams in once dP^T of the
// current one has retired) and the dS^T tiles: about 226 KB at HDP = 128 and 256 keys.
// Operands arrive by TMA when hd is a multiple of 8; columns [hd, HDP) of Q and dO then hold the
// next head's values and are zeroed before the MMAs that contract over the head dimension read
// them (S^T and dP^T).  Otherwise the head's offset h*hd is not 16-byte aligned, which a TMA box
// start must be, and warp 0 stages every tile with thread loads, zeros past column hd included.
// The padded columns of dQ, dK and dV are never stored; every output leaves through thread stores
// of exactly hd columns.
// Dropout: mask index ((b*H + h)*Nq + i)*round16(Nk) + j, as the forward kernels use it.
#include <cuda_bf16.h>

#include "attention_kernels.cuh"
#include "attention_xr.cuh"
#include "common.h"
#include "dropout.cuh"
#include "ptx.cuh"

namespace vitk {
using namespace ptx;

namespace {

// warp 0 TMA, 1 MMA, 2 TMEM alloc, 2-3 per-row vectors, 4-11 softmax backward / epilogue
constexpr int kThreads = 12 * 32;
constexpr uint32_t kColS = 0, kColDP = 128, kColDV = 256, kColDK = 384, kColDQ = 0;
constexpr uint32_t kBox = 128u * 128u;  // one 64-column box of 128 rows
constexpr uint32_t kDsTile = 2u * kBox; // dS^T of one key tile: 128 keys x 2 chunks of 64 queries

struct XrBwdParams {
  const __nv_bfloat16 *ctx, *dctx;
  __nv_bfloat16 *dq, *dk, *dv;
  const float* lse;
  long long ctx_img, dq_img, dkv_img;
  int ldc, lddq, lddkv;
  int B, H, Nq, Nq16, Nkeys, Nk16, n_kt, hd, vw_q, vw_kv;
  float scale;
  DropParams drop;
  // operands for the thread-staged path (tma == 0: hd not a multiple of 8)
  const __nv_bfloat16 *q, *k, *v;
  long long q_img, kv_img;
  int ldq, ldkv, tma;
};

template <int HDP>
__global__ void __launch_bounds__(kThreads, 1)
attn_xr_bwd_kernel(const __grid_constant__ CUtensorMap tm_q, const __grid_constant__ CUtensorMap tm_do,
                   const __grid_constant__ CUtensorMap tm_k, const __grid_constant__ CUtensorMap tm_v,
                   const XrBwdParams p) {
  constexpr int NB = (HDP + 63) / 64;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = smem_u32(smem_raw);
  const uint32_t base = (raw_addr + 1023u) & ~1023u;
  uint8_t* smem = smem_raw + (base - raw_addr);

  const int n_kt = p.n_kt, hd = p.hd, Nq16 = p.Nq16;
  const uint32_t sQ = base, sdO = sQ + NB * kBox, sK = sdO + NB * kBox;
  const uint32_t sV = sK + static_cast<uint32_t>(n_kt) * NB * kBox;
  const uint32_t sdS = sV + NB * kBox;
  const uint32_t vec_off = sdS + static_cast<uint32_t>(n_kt) * kDsTile - base;
  float* sLse = reinterpret_cast<float*>(smem + vec_off);  // lse_q * log2(e), +inf past Nq
  float* sD = sLse + 128;                                   // -scale * rowsum(dO * O)
  const uint32_t bar_base = base + vec_off + 1024u;
  auto bar = [&](int i) { return bar_base + 8u * i; };
  // 0 ld_full, 1 op_free, 2 v_full, 3 v_free, 4 s_full, 5 sm_done, 6 dkv_full, 7 dkv_free,
  // 8 dq_full, 9 dq_free, 10 vec_full, 11 vec_free
  volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(smem + vec_off + 1024 + 128);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int num_items = p.B * p.H;
  auto rows_in_tile = [&](int t) { return min(128, p.Nk16 - t * 128); };  // multiple of 16

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tm_q);
    prefetch_tmap(&tm_do);
    prefetch_tmap(&tm_k);
    prefetch_tmap(&tm_v);
  }
  if (warp == 1 && lane == 0) {
    const uint32_t counts[12] = {1, 1, 1, 1, 1, 8, 1, 8, 1, 8, 2, 8};
    for (int i = 0; i < 12; ++i) mbar_init(bar(i), counts[i]);
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
    // (rows up to Nq16 / the key tile's 16-rounded end are written, zeros past the valid ones:
    // the MMAs read them, and a zero probability times a stale value must stay zero)
    int it = 0;
    uint32_t tc = 0;
    for (int item = blockIdx.x; item < num_items; item += gridDim.x, ++it) {
      const int b = item / p.H, h = item - b * p.H;
      mbar_wait(bar(1), (it & 1) ^ 1u);
      const __nv_bfloat16* kb = p.k + b * p.kv_img + h * hd;
      const __nv_bfloat16* vb = p.v + b * p.kv_img + h * hd;
      xr::load_tile(sQ, kBox, p.q + b * p.q_img + h * hd, p.ldq, Nq16, p.Nq, hd, HDP, lane, 32);
      xr::load_tile(sdO, kBox, p.dctx + b * p.ctx_img + h * hd, p.ldc, Nq16, p.Nq, hd, HDP, lane, 32);
      for (int kt = 0; kt < n_kt; ++kt)
        xr::load_tile(sK + kt * NB * kBox, kBox, kb + static_cast<long long>(kt) * 128 * p.ldkv,
                      p.ldkv, rows_in_tile(kt), p.Nkeys - kt * 128, hd, HDP, lane, 32);
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) mbar_arrive(bar(0));
      for (int kt = 0; kt < n_kt; ++kt, ++tc) {
        mbar_wait(bar(3), (tc & 1) ^ 1u);
        xr::load_tile(sV, kBox, vb + static_cast<long long>(kt) * 128 * p.ldkv, p.ldkv,
                      rows_in_tile(kt), p.Nkeys - kt * 128, hd, HDP, lane, 32);
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) mbar_arrive(bar(2));
      }
    }
  } else if (warp == 0) {
    // ======================= TMA producer =======================
    if (lane == 0) {
      int it = 0;
      uint32_t tc = 0;  // running key-tile counter (phases of v_full / v_free)
      for (int item = blockIdx.x; item < num_items; item += gridDim.x, ++it) {
        const int b = item / p.H, h = item - b * p.H;
        mbar_wait(bar(1), (it & 1) ^ 1u);  // every MMA of the previous item has retired
        mbar_arrive_expect_tx(bar(0), static_cast<uint32_t>(2 + n_kt) * NB * kBox);
        for (int x = 0; x < NB; ++x) {
          tma_load_3d(sQ + x * kBox, &tm_q, bar(0), h * hd + 64 * x, 0, b);
          tma_load_3d(sdO + x * kBox, &tm_do, bar(0), h * hd + 64 * x, 0, b);
          for (int kt = 0; kt < n_kt; ++kt)
            tma_load_3d(sK + (kt * NB + x) * kBox, &tm_k, bar(0), h * hd + 64 * x, kt * 128, b);
        }
        for (int kt = 0; kt < n_kt; ++kt, ++tc) {
          mbar_wait(bar(3), (tc & 1) ^ 1u);  // dP^T of the previous tile has read the V buffer
          mbar_arrive_expect_tx(bar(2), NB * kBox);
          for (int x = 0; x < NB; ++x)
            tma_load_3d(sV + x * kBox, &tm_v, bar(2), h * hd + 64 * x, kt * 128, b);
        }
      }
    }
  } else if (warp == 1) {
    // ============ MMA issuer (whole warp: it zeroes the padding, one elected lane issues) ============
    const uint32_t idesc_s = make_idesc_bf16(128, Nq16);
    const uint32_t idesc_mn = make_idesc_bf16(128, 64, 0, 1);  // A K-major / TMEM, B MN-major
    const uint32_t idesc_dq = make_idesc_bf16(128, 64, 1, 1);  // A and B MN-major
    int it = 0;
    uint32_t tc = 0;
    for (int item = blockIdx.x; item < num_items; item += gridDim.x, ++it) {
      mbar_wait(bar(0), it & 1);
      if (p.tma && hd < HDP) {
        xr::zero_pad_cols(sQ, kBox, 128, hd, HDP, lane, 32);
        xr::zero_pad_cols(sdO, kBox, 128, hd, HDP, lane, 32);
        fence_proxy_async_smem();
      }
      __syncwarp();
      mbar_wait(bar(9), (it & 1) ^ 1u);  // dQ of the previous item has been read out of TMEM
      tc_fence_after();
      for (int kt = 0; kt < n_kt; ++kt, ++tc) {
        mbar_wait(bar(2), tc & 1);  // V tile
        tc_fence_after();
        if (elect_one_sync()) {
#pragma unroll
          for (int ks = 0; ks < HDP / 16; ++ks) {
            const int x = ks >> 2, kk = ks & 3;
            const uint64_t ak = make_desc_sw128(sK + (kt * NB + x) * kBox, 16, 1024) + 2u * kk;
            const uint64_t bq = make_desc_sw128(sQ + x * kBox, 16, 1024) + 2u * kk;
            mma_bf16_ss(tmem_base + kColS, ak, bq, idesc_s, ks > 0 ? 1u : 0u);
          }
#pragma unroll
          for (int ks = 0; ks < HDP / 16; ++ks) {
            const int x = ks >> 2, kk = ks & 3;
            const uint64_t av = make_desc_sw128(sV + x * kBox, 16, 1024) + 2u * kk;
            const uint64_t bdo = make_desc_sw128(sdO + x * kBox, 16, 1024) + 2u * kk;
            mma_bf16_ss(tmem_base + kColDP, av, bdo, idesc_s, ks > 0 ? 1u : 0u);
          }
          mma_commit(bar(4));  // S^T, dP^T ready
          mma_commit(bar(3));  // V buffer free
        }
        __syncwarp();
        mbar_wait(bar(5), tc & 1);         // P^T / dS^T in TMEM, dS^T in smem
        mbar_wait(bar(7), (tc & 1) ^ 1u);  // dV / dK of the previous tile have been read
        tc_fence_after();
        if (elect_one_sync()) {
          for (int ks = 0; ks < Nq16 / 16; ++ks) {
            // 16 queries per step: bf16 pairs at the start of their 32-column chunk
            const uint32_t acol = static_cast<uint32_t>((ks >> 1) * 32 + (ks & 1) * 8);
#pragma unroll
            for (int x = 0; x < NB; ++x) {
              const uint64_t b_do = make_desc_sw128(sdO + x * kBox, kBox, 1024) + static_cast<uint64_t>(ks) * 128u;
              const uint64_t b_q = make_desc_sw128(sQ + x * kBox, kBox, 1024) + static_cast<uint64_t>(ks) * 128u;
              mma_bf16_ts(tmem_base + kColDV + 64 * x, tmem_base + kColS + acol, b_do, idesc_mn,
                          ks > 0 ? 1u : 0u);
              mma_bf16_ts(tmem_base + kColDK + 64 * x, tmem_base + kColDP + acol, b_q, idesc_mn,
                          ks > 0 ? 1u : 0u);
            }
          }
          mma_commit(bar(6));  // dV_kt, dK_kt complete
        }
        __syncwarp();
      }
      // ---- dQ = sum over key tiles of dS K (A = dS^T tile as MN-major: 2 chunks of 64 queries)
      if (elect_one_sync()) {
        for (int kt = 0; kt < n_kt; ++kt) {
          const uint64_t a_ds = make_desc_sw128(sdS + kt * kDsTile, kBox, 1024);
          for (int ks = 0; ks < rows_in_tile(kt) / 16; ++ks) {
#pragma unroll
            for (int x = 0; x < NB; ++x) {
              const uint64_t b_k = make_desc_sw128(sK + (kt * NB + x) * kBox, kBox, 1024) +
                                   static_cast<uint64_t>(ks) * 128u;
              mma_bf16_ss(tmem_base + kColDQ + 64 * x, a_ds + static_cast<uint64_t>(ks) * 128u, b_k,
                          idesc_dq, (kt > 0 || ks > 0) ? 1u : 0u);
            }
          }
        }
        mma_commit(bar(8));  // dQ complete
        mma_commit(bar(1));  // operands of this item no longer needed
      }
      __syncwarp();
    }
  } else if (warp == 2 || warp == 3) {
    // ============ per-row vectors: lse_q * log2(e), -scale * rowsum(dO * O) (a warp per row) ====
    int it = 0;
    for (int item = blockIdx.x; item < num_items; item += gridDim.x, ++it) {
      const int b = item / p.H, h = item - b * p.H;
      mbar_wait(bar(11), (it & 1) ^ 1u);  // the previous item's softmax is done with the vectors
      const __nv_bfloat16* ob = p.ctx + b * p.ctx_img + h * hd;
      const __nv_bfloat16* dob = p.dctx + b * p.ctx_img + h * hd;
      for (int r = warp - 2; r < 128; r += 2) {
        float dsum = 0.f;
        if (r < p.Nq) {
          const long long ro = static_cast<long long>(r) * p.ldc;
          for (int c = lane; c < hd; c += 32)
            dsum += __bfloat162float(ob[ro + c]) * __bfloat162float(dob[ro + c]);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) dsum += __shfl_xor_sync(0xffffffffu, dsum, o);
        if (lane == 0) {
          sLse[r] = r < p.Nq ? p.lse[static_cast<long long>(item) * p.Nq + r] * kLog2e : INFINITY;
          sD[r] = -dsum * p.scale;
        }
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(bar(10));
    }
  } else if (warp >= 4) {
    // ======================= softmax backward + outputs =======================
    const int q4 = warp & 3;
    const int hf = (warp - 4) >> 2;  // which half of the query chunks
    const int row_in_tile = q4 * 32 + lane;
    const float c = p.scale * kLog2e;
    const uint32_t lane_base = tmem_base + (static_cast<uint32_t>(q4 * 32) << 16);
    const bool dropping = p.drop.thresh != 0u;
    const int nch = (Nq16 + 31) / 32;
    const int ch_mid = (nch + 1) >> 1;
    int it = 0;
    uint32_t tc = 0;

    // 16-column chunks [ch0, ch1) step `step` of this warp's TMEM rows -> bf16 row `dst`
    auto store_rows = [&](uint32_t col0, int ch0, int step, __nv_bfloat16* dst, bool row_ok, int vw) {
      for (int ch = ch0; ch < HDP / 16; ch += step) {
        uint32_t o[16];
        tmem_ld_32x32b_x16(lane_base + col0 + ch * 16, o);
        tmem_ld_wait();
        float f[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) f[j] = __uint_as_float(o[j]);
        if (row_ok) xr::store_cols16(dst, ch * 16, hd, vw, f);
      }
    };

    for (int item = blockIdx.x; item < num_items; item += gridDim.x, ++it) {
      const int b = item / p.H, h = item - b * p.H;
      mbar_wait(bar(10), it & 1);
      const uint32_t drop_item = static_cast<uint32_t>(item) * static_cast<uint32_t>(p.Nq);
      for (int kt = 0; kt < n_kt; ++kt, ++tc) {
        const int key = kt * 128 + row_in_tile;
        const bool key_ok = key < p.Nkeys;
        mbar_wait(bar(4), tc & 1);
        tc_fence_after();
        for (int ch = hf == 0 ? 0 : ch_mid; ch < (hf == 0 ? ch_mid : nch); ++ch) {
          // chunks of 32 queries; the last chunk of a ragged tile holds 16
          const bool half_chunk = (ch * 32 + 32 > Nq16);
          uint32_t s[32], dp[32];
          if (half_chunk) {
            uint32_t s16[16], d16[16];
            tmem_ld_32x32b_x16(lane_base + kColS + ch * 32, s16);
            tmem_ld_32x32b_x16(lane_base + kColDP + ch * 32, d16);
            tmem_ld_wait();
#pragma unroll
            for (int j = 0; j < 16; ++j) {
              s[j] = s16[j];
              dp[j] = d16[j];
              s[16 + j] = 0u;
              dp[16 + j] = 0u;
            }
          } else {
            tmem_ld_32x32b_x32(lane_base + kColS + ch * 32, s);
            tmem_ld_32x32b_x32(lane_base + kColDP + ch * 32, dp);
            tmem_ld_wait();
          }
          uint32_t pp[16], ds[16];
          const int q0 = ch * 32;
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            const int qa = q0 + 2 * j;
            const float l0 = sLse[qa], l1 = sLse[qa + 1];
            const float d0 = sD[qa], d1 = sD[qa + 1];
            const float p0 = ex2_approx(fmaf(__uint_as_float(s[2 * j]), c, -l0));
            const float p1 = ex2_approx(fmaf(__uint_as_float(s[2 * j + 1]), c, -l1));
            const float g0 = __uint_as_float(dp[2 * j]), g1 = __uint_as_float(dp[2 * j + 1]);
            float pd0 = p0, pd1 = p1, gs0 = p.scale, gs1 = p.scale;
            if (dropping) {
              const uint32_t i0 = (drop_item + static_cast<uint32_t>(qa)) * static_cast<uint32_t>(p.Nk16) +
                                  static_cast<uint32_t>(key);
              const bool k0 = drop_keep(i0, p.drop.key, p.drop.thresh);
              const bool k1 = drop_keep(i0 + static_cast<uint32_t>(p.Nk16), p.drop.key, p.drop.thresh);
              pd0 = k0 ? p0 * p.drop.scale : 0.f;
              pd1 = k1 ? p1 * p.drop.scale : 0.f;
              gs0 = k0 ? p.drop.scale * p.scale : 0.f;
              gs1 = k1 ? p.drop.scale * p.scale : 0.f;
            }
            // dS = P (drop(dP) - D) scale; the dV product uses the dropped probabilities
            pp[j] = pack_bf16x2(pd0, pd1);
            ds[j] = pack_bf16x2(p0 * fmaf(g0, gs0, d0), p1 * fmaf(g1, gs1, d1));
          }
          if (!key_ok) {
#pragma unroll
            for (int j = 0; j < 16; ++j) {
              pp[j] = 0u;
              ds[j] = 0u;
            }
          }
          if (half_chunk) {
            uint32_t a8[8], b8[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              a8[j] = pp[j];
              b8[j] = ds[j];
            }
            tmem_st_32x32b_x8(lane_base + kColS + ch * 32, a8);
            tmem_st_32x32b_x8(lane_base + kColDP + ch * 32, b8);
          } else {
            tmem_st_32x32b_x16(lane_base + kColS + ch * 32, pp);
            tmem_st_32x32b_x16(lane_base + kColDP + ch * 32, ds);
          }
          // dS^T row -> smem tile kt: chunk of 64 queries (ch / 2), 16-byte pieces (ch & 1) * 4 + j
          const uint32_t rowa = sdS + static_cast<uint32_t>(kt) * kDsTile +
                                static_cast<uint32_t>(ch >> 1) * kBox +
                                static_cast<uint32_t>(row_in_tile) * 128u;
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const int piece = (ch & 1) * 4 + j;
            st_shared_v4(rowa + (static_cast<uint32_t>(piece ^ (row_in_tile & 7)) << 4),
                         ds[4 * j], ds[4 * j + 1], ds[4 * j + 2], ds[4 * j + 3]);
          }
        }
        tmem_st_wait();
        fence_proxy_async_smem();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(bar(5));
        // ---- dK_kt (warps 4-7) / dV_kt (warps 8-11) complete: store rows of valid keys
        mbar_wait(bar(6), tc & 1);
        tc_fence_after();
        if (kt * 128 + q4 * 32 < p.Nkeys) {
          const long long ro = b * p.dkv_img + static_cast<long long>(key) * p.lddkv + h * hd;
          if (hf == 0) store_rows(kColDK, 0, 1, p.dk + ro, key_ok, p.vw_kv);
          else store_rows(kColDV, 0, 1, p.dv + ro, key_ok, p.vw_kv);
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(bar(7));
      }
      // ---- dQ: even 16-column chunks from warps 4-7, odd ones from warps 8-11
      mbar_wait(bar(8), it & 1);
      tc_fence_after();
      if (q4 * 32 < p.Nq) {
        __nv_bfloat16* dst = p.dq + b * p.dq_img + static_cast<long long>(row_in_tile) * p.lddq + h * hd;
        store_rows(kColDQ, hf, 2, dst, row_in_tile < p.Nq, p.vw_q);
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        mbar_arrive(bar(9));
        mbar_arrive(bar(11));
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

size_t xr_bwd_smem(int hd, int Nk) {
  const size_t nb = (xr::pad16(hd) + 63) / 64, n_kt = (Nk + 127) / 128;
  return (3 + n_kt) * nb * kBox + n_kt * kDsTile + 1024 + 256 + 1024;
}

template <int HDP>
int launch_xr_bwd(const CUtensorMap& tq, const CUtensorMap& tdo, const CUtensorMap& tk,
                  const CUtensorMap& tv, const XrBwdParams& prm, size_t smem, cudaStream_t stream) {
  VITK_TRY(opt_in_smem<attn_xr_bwd_kernel<HDP>>(232448, "attn_xr_bwd_kernel"));
  const int grid = persistent_grid(static_cast<long long>(prm.B) * prm.H);
  attn_xr_bwd_kernel<HDP><<<grid, kThreads, smem, stream>>>(tq, tdo, tk, tv, prm);
  VITK_CHECK_LAUNCH("attn_xr_bwd_kernel");
  return VITK_OK;
}

bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

}  // namespace

int attention_xr_bwd(const AttnXSrc& s, const void* ctx, const void* dctx, long long ctx_img,
                     int ldc, const float* lse, void* dq, long long dq_img, int lddq, void* dk,
                     void* dv, long long dkv_img, int lddkv, int B, int Nq, int Nk, int H, int hd,
                     cudaStream_t stream, const DropParams* drop) {
  VITK_REQUIRE(s.q && s.k && s.v && ctx && dctx && lse && dq && dk && dv,
               "attention_bwd(xr): null operand");
  VITK_REQUIRE(B > 0 && H > 0 && attention_src_supported(Nq, Nk, hd),
               "attention_bwd(xr): needs head_dim 16..128, <= 128 queries and <= 256 keys (got %d x "
               "%d, head_dim %d)", Nq, Nk, hd);
  VITK_REQUIRE(device_cc() >= 100, "attention_bwd(xr): needs an sm_100 device");
  long long q_img = s.q_img, kv_img = s.kv_img, c_img = ctx_img;
  if (B == 1) {  // a single image has no batch stride: any positive pitch describes it
    if (q_img <= 0) q_img = static_cast<long long>(Nq) * s.ldq;
    if (kv_img <= 0) kv_img = static_cast<long long>(Nk) * s.ldkv;
    if (c_img <= 0) c_img = static_cast<long long>(Nq) * ldc;
  }
  // TMA operands (q, k, v, d_ctx): 16-byte aligned bases, pitches and image strides
  VITK_REQUIRE(aligned16(s.q) && aligned16(s.k) && aligned16(s.v) && aligned16(dctx) &&
                   s.ldq % 8 == 0 && s.ldkv % 8 == 0 && ldc % 8 == 0 && q_img % 8 == 0 &&
                   kv_img % 8 == 0 && c_img % 8 == 0 && q_img > 0 && kv_img > 0 && c_img > 0,
               "attention_bwd(xr): q / k / v / d_ctx need 16-byte aligned bases and pitches "
               "(multiples of 8 elements)");
  VITK_REQUIRE((reinterpret_cast<uintptr_t>(ctx) & 1) == 0 && (reinterpret_cast<uintptr_t>(dq) & 1) == 0 &&
                   (reinterpret_cast<uintptr_t>(dk) & 1) == 0 && (reinterpret_cast<uintptr_t>(dv) & 1) == 0,
               "attention_bwd(xr): misaligned operand");
  VITK_REQUIRE(drop == nullptr || drop->thresh == 0u ||
                   static_cast<long long>(B) * H * Nq * xr::pad16(Nk) < (1ll << 32),
               "attention dropout: batch * heads * queries * keys must stay below 2^32");
  const size_t smem = xr_bwd_smem(hd, Nk);
  VITK_REQUIRE(smem <= 232448, "attention_bwd(xr): shared memory budget exceeded");
  XrBwdParams prm;
  prm.ctx = static_cast<const __nv_bfloat16*>(ctx);
  prm.dctx = static_cast<const __nv_bfloat16*>(dctx);
  prm.dq = static_cast<__nv_bfloat16*>(dq);
  prm.dk = static_cast<__nv_bfloat16*>(dk);
  prm.dv = static_cast<__nv_bfloat16*>(dv);
  prm.lse = lse;
  prm.ctx_img = B == 1 ? 0 : ctx_img;
  prm.dq_img = B == 1 ? 0 : dq_img;
  prm.dkv_img = B == 1 ? 0 : dkv_img;
  prm.ldc = ldc;
  prm.lddq = lddq;
  prm.lddkv = lddkv;
  prm.B = B;
  prm.H = H;
  prm.Nq = Nq;
  prm.Nq16 = xr::pad16(Nq);
  prm.Nkeys = Nk;
  prm.Nk16 = xr::pad16(Nk);
  prm.n_kt = (Nk + 127) / 128;
  prm.hd = hd;
  prm.vw_q = xr::store_width(dq, dq_img, lddq, hd, B);
  const int vk = xr::store_width(dk, dkv_img, lddkv, hd, B), vv = xr::store_width(dv, dkv_img, lddkv, hd, B);
  prm.vw_kv = vk < vv ? vk : vv;
  prm.scale = 1.0f / sqrtf(static_cast<float>(hd));
  if (drop != nullptr) prm.drop = *drop;
  prm.q = static_cast<const __nv_bfloat16*>(s.q);
  prm.k = static_cast<const __nv_bfloat16*>(s.k);
  prm.v = static_cast<const __nv_bfloat16*>(s.v);
  prm.q_img = B == 1 ? 0 : q_img;
  prm.kv_img = B == 1 ? 0 : kv_img;
  prm.ldq = s.ldq;
  prm.ldkv = s.ldkv;
  prm.tma = hd % 8 == 0;
  const int D = H * hd;
  CUtensorMap tq, tdo, tk, tv;
  VITK_TRY(make_row_map(&tq, s.q, B, Nq, D, s.ldq, 128, q_img));
  VITK_TRY(make_row_map(&tdo, dctx, B, Nq, D, ldc, 128, c_img));
  VITK_TRY(make_row_map(&tk, s.k, B, Nk, D, s.ldkv, 128, kv_img));
  VITK_TRY(make_row_map(&tv, s.v, B, Nk, D, s.ldkv, 128, kv_img));
  ProfileScope prof(PROF_ATTN, attention_flops(B, H, Nq, Nk, hd, true), stream);
  switch (xr::pad16(hd)) {
    case 16: return launch_xr_bwd<16>(tq, tdo, tk, tv, prm, smem, stream);
    case 32: return launch_xr_bwd<32>(tq, tdo, tk, tv, prm, smem, stream);
    case 48: return launch_xr_bwd<48>(tq, tdo, tk, tv, prm, smem, stream);
    case 64: return launch_xr_bwd<64>(tq, tdo, tk, tv, prm, smem, stream);
    case 80: return launch_xr_bwd<80>(tq, tdo, tk, tv, prm, smem, stream);
    case 96: return launch_xr_bwd<96>(tq, tdo, tk, tv, prm, smem, stream);
    case 112: return launch_xr_bwd<112>(tq, tdo, tk, tv, prm, smem, stream);
    default: return launch_xr_bwd<128>(tq, tdo, tk, tv, prm, smem, stream);
  }
}

}  // namespace vitk
