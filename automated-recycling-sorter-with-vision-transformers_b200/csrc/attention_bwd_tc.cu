// tcgen05 backward of the attention core for N <= 256 tokens, head_dim 64 (autograd of
// train.py:543-549).  One (image, head) per work item, persistent CTAs, all five contractions on the
// 5th-gen tensor cores with accumulators in TMEM:
//
//   for key tile kt (128 keys) / query tile qt (128 queries):
//     S^T  = K_kt Q_qt^T           A,B from smem (K-major)              -> TMEM [128 x 128]
//     dP^T = V_kt dO_qt^T          A,B from smem (K-major)              -> TMEM [128 x 128]
//     warps 4-11 (thread = key row x half of the query chunks): P^T = exp2(S^T c - lse_q),
//           dS^T = P^T (dP^T - D_q) scale; P^T, dS^T -> TMEM (bf16, in place at the start of each
//           32-column chunk of S^T / dP^T); dS^T also -> smem
//     dV_kt += P^T  dO_qt          A from TMEM, B = dO from smem (MN-major)
//     dK_kt += dS^T Q_qt           A from TMEM, B = Q  from smem (MN-major)
//     dQ_qt += dS   K_kt           A = dS^T tile in smem read as an MN-major operand, B = K (MN-major)
//
// TMEM map (512 columns): S^T/P^T [0,128) | dP^T/dS^T [128,256) | dV [256,320) | dK [320,384) |
// dQ_0 [384,448) | dQ_1 [448,512).  q, k, v, d_ctx arrive by 3-D TMA from the packed activations
// (rows >= N zero-filled); d_qkv leaves through TMA stores whose 3-D map clips rows >= N.
#include <cuda_bf16.h>

#include "attention_kernels.cuh"
#include "common.h"
#include "dropout.cuh"
#include "ptx.cuh"

namespace vitk {
using namespace ptx;

namespace {

// warp 0 TMA, 1 MMA, 2 TMEM alloc, 2-3 per-row vectors of the next item, 4-11 softmax-backward /
// epilogue (warps 4-7 own the first half of a block's query chunks, warps 8-11 the second half)
constexpr int kThreads = 12 * 32;
constexpr uint32_t kColS = 0, kColDP = 128, kColDV = 256, kColDK = 320, kColDQ = 384;

// DROP: attention-probability dropout compiled in (a separate instantiation, so that the p = 0
// kernel carries neither the extra registers nor the per-element branch).
template <bool DROP>
__global__ void __launch_bounds__(kThreads, 1)
attn_bwd_tc_kernel(const __grid_constant__ CUtensorMap tm_qkv,   // box {64, Nk, 1} over qkv
                   const __grid_constant__ CUtensorMap tm_do,    // box {64, Nk, 1} over d_ctx
                   const __grid_constant__ CUtensorMap tm_out,   // box {64, 32, 1} over d_qkv
                   const BwdParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = smem_u32(smem_raw);
  const uint32_t base = (raw_addr + 1023u) & ~1023u;
  uint8_t* smem = smem_raw + (base - raw_addr);

  const int Nk = p.Nk, N = p.N;
  const uint32_t tile_bytes = static_cast<uint32_t>(Nk) * 128u;
  const uint32_t sQ = base, sK = sQ + tile_bytes, sV = sK + tile_bytes, sdO = sV + tile_bytes;
  const uint32_t sdS = sdO + tile_bytes;        // 2 chunks x [128 keys x 128 B]
  const uint32_t sStage = sdS + 32768u;         // 8 warps x 4 KB
  const uint32_t vec_off = 4u * tile_bytes + 32768u + 32768u;
  // two item parities x { lse_q * log2(e) [256], -scale * D_q [256] with D_q = rowsum(d_ctx * ctx) }
  float* sVec = reinterpret_cast<float*>(smem + vec_off);
  const uint32_t bar_base = base + vec_off + 4096u;
  auto bar = [&](int i) { return bar_base + 8u * i; };
  // 0 ld_full, 1 ld_free, 2 s_full, 3 sm_done, 4 ds_free, 5 dkv_full, 6 dkv_free, 7 dq_full,
  // 8 dq_free, 9-10 vec_full[2], 11-12 vec_free[2]
  volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(smem + vec_off + 4096 + 120);
  // column sums of everything this CTA stores (bf16-rounded values, as a pass over d_qkv would see
  // them): the qkv bias gradient without re-reading d_qkv.  One global atomic per column at the end.
  float* colacc = reinterpret_cast<float*>(smem + vec_off + 4096 + 256);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int num_items = p.B * p.H;
  const int D = p.H * 64;
  const int n_kt = (Nk + 127) / 128;  // key tiles == query tiles

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tm_qkv);
    prefetch_tmap(&tm_do);
    prefetch_tmap(&tm_out);
  }
  if (warp == 1 && lane == 0) {
    mbar_init(bar(0), 1);
    mbar_init(bar(1), 1);
    mbar_init(bar(2), 1);
    mbar_init(bar(3), 8);
    mbar_init(bar(4), 1);
    mbar_init(bar(5), 1);
    mbar_init(bar(6), 8);
    mbar_init(bar(7), 1);
    mbar_init(bar(8), 8);
    mbar_init(bar(9), 2);
    mbar_init(bar(10), 2);
    mbar_init(bar(11), 8);
    mbar_init(bar(12), 8);
    fence_mbar_init();
  }
  if (warp == 2) {
    tmem_alloc(smem_u32(const_cast<uint32_t*>(tmem_slot)), 512);
    tmem_relinquish();
  }
  if (p.dbias != nullptr)
    for (int i = threadIdx.x; i < 3 * p.H * 64; i += kThreads) colacc[i] = 0.f;
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  auto rows_in_tile = [&](int t) { return min(128, Nk - t * 128); };  // multiple of 16

  if (warp == 0) {
    // ======================= TMA producer =======================
    if (lane == 0) {
      int it = 0;
      for (int item = blockIdx.x; item < num_items; item += gridDim.x, ++it) {
        const int b = item / p.H, h = item - b * p.H;
        mbar_wait(bar(1), (it & 1) ^ 1u);  // every MMA of the previous item has retired
        mbar_arrive_expect_tx(bar(0), 4u * tile_bytes);
        tma_load_3d(sQ, &tm_qkv, bar(0), h * 64, 0, b);
        tma_load_3d(sK, &tm_qkv, bar(0), D + h * 64, 0, b);
        tma_load_3d(sV, &tm_qkv, bar(0), 2 * D + h * 64, 0, b);
        tma_load_3d(sdO, &tm_do, bar(0), h * 64, 0, b);
      }
    }
  } else if (warp == 1) {
    // ============ MMA issuer (whole warp converged, one elected lane issues) ============
    {
      const uint32_t idesc_mn64 = make_idesc_bf16(128, 64, 0, 1);  // A K-major/TMEM, B MN-major
      const uint32_t idesc_dq = make_idesc_bf16(128, 64, 1, 1);    // A and B MN-major
      int it = 0;
      uint32_t blk = 0;   // running (kt, qt) block counter -> phases of s_full / sm_done / ds_free
      uint32_t ktc = 0;   // running key-tile counter      -> phases of dkv_full / dkv_free
      for (int item = blockIdx.x; item < num_items; item += gridDim.x, ++it) {
        mbar_wait(bar(0), it & 1);
        tc_fence_after();
        mbar_wait(bar(8), (it & 1) ^ 1u);  // dQ accumulators of the previous item have been read
        tc_fence_after();
        for (int kt = 0; kt < n_kt; ++kt) {
          const int kcount = rows_in_tile(kt);
          mbar_wait(bar(6), (ktc & 1) ^ 1u);  // dV / dK accumulators of the previous key tile read
          tc_fence_after();
          for (int qt = 0; qt < n_kt; ++qt, ++blk) {
            const int nq = rows_in_tile(qt);
            const uint32_t idesc_s = make_idesc_bf16(128, nq);
            // ---- S^T = K Q^T and dP^T = V dO^T (both 128 x nq, K = 64)
            const uint64_t ak = make_desc_sw128(sK + kt * 16384u, 16, 1024);
            const uint64_t av = make_desc_sw128(sV + kt * 16384u, 16, 1024);
            const uint64_t bq = make_desc_sw128(sQ + qt * 16384u, 16, 1024);
            const uint64_t bdo = make_desc_sw128(sdO + qt * 16384u, 16, 1024);
            if (elect_one_sync()) {
#pragma unroll
              for (int k = 0; k < 4; ++k)
                mma_bf16_ss(tmem_base + kColS, ak + 2u * k, bq + 2u * k, idesc_s, k > 0);
#pragma unroll
              for (int k = 0; k < 4; ++k)
                mma_bf16_ss(tmem_base + kColDP, av + 2u * k, bdo + 2u * k, idesc_s, k > 0);
              mma_commit(bar(2));
            }
            __syncwarp();
            // ---- wait for P^T / dS^T (TMEM) and dS^T (smem)
            mbar_wait(bar(3), blk & 1);
            tc_fence_after();
            // dV_kt += P^T dO_qt ; dK_kt += dS^T Q_qt      (K = nq queries, 16 per MMA)
            const uint64_t b_do_mn = make_desc_sw128(sdO + qt * 16384u, tile_bytes, 1024);
            const uint64_t b_q_mn = make_desc_sw128(sQ + qt * 16384u, tile_bytes, 1024);
            // dQ_qt += dS K_kt : A = dS^T smem tile as MN-major (2 x 64-query chunks, 16 KB apart),
            // B = K rows of this key tile (MN-major); K = kcount keys
            const uint64_t a_ds = make_desc_sw128(sdS, 16384, 1024);
            const uint64_t b_k_mn = make_desc_sw128(sK + kt * 16384u, tile_bytes, 1024);
            if (elect_one_sync()) {
              // fully unrolled, predicated MMA issue (two instructions per MMA instead of a rolled
              // loop's eight: the issuing warp competes with busy warps for issue slots)
#pragma unroll
              for (int ks = 0; ks < 8; ++ks) {
                if (ks < nq / 16) {
                  // 16 queries per step: bf16 pairs at the start of their 32-column chunk
                  const uint32_t acol = static_cast<uint32_t>((ks >> 1) * 32 + (ks & 1) * 8);
                  mma_bf16_ts(tmem_base + kColDV, tmem_base + kColS + acol,
                              b_do_mn + static_cast<uint64_t>(ks) * 128u, idesc_mn64,
                              (qt > 0 || ks > 0) ? 1u : 0u);
                  mma_bf16_ts(tmem_base + kColDK, tmem_base + kColDP + acol,
                              b_q_mn + static_cast<uint64_t>(ks) * 128u, idesc_mn64,
                              (qt > 0 || ks > 0) ? 1u : 0u);
                }
              }
#pragma unroll
              for (int ks = 0; ks < 8; ++ks)
                if (ks < kcount / 16)
                  mma_bf16_ss(tmem_base + kColDQ + qt * 64, a_ds + static_cast<uint64_t>(ks) * 128u,
                              b_k_mn + static_cast<uint64_t>(ks) * 128u, idesc_dq,
                              (kt > 0 || ks > 0) ? 1u : 0u);
              mma_commit(bar(4));  // dS^T smem tile (and P^T / dS^T in TMEM) consumed
              if (qt == n_kt - 1) mma_commit(bar(5));  // dV_kt, dK_kt complete
              if (qt == n_kt - 1 && kt == n_kt - 1) {
                mma_commit(bar(7));  // dQ complete
                mma_commit(bar(1));  // operands of this item no longer needed
              }
            }
            __syncwarp();
          }
          ++ktc;
        }
      }
    }
  } else if (warp == 2 || warp == 3) {
    // ============ per-row vectors, one item ahead: D_q = rowsum(d_ctx * ctx), lse_q * log2(e) ====
    int it = 0;
    for (int item = blockIdx.x; item < num_items; item += gridDim.x, ++it) {
      const int b = item / p.H, h = item - b * p.H;
      float* vLse = sVec + (it & 1) * 512;
      float* vD = vLse + 256;
      mbar_wait(bar(11 + (it & 1)), ((it >> 1) & 1) ^ 1u);
      const __nv_bfloat16* obase = p.ctx + static_cast<long long>(b) * N * D + h * 64;
      const __nv_bfloat16* dobase = p.dctx + static_cast<long long>(b) * N * D + h * 64;
      for (int r = (warp - 2) * 32 + lane; r < 256; r += 64) {
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
          l2 = p.lse[(static_cast<long long>(b) * p.H + h) * N + r] * kLog2e;
        }
        vLse[r] = l2;
        vD[r] = -dsum * p.scale;
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(bar(9 + (it & 1)));
    }
  } else if (warp >= 4) {
    // ======================= softmax backward + output (thread == key row / output row) =========
    const int q4 = warp & 3;
    const int hf = (warp - 4) >> 2;  // which half of the query chunks / which accumulator to store
    const int row_in_tile = q4 * 32 + lane;
    const float c = p.scale * kLog2e;
    const uint32_t lane_base = tmem_base + (static_cast<uint32_t>(q4 * 32) << 16);
    const uint32_t slab = sStage + static_cast<uint32_t>(warp - 4) * 4096u;
    int it = 0;
    uint32_t blk = 0, ktc = 0;

    // out[32 rows x 64] (TMEM cols col0..col0+63 of this warp's lanes) -> bf16 -> TMA store
    auto store_acc = [&](uint32_t col0, int gcol, int row0, int b) {
      uint32_t o0[32], o1[32];
      tmem_ld_32x32b_x32(lane_base + col0, o0);
      tmem_ld_32x32b_x32(lane_base + col0 + 32, o1);
      tmem_ld_wait();
      uint32_t pk[32];
#pragma unroll
      for (int j = 0; j < 16; ++j) {
        pk[j] = pack_bf16x2(__uint_as_float(o0[2 * j]), __uint_as_float(o0[2 * j + 1]));
        pk[16 + j] = pack_bf16x2(__uint_as_float(o1[2 * j]), __uint_as_float(o1[2 * j + 1]));
      }
      if (lane == 0) tma_store_wait_read<0>();
      __syncwarp();
      const uint32_t rowa = slab + static_cast<uint32_t>(lane) * 128u;
#pragma unroll
      for (int j = 0; j < 8; ++j)
        st_shared_v4(rowa + (static_cast<uint32_t>(j ^ (lane & 7)) << 4), pk[4 * j], pk[4 * j + 1],
                     pk[4 * j + 2], pk[4 * j + 3]);
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) {
        tma_store_3d(&tm_out, slab, gcol, row0, b);
        tma_store_commit();
      }
      if (p.dbias != nullptr) {
        // lane sums columns 2*lane, 2*lane+1 over the 32 staged rows (rows >= N are exact zeros)
        float s0 = 0.f, s1 = 0.f;
#pragma unroll 8
        for (int r = 0; r < 32; ++r) {
          uint32_t w;
          const uint32_t a = slab + static_cast<uint32_t>(r) * 128u +
                             ((static_cast<uint32_t>(lane >> 2) ^ static_cast<uint32_t>(r & 7)) << 4) +
                             static_cast<uint32_t>(lane & 3) * 4u;
          asm volatile("ld.shared.b32 %0, [%1];" : "=r"(w) : "r"(a));
          s0 += bf16lo_to_f32(w);
          s1 += bf16hi_to_f32(w);
        }
        atomicAdd(&colacc[gcol + 2 * lane], s0);
        atomicAdd(&colacc[gcol + 2 * lane + 1], s1);
      }
    };

    for (int item = blockIdx.x; item < num_items; item += gridDim.x, ++it) {
      const int b = item / p.H, h = item - b * p.H;
      // ---- per-row vectors of this item (written by warps 2-3 one item ahead)
      const float* sLse = sVec + (it & 1) * 512;
      const float* sD = sLse + 256;
      mbar_wait(bar(9 + (it & 1)), (it >> 1) & 1);

      for (int kt = 0; kt < n_kt; ++kt) {
        const int key = kt * 128 + row_in_tile;
        const bool key_ok = key < N;
        const uint32_t drop_item_rows = static_cast<uint32_t>(item) * static_cast<uint32_t>(N);
        for (int qt = 0; qt < n_kt; ++qt, ++blk) {
          const int nq = rows_in_tile(qt);
          mbar_wait(bar(2), blk & 1);
          tc_fence_after();
          if (blk > 0) mbar_wait(bar(4), (blk - 1) & 1);  // previous dS^T smem tile consumed
          const int nch = nq / 32 + ((nq & 31) ? 1 : 0);
          const int ch_mid = (nch + 1) >> 1;
          for (int ch = hf == 0 ? 0 : ch_mid; ch < (hf == 0 ? ch_mid : nch); ++ch) {
            // chunks of 32 queries; the last chunk of a ragged tile holds 16
            const bool half_chunk = (ch * 32 + 32 > nq);
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
            const int q0 = qt * 128 + ch * 32;
            // branch-free over the key mask (sixteen predicated regions would serialise the
            // lse load -> exp2 -> product chains of the pairs); rows of missing keys are zeroed after
#pragma unroll
            for (int j = 0; j < 16; ++j) {
              const float2 l2 = *reinterpret_cast<const float2*>(sLse + q0 + 2 * j);
              const float2 dn = *reinterpret_cast<const float2*>(sD + q0 + 2 * j);  // -D_q * scale
              float p0 = ex2_approx(fmaf(__uint_as_float(s[2 * j]), c, -l2.x));
              float p1 = ex2_approx(fmaf(__uint_as_float(s[2 * j + 1]), c, -l2.y));
              const float g0 = __uint_as_float(dp[2 * j]), g1 = __uint_as_float(dp[2 * j + 1]);
              float pd0 = p0, pd1 = p1, gs0 = p.scale, gs1 = p.scale;
              if constexpr (DROP) {
                // The mask's pairs run along the keys and the thread owns one key, so a hash serves
                // the two lanes of a key pair: the even lane hashes query 2j, the odd lane query
                // 2j + 1, and they swap (one hash + one shuffle per two elements instead of two).
                const uint32_t half_nk = static_cast<uint32_t>(Nk >> 1);
                const uint32_t kp = static_cast<uint32_t>(key >> 1);
                const uint32_t hm = drop_bits(
                    (drop_item_rows + q0 + 2 * j + (lane & 1)) * half_nk + kp, p.drop.key);
                const uint32_t ho = __shfl_xor_sync(0xffffffffu, hm, 1);
                const uint32_t b0 = (lane & 1) ? ho : hm;
                const uint32_t b1 = (lane & 1) ? hm : ho;
                // this key's 16 bits moved to the top: keep iff (bits << sh) >= thresh << 16
                const uint32_t sh = (key & 1) ? 0u : 16u;
                const uint32_t t16 = p.drop.thresh << 16;
                const bool k0 = (b0 << sh) >= t16, k1 = (b1 << sh) >= t16;
                pd0 = p0 * (k0 ? p.drop.scale : 0.f);
                pd1 = p1 * (k1 ? p.drop.scale : 0.f);
                gs0 = k0 ? p.drop.scale * p.scale : 0.f;   // dropout mask and scale of dP in one factor
                gs1 = k1 ? p.drop.scale * p.scale : 0.f;
              }
              // dS = P (dP - D) scale; the dV product uses the dropped probabilities
              pp[j] = pack_bf16x2(pd0, pd1);
              ds[j] = pack_bf16x2(p0 * fmaf(g0, gs0, dn.x), p1 * fmaf(g1, gs1, dn.y));
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
            // dS^T row -> smem: chunk of 64 queries (ch / 2), 16-byte pieces (ch & 1) * 4 .. + 3
            const uint32_t rowa = sdS + static_cast<uint32_t>(ch >> 1) * 16384u +
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
          if (lane == 0) mbar_arrive(bar(3));
        }
        // ---- dV_kt / dK_kt are complete: convert and store rows [kt*128 + q4*32, +32)
        mbar_wait(bar(5), ktc & 1);
        tc_fence_after();
        const int row0 = kt * 128 + q4 * 32;
        if (row0 < N) {
          if (hf == 0) store_acc(kColDK, D + h * 64, row0, b);
          else store_acc(kColDV, 2 * D + h * 64, row0, b);
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(bar(6));
        ++ktc;
      }
      // ---- dQ
      mbar_wait(bar(7), it & 1);
      tc_fence_after();
      for (int qt = hf; qt < n_kt; qt += 2) {
        const int row0 = qt * 128 + q4 * 32;
        if (row0 < N) store_acc(kColDQ + qt * 64, h * 64, row0, b);
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        mbar_arrive(bar(8));
        mbar_arrive(bar(11 + (it & 1)));  // this item's row vectors may be overwritten
      }
    }
    if (lane == 0) tma_store_wait<0>();
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
  if (p.dbias != nullptr)
    for (int i = threadIdx.x; i < 3 * p.H * 64; i += kThreads) atomicAdd(p.dbias + i, colacc[i]);
}

}  // namespace

int attention_bwd_tc(const void* qkv, const void* ctx, const void* dctx, const float* lse,
                     void* dqkv, int B, int N, int H, int hd, cudaStream_t stream,
                     const DropParams* drop, float* dbias) {
  VITK_REQUIRE(qkv && ctx && dctx && lse && dqkv, "attention_bwd: null operand");
  VITK_REQUIRE(hd == 64 && N >= 1 && N <= 256, "attention_bwd(tc): needs head_dim 64, N <= 256");
  const int Nk = (N + 15) & ~15;
  const int D = H * 64;
  const size_t smem = 4 * static_cast<size_t>(Nk) * 128 + 32768 + 32768 + 4096 + 256 + 1024 +
                      (dbias != nullptr ? static_cast<size_t>(3) * D * 4 : 0);
  VITK_REQUIRE(smem <= 232448, "attention_bwd(tc): shared memory budget exceeded");
  VITK_TRY(opt_in_smem<attn_bwd_tc_kernel<false>>(232448, "attn_bwd_tc_kernel<false>"));
  VITK_TRY(opt_in_smem<attn_bwd_tc_kernel<true>>(232448, "attn_bwd_tc_kernel<true>"));
  CUtensorMap tq, tdo, tout;
  VITK_TRY(make_row_map(&tq, qkv, B, N, 3 * D, 3 * D, Nk));
  VITK_TRY(make_row_map(&tdo, dctx, B, N, D, D, Nk));
  VITK_TRY(make_row_map(&tout, dqkv, B, N, 3 * D, 3 * D, 32));
  BwdParams prm;
  prm.B = B;
  prm.N = N;
  prm.H = H;
  prm.Nk = Nk;
  prm.scale = 1.0f / sqrtf(static_cast<float>(hd));
  prm.ctx = static_cast<const __nv_bfloat16*>(ctx);
  prm.dctx = static_cast<const __nv_bfloat16*>(dctx);
  prm.lse = lse;
  if (drop != nullptr) prm.drop = *drop;
  prm.dbias = dbias;
  const int grid = persistent_grid(B * H);
  ProfileScope prof(PROF_ATTN, attention_flops(B, H, N, N, hd, true), stream);
  if (prm.drop.thresh != 0u)
    attn_bwd_tc_kernel<true><<<grid, kThreads, smem, stream>>>(tq, tdo, tout, prm);
  else
    attn_bwd_tc_kernel<false><<<grid, kThreads, smem, stream>>>(tq, tdo, tout, prm);
  VITK_CHECK_LAUNCH("attn_bwd_tc_kernel");
  return VITK_OK;
}

}  // namespace vitk
