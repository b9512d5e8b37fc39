// tcgen05 backward of the attention core for N <= 224 tokens, head_dim 64 (autograd of
// train.py:543-549), software-pipelined: the same five contractions and TMEM-resident accumulators
// as attention_bwd_tc.cu, but walked in sub-blocks of 128 keys x 64 queries with the score tiles
// double-buffered in TMEM, so that the MMAs of sub-block s+1 (S^T, dP^T) and of sub-block s-1
// (dV, dK, dQ) run under the softmax-backward arithmetic of sub-block s instead of alternating
// with it.
//
//   for key tile kt (128 keys) / query sub-tile q64 (64 queries), buffer b = running count & 1:
//     S^T_b  = K_kt Q_q64^T         A,B from smem (K-major)             -> TMEM [128 x 64]
//     dP^T_b = V_kt dO_q64^T        A,B from smem (K-major)             -> TMEM [128 x 64]
//     warps 4-11 (thread = key row; warps 4-7 the first 32 queries, 8-11 the second 32):
//           P^T = exp2(S^T c - lse_q), dS^T = P^T (dP^T - D_q) scale; P^T, dS^T -> TMEM (bf16, in
//           place at the start of their 32-column chunk); dS^T also -> smem (one of 4 chunks)
//     dV_kt += P^T  dO_q64          A from TMEM, B = dO from smem (MN-major)
//     dK_kt += dS^T Q_q64           A from TMEM, B = Q  from smem (MN-major)
//     every second sub-tile (a 128-query tile complete):
//     dQ_qt += dS   K_kt            A = the pair of dS^T chunks read MN-major, B = K (MN-major)
//
// Around that: finished accumulators are stored one sub-block late (their MMAs have retired by
// then) and handed back as soon as they sit in registers; the operand tiles are loaded and released
// in three groups, so that the next item's first tiles arrive during this item's second key tile.
//
// TMEM map (512 columns): buffer 0 { S^T [0,64) | dP^T [64,128) } | buffer 1 { [128,192) |
// [192,256) } | dV [256,320) | dK [320,384) | dQ_0 [384,448) | dQ_1 [448,512).  Shared memory: the
// four operand tiles, 4 x 16 KB of dS^T chunks (two query tiles in flight), 8 x 4 KB of store
// staging - which is what limits this kernel to Nk <= 224; attention_bwd_tc.cu covers 225..256.
#include <cuda_bf16.h>

#include "attention_kernels.cuh"
#include "common.h"
#include "dropout.cuh"
#include "ptx.cuh"

namespace vitk {
using namespace ptx;

// Debug aid (build with -DVITK_ATTN_TRACE): SM clocks the first softmax warp and the MMA warp of
// every CTA spend in each phase; tests/trace_attn_bwd.py reads them back.
#ifdef VITK_ATTN_TRACE
__device__ long long g_attn_trace[320][16];
#define AT_BEGIN(v) const long long v = clock64()
#define AT_ADD(acc, v) acc += clock64() - v
#else
#define AT_BEGIN(v) do { } while (0)
#define AT_ADD(acc, v) do { } while (0)
#endif

namespace {

// warp 0 TMA, 1 MMA, 2 TMEM alloc, 2-3 per-row vectors of the next item, 4-11 softmax-backward /
// epilogue (warps 4-7 own the first half of a block's query chunks, warps 8-11 the second half)
constexpr int kThreads = 12 * 32;
constexpr uint32_t kColDPofs = 64, kColDV = 256, kColDK = 320, kColDQ = 384;  // S at buffer * 128

// Per-row vectors of one (image, head): vLse[r] = lse_r * log2(e) (+inf for rows >= N, so that
// P = 2^(-inf) = 0) and vD[r] = -scale * rowsum(d_ctx_r * ctx_r), r < 256.  Called by a group of nw
// warps (w = this warp's index in the group); every warp takes 64 / nw groups of four rows, BATCH
// groups in flight.  Eight lanes per row (16 bytes each): one instruction reads four whole
// 128-byte rows instead of touching 32 different lines; three shuffles reduce.
template <int BATCH>
__device__ __forceinline__ void bwd_row_vectors(const BwdParams& p, int b, int h, float* vLse,
                                                float* vD, int w, int nw, int lane) {
  const int N = p.N, D = p.H * 64;
  const __nv_bfloat16* obase = p.ctx + static_cast<long long>(b) * N * D + h * 64;
  const __nv_bfloat16* dobase = p.dctx + static_cast<long long>(b) * N * D + h * 64;
  const float* lrow = p.lse + (static_cast<long long>(b) * p.H + h) * N;
  for (int r = w * 32 + lane; r < 256; r += nw * 32)
    vLse[r] = r < N ? __ldg(lrow + r) * kLog2e : INFINITY;
  const int seg = lane & 7;
  const int per_warp = 64 / nw;
#pragma unroll 1
  for (int g0 = w * per_warp; g0 < (w + 1) * per_warp; g0 += BATCH) {
    // all loads first (rows >= N re-read row N-1 and are zeroed below, so that no branch separates
    // the loads)
    uint4 a[BATCH], d[BATCH];
#pragma unroll
    for (int u = 0; u < BATCH; ++u) {
      const int r = min((g0 + u) * 4 + (lane >> 3), N - 1);
      a[u] = __ldg(reinterpret_cast<const uint4*>(obase + static_cast<long long>(r) * D) + seg);
      d[u] = __ldg(reinterpret_cast<const uint4*>(dobase + static_cast<long long>(r) * D) + seg);
    }
#pragma unroll
    for (int u = 0; u < BATCH; ++u) {
      const int r = (g0 + u) * 4 + (lane >> 3);
      float dsum = bf16lo_to_f32(a[u].x) * bf16lo_to_f32(d[u].x) + bf16hi_to_f32(a[u].x) * bf16hi_to_f32(d[u].x);
      dsum += bf16lo_to_f32(a[u].y) * bf16lo_to_f32(d[u].y) + bf16hi_to_f32(a[u].y) * bf16hi_to_f32(d[u].y);
      dsum += bf16lo_to_f32(a[u].z) * bf16lo_to_f32(d[u].z) + bf16hi_to_f32(a[u].z) * bf16hi_to_f32(d[u].z);
      dsum += bf16lo_to_f32(a[u].w) * bf16lo_to_f32(d[u].w) + bf16hi_to_f32(a[u].w) * bf16hi_to_f32(d[u].w);
      dsum += __shfl_xor_sync(0xffffffffu, dsum, 1);
      dsum += __shfl_xor_sync(0xffffffffu, dsum, 2);
      dsum += __shfl_xor_sync(0xffffffffu, dsum, 4);
      if (seg == 0) vD[r] = r < N ? -dsum * p.scale : 0.f;
    }
  }
}

// DROP: attention-probability dropout compiled in (a separate instantiation, so that the p = 0
// kernel carries neither the extra registers nor the per-element branch).
template <bool DROP>
__global__ void __launch_bounds__(kThreads, 1)
attn_bwd_tc2_kernel(const __grid_constant__ CUtensorMap tm_qkv,   // box {64, min(Nk, 128), 1} over qkv
                   const __grid_constant__ CUtensorMap tm_do,    // the same box over d_ctx
                   const __grid_constant__ CUtensorMap tm_qkv1,  // box {64, Nk - 128, 1} (Nk > 128)
                   const __grid_constant__ CUtensorMap tm_do1,
                   const __grid_constant__ CUtensorMap tm_out,   // box {64, 32, 1} over d_qkv
                   const BwdParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = smem_u32(smem_raw);
  const uint32_t base = (raw_addr + 1023u) & ~1023u;
  uint8_t* smem = smem_raw + (base - raw_addr);

  const int Nk = p.Nk, N = p.N;
  const uint32_t tile_bytes = static_cast<uint32_t>(Nk) * 128u;
  const uint32_t sQ = base, sK = sQ + tile_bytes, sV = sK + tile_bytes, sdO = sV + tile_bytes;
  const uint32_t sdS = sdO + tile_bytes;        // 4 chunks x [128 keys x 128 B], pairs per query tile
  const uint32_t sStage = sdS + 65536u;         // 8 warps x 4 KB
  const uint32_t vec_off = 4u * tile_bytes + 65536u + 32768u;
  // two item parities x { lse_q * log2(e) [256], -scale * D_q [256] with D_q = rowsum(d_ctx * ctx) }
  float* sVec = reinterpret_cast<float*>(smem + vec_off);
  const uint32_t bar_base = base + vec_off + 4096u;
  auto bar = [&](int i) { return bar_base + 8u * i; };
  // Operand groups, loaded and released separately so that the next item's first tiles arrive while
  // this item is still in its second key tile: A = K, V rows 0-127; B = Q, dO rows 0-127; C = rows
  // 128.. of all four.  0-2 ld_full[A,B,C], 3-5 ld_free[A,B,C], 6-7 s_full[2], 8-9 sm_done[2],
  // 10-11 ds_free[2], 12 dkv_full, 13 dkv_free, 14 dq_full, 15 dq_free, 16-17 vec_full[2], 18-19
  // vec_free[2]
  enum { LD_FULL = 0, LD_FREE = 3, S_FULL = 6, SM_DONE = 8, DS_FREE = 10, DKV_FULL = 12, DKV_FREE,
         DQ_FULL, DQ_FREE, VEC_FULL, VEC_FREE = 18 };
  volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(smem + vec_off + 4096 + 192);
  // column sums of everything this CTA stores (bf16-rounded values, as a pass over d_qkv would see
  // them): the qkv bias gradient without re-reading d_qkv.  One global atomic per column at the end.
  float* colacc = reinterpret_cast<float*>(smem + vec_off + 4096 + 256);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int num_items = p.B * p.H;
  const int D = p.H * 64;
  const int n_kt = (Nk + 127) / 128;  // key tiles == query tiles
  const int n_q64 = (Nk + 63) / 64;   // query sub-tiles

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tm_qkv);
    prefetch_tmap(&tm_do);
    prefetch_tmap(&tm_qkv1);
    prefetch_tmap(&tm_do1);
    prefetch_tmap(&tm_out);
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < 3; ++i) {
      mbar_init(bar(LD_FULL + i), 1);
      mbar_init(bar(LD_FREE + i), 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(bar(S_FULL + i), 1);
      mbar_init(bar(SM_DONE + i), 8);
      mbar_init(bar(DS_FREE + i), 1);
      mbar_init(bar(VEC_FULL + i), 2);
      mbar_init(bar(VEC_FREE + i), 8);
    }
    mbar_init(bar(DKV_FULL), 1);
    mbar_init(bar(DKV_FREE), 8);
    mbar_init(bar(DQ_FULL), 1);
    mbar_init(bar(DQ_FREE), 8);
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
        const uint32_t ph = (it & 1) ^ 1u;
        const uint32_t bytes0 = static_cast<uint32_t>(min(Nk, 128)) * 128u;
        mbar_wait(bar(LD_FREE + 0), ph);  // the previous item's last MMA on K / V rows 0-127 retired
        mbar_arrive_expect_tx(bar(LD_FULL + 0), 2u * bytes0);
        tma_load_3d(sK, &tm_qkv, bar(LD_FULL + 0), D + h * 64, 0, b);
        tma_load_3d(sV, &tm_qkv, bar(LD_FULL + 0), 2 * D + h * 64, 0, b);
        mbar_wait(bar(LD_FREE + 1), ph);  // ... on Q / dO rows 0-127
        mbar_arrive_expect_tx(bar(LD_FULL + 1), 2u * bytes0);
        tma_load_3d(sQ, &tm_qkv, bar(LD_FULL + 1), h * 64, 0, b);
        tma_load_3d(sdO, &tm_do, bar(LD_FULL + 1), h * 64, 0, b);
        if (n_kt > 1) {
          mbar_wait(bar(LD_FREE + 2), ph);  // every MMA of the previous item retired
          mbar_arrive_expect_tx(bar(LD_FULL + 2), 4u * (tile_bytes - 16384u));
          tma_load_3d(sQ + 16384u, &tm_qkv1, bar(LD_FULL + 2), h * 64, 128, b);
          tma_load_3d(sdO + 16384u, &tm_do1, bar(LD_FULL + 2), h * 64, 128, b);
          tma_load_3d(sK + 16384u, &tm_qkv1, bar(LD_FULL + 2), D + h * 64, 128, b);
          tma_load_3d(sV + 16384u, &tm_qkv1, bar(LD_FULL + 2), 2 * D + h * 64, 128, b);
        }
      }
    }
  } else if (warp == 1) {
    // ============ MMA issuer (whole warp converged, one elected lane issues) ============
    {
      const uint32_t idesc_mn64 = make_idesc_bf16(128, 64, 0, 1);  // A K-major/TMEM, B MN-major
      const uint32_t idesc_dq = make_idesc_bf16(128, 64, 1, 1);    // A and B MN-major
      const int n_sb = n_kt * n_q64;
      [[maybe_unused]] long long at_is = 0, at_ia = 0;
      auto cols_in_sub = [&](int q64) { return min(64, Nk - q64 * 64); };  // multiple of 16
      // S^T and dP^T of sub-block (kt, q64) into buffer buf
      auto issue_scores = [&](int kt, int q64, uint32_t buf) {
        AT_BEGIN(at_x);
        const uint32_t idesc_s = make_idesc_bf16(128, cols_in_sub(q64));
        const uint64_t ak = make_desc_sw128(sK + kt * 16384u, 16, 1024);
        const uint64_t av = make_desc_sw128(sV + kt * 16384u, 16, 1024);
        const uint64_t bq = make_desc_sw128(sQ + q64 * 8192u, 16, 1024);
        const uint64_t bdo = make_desc_sw128(sdO + q64 * 8192u, 16, 1024);
        if (elect_one_sync()) {
#pragma unroll
          for (int k = 0; k < 4; ++k)
            mma_bf16_ss(tmem_base + buf * 128u, ak + 2u * k, bq + 2u * k, idesc_s, k > 0);
#pragma unroll
          for (int k = 0; k < 4; ++k)
            mma_bf16_ss(tmem_base + buf * 128u + kColDPofs, av + 2u * k, bdo + 2u * k, idesc_s, k > 0);
          mma_commit(bar(S_FULL + buf));
        }
        __syncwarp();
        AT_ADD(at_is, at_x);
      };
      [[maybe_unused]] long long at_ld = 0, at_sm = 0, at_free = 0;
      AT_BEGIN(at_m0);
      int it = 0;
      uint32_t sbc = 0;   // running sub-block counter  -> buffer, phases of s_full / sm_done
      uint32_t qtc = 0;   // running query-tile counter -> dS^T chunk pair, phase of ds_free
      uint32_t ktc = 0;   // running key-tile counter   -> phases of dkv_full / dkv_free
      for (int item = blockIdx.x; item < num_items; item += gridDim.x, ++it) {
        AT_BEGIN(at_a);
        mbar_wait(bar(LD_FULL + 0), it & 1);
        mbar_wait(bar(LD_FULL + 1), it & 1);
        AT_ADD(at_ld, at_a);
        tc_fence_after();
        issue_scores(0, 0, sbc & 1u);
        int kt = 0, q64 = 0;
        for (int s = 0; s < n_sb; ++s, ++sbc) {
          const uint32_t buf = sbc & 1u;
          const bool last_q = (q64 == n_q64 - 1);
          // The next sub-block's scores go to the other buffer while this one's are being turned
          // into P^T / dS^T (that buffer's previous readers, dV / dK of sub-block s-1, are earlier
          // in the in-order tensor pipe).  Issuing them two sub-blocks ahead instead (after dV / dK
          // of s) measured 1 % slower: the tensor pipe is shared-memory-bound on these small MMAs
          // (48 clocks per 128 x 64 x 16 with both operands in smem), not latency-bound.
          if (s + 1 < n_sb) {
            if (s + 1 == 2 && n_kt > 1) {  // first use of rows 128.. (Q / dO sub-tile 2)
              AT_BEGIN(at_a2);
              mbar_wait(bar(LD_FULL + 2), it & 1);
              AT_ADD(at_ld, at_a2);
              tc_fence_after();
            }
            issue_scores(last_q ? kt + 1 : kt, last_q ? 0 : q64 + 1, buf ^ 1u);
          }
          AT_BEGIN(at_b);
          if (q64 == 0) {
            mbar_wait(bar(DKV_FREE), (ktc & 1) ^ 1u);  // dV / dK of the previous key tile read
            if (s == 0) mbar_wait(bar(DQ_FREE), (it & 1) ^ 1u);  // dQ of the previous item read
          }
          AT_ADD(at_free, at_b);
          AT_BEGIN(at_c);
          mbar_wait(bar(SM_DONE + buf), (sbc >> 1) & 1u);
          AT_ADD(at_sm, at_c);
          tc_fence_after();
          AT_BEGIN(at_y);
          const int nq = cols_in_sub(q64);
          const int kcount = rows_in_tile(kt);
          const int qt = q64 >> 1;
          const bool tile_done = (q64 & 1) || last_q;
          // dV_kt += P^T dO ; dK_kt += dS^T Q   (K = nq queries, 16 per MMA; A = P^T / dS^T in the
          // score buffer: an A operand from shared memory would make these small MMAs
          // shared-memory-bound, 6 KB per 128 x 64 x 16)
          const uint64_t b_do_mn = make_desc_sw128(sdO + q64 * 8192u, tile_bytes, 1024);
          const uint64_t b_q_mn = make_desc_sw128(sQ + q64 * 8192u, tile_bytes, 1024);
          if (elect_one_sync()) {
#pragma unroll
            for (int ks = 0; ks < 4; ++ks) {
              if (ks < nq / 16) {
                // 16 queries per step: bf16 pairs at the start of their 32-column chunk
                const uint32_t acol = buf * 128u + static_cast<uint32_t>((ks >> 1) * 32 + (ks & 1) * 8);
                mma_bf16_ts(tmem_base + kColDV, tmem_base + acol,
                            b_do_mn + static_cast<uint64_t>(ks) * 128u, idesc_mn64,
                            (q64 > 0 || ks > 0) ? 1u : 0u);
                mma_bf16_ts(tmem_base + kColDK, tmem_base + kColDPofs + acol,
                            b_q_mn + static_cast<uint64_t>(ks) * 128u, idesc_mn64,
                            (q64 > 0 || ks > 0) ? 1u : 0u);
              }
            }
          }
          __syncwarp();
          // dQ_qt += dS K_kt : A = the dS^T chunk pair read MN-major (64-query chunks 16 KB apart),
          // B = K rows of this key tile (MN-major); K = kcount keys
          const uint64_t a_ds = make_desc_sw128(sdS + (qtc & 1u) * 32768u, 16384, 1024);
          const uint64_t b_k_mn = make_desc_sw128(sK + kt * 16384u, tile_bytes, 1024);
          if (elect_one_sync()) {
            if (tile_done) {
#pragma unroll
              for (int ks = 0; ks < 8; ++ks)
                if (ks < kcount / 16)
                  mma_bf16_ss(tmem_base + kColDQ + qt * 64, a_ds + static_cast<uint64_t>(ks) * 128u,
                              b_k_mn + static_cast<uint64_t>(ks) * 128u, idesc_dq,
                              (kt > 0 || ks > 0) ? 1u : 0u);
              mma_commit(bar(DS_FREE + (qtc & 1u)));  // this pair of dS^T chunks consumed
            }
            if (last_q) mma_commit(bar(DKV_FULL));  // dV_kt, dK_kt complete
            if (s == n_q64 - 1) mma_commit(bar(LD_FREE + 0));  // K / V rows 0-127: key tile 0 done
            if (s == (n_kt - 1) * n_q64 + min(1, n_q64 - 1))
              mma_commit(bar(LD_FREE + 1));                    // Q / dO rows 0-127: last use
            if (s == n_sb - 1) {
              mma_commit(bar(DQ_FULL));  // dQ complete
              if (n_kt > 1) mma_commit(bar(LD_FREE + 2));
            }
          }
          __syncwarp();
          AT_ADD(at_ia, at_y);
          if (tile_done) ++qtc;
          if (last_q) {
            ++ktc;
            ++kt;
            q64 = 0;
          } else {
            ++q64;
          }
        }
      }
#ifdef VITK_ATTN_TRACE
      if (lane == 0 && blockIdx.x < 160) {
        g_attn_trace[blockIdx.x][0] = clock64() - at_m0;
        g_attn_trace[blockIdx.x][1] = at_ld;
        g_attn_trace[blockIdx.x][2] = at_sm;
        g_attn_trace[blockIdx.x][3] = at_free;
        g_attn_trace[blockIdx.x + 160][0] = at_is;
        g_attn_trace[blockIdx.x + 160][1] = at_ia;
      }
#endif
    }
  } else if (warp == 2 || warp == 3) {
    // ============ per-row vectors, one item ahead (the first item's are computed by the softmax
    // warps themselves, which have nothing else to do while the first tiles load) ============
    int it = 1;
    [[maybe_unused]] long long at_vwait = 0;
    AT_BEGIN(at_v0);
    for (int item = blockIdx.x + gridDim.x; item < num_items; item += gridDim.x, ++it) {
      const int b = item / p.H, h = item - b * p.H;
      float* vLse = sVec + (it & 1) * 512;
      AT_BEGIN(at_v);
      mbar_wait(bar(VEC_FREE + (it & 1)), ((it >> 1) & 1) ^ 1u);
      AT_ADD(at_vwait, at_v);
      bwd_row_vectors<16>(p, b, h, vLse, vLse + 256, warp - 2, 2, lane);
      __syncwarp();
      if (lane == 0) mbar_arrive(bar(VEC_FULL + (it & 1)));
    }
#ifdef VITK_ATTN_TRACE
    if (lane == 0 && warp == 2 && blockIdx.x < 160) {
      g_attn_trace[blockIdx.x][15] = clock64() - at_v0 - at_vwait;  // busy time of a vector warp
    }
#endif
  } else if (warp >= 4) {
    // ======================= softmax backward + output (thread == key row / output row) =========
    const int q4 = warp & 3;
    const int hf = (warp - 4) >> 2;  // which 32 queries of a sub-block / which accumulator to store
    const int row_in_tile = q4 * 32 + lane;
    const float c = p.scale * kLog2e;
    const uint32_t lane_base = tmem_base + (static_cast<uint32_t>(q4 * 32) << 16);
    const uint32_t slab = sStage + static_cast<uint32_t>(warp - 4) * 4096u;
    int it = 0;
    uint32_t sbc = 0, qtc = 0, ktc = 0;  // as in the MMA warp
    [[maybe_unused]] long long at_vec = 0, at_dsf = 0, at_sf = 0, at_tld = 0, at_math = 0, at_st = 0,
                               at_wkv = 0, at_skv = 0, at_wq = 0, at_sq = 0;
    AT_BEGIN(at_s0);

    // out[32 rows x 64] (TMEM cols col0..col0+63 of this warp's lanes) -> bf16 -> TMA store
    // release(): hands the accumulator back to the MMA warp as soon as it sits in registers - the
    // conversion, the staging and the bias-gradient sums are off the MMA warp's critical path
    auto store_acc = [&](uint32_t col0, int gcol, int row0, int b, auto&& release) {
      uint32_t o0[32], o1[32];
      tmem_ld_32x32b_x32(lane_base + col0, o0);
      tmem_ld_32x32b_x32(lane_base + col0 + 32, o1);
      tmem_ld_wait();
      release();
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

    // Stores of finished accumulators, deferred by one sub-block: dK / dV of a key tile after the
    // first sub-block of the next key tile (or item), dQ after the first sub-block of the next item.
    bool pend_kv = false, pend_q = false;
    int pend_kt = 0, pend_b = 0, pend_h = 0, pend_it = 0;
    uint32_t pend_ktc = 0;
    auto flush_stores = [&]() {
      if (pend_kv) {
        AT_BEGIN(at_f);
        mbar_wait(bar(DKV_FULL), pend_ktc & 1);
        AT_ADD(at_wkv, at_f);
        AT_BEGIN(at_g);
        tc_fence_after();
        const int row0 = pend_kt * 128 + q4 * 32;
        auto release = [&]() {
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(bar(DKV_FREE));
        };
        if (row0 >= N) release();
        else if (hf == 0) store_acc(kColDK, D + pend_h * 64, row0, pend_b, release);
        else store_acc(kColDV, 2 * D + pend_h * 64, row0, pend_b, release);
        AT_ADD(at_skv, at_g);
        pend_kv = false;
      }
      if (pend_q) {
        AT_BEGIN(at_h);
        mbar_wait(bar(DQ_FULL), pend_it & 1);
        AT_ADD(at_wq, at_h);
        AT_BEGIN(at_i);
        tc_fence_after();
        // at most two query tiles (N <= 256): warps 4-7 own tile 0, warps 8-11 tile 1
        const int row0 = hf * 128 + q4 * 32;
        auto release = [&]() {
          tc_fence_before();
          __syncwarp();
          if (lane == 0) {
            mbar_arrive(bar(DQ_FREE));
            mbar_arrive(bar(VEC_FREE + (pend_it & 1)));  // that item's row vectors may be overwritten
          }
        };
        if (hf < n_kt && row0 < N) store_acc(kColDQ + hf * 64, pend_h * 64, row0, pend_b, release);
        else release();
        AT_ADD(at_sq, at_i);
        pend_q = false;
      }
    };

    // the first item's row vectors: all eight warps, while the first tiles are on their way
    if (static_cast<int>(blockIdx.x) < num_items) {
      const int b0 = blockIdx.x / p.H, h0 = blockIdx.x - b0 * p.H;
      bwd_row_vectors<8>(p, b0, h0, sVec, sVec + 256, warp - 4, 8, lane);
      asm volatile("bar.sync 1, 256;" ::: "memory");
      if (lane == 0 && warp < 6) mbar_arrive(bar(VEC_FULL + 0));  // the two arrivals of phase 0
    }

    for (int item = blockIdx.x; item < num_items; item += gridDim.x, ++it) {
      const int b = item / p.H, h = item - b * p.H;
      // ---- per-row vectors of this item (written by warps 2-3 one item ahead)
      const float* sLse = sVec + (it & 1) * 512;
      const float* sD = sLse + 256;
      AT_BEGIN(at_a);
      mbar_wait(bar(VEC_FULL + (it & 1)), (it >> 1) & 1);
      AT_ADD(at_vec, at_a);

      for (int kt = 0; kt < n_kt; ++kt) {
        const int key = kt * 128 + row_in_tile;
        const bool key_ok = key < N;
        const uint32_t drop_item_rows = static_cast<uint32_t>(item) * static_cast<uint32_t>(N);
        for (int q64 = 0; q64 < n_q64; ++q64, ++sbc) {
          const int nq = min(64, Nk - q64 * 64);
          const uint32_t buf = sbc & 1u;
          const uint32_t pair = qtc & 1u;
          // first sub-tile of a query tile: the dQ MMAs that read this chunk pair two query tiles
          // ago have retired
          AT_BEGIN(at_b);
          if ((q64 & 1) == 0) mbar_wait(bar(DS_FREE + pair), ((qtc >> 1) & 1u) ^ 1u);
          AT_ADD(at_dsf, at_b);
          AT_BEGIN(at_c);
          mbar_wait(bar(S_FULL + buf), (sbc >> 1) & 1u);
          AT_ADD(at_sf, at_c);
          tc_fence_after();
          AT_BEGIN(at_d);
          if (hf * 32 < nq) {
            // 32 queries per warp; the last chunk of a ragged sub-tile holds 16
            const bool half_chunk = (hf * 32 + 32 > nq);
            const uint32_t col_s = lane_base + buf * 128u + static_cast<uint32_t>(hf * 32);
            const uint32_t col_dp = col_s + kColDPofs;
            uint32_t s[32], dp[32];
            if (half_chunk) {
              uint32_t s16[16], d16[16];
              tmem_ld_32x32b_x16(col_s, s16);
              tmem_ld_32x32b_x16(col_dp, d16);
              tmem_ld_wait();
#pragma unroll
              for (int j = 0; j < 16; ++j) {
                s[j] = s16[j];
                dp[j] = d16[j];
                s[16 + j] = 0u;
                dp[16 + j] = 0u;
              }
            } else {
              tmem_ld_32x32b_x32(col_s, s);
              tmem_ld_32x32b_x32(col_dp, dp);
              tmem_ld_wait();
            }
            AT_ADD(at_tld, at_d);
            AT_BEGIN(at_e);
            uint32_t pp[16], ds[16];
            const int q0 = q64 * 64 + hf * 32;
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
            AT_ADD(at_math, at_e);
            if (half_chunk) {
              uint32_t a8[8], b8[8];
#pragma unroll
              for (int j = 0; j < 8; ++j) {
                a8[j] = pp[j];
                b8[j] = ds[j];
              }
              tmem_st_32x32b_x8(col_s, a8);
              tmem_st_32x32b_x8(col_dp, b8);
            } else {
              tmem_st_32x32b_x16(col_s, pp);
              tmem_st_32x32b_x16(col_dp, ds);
            }
            // dS^T row -> smem: chunk (pair, q64 & 1), 16-byte pieces hf * 4 .. + 3
            const uint32_t rowa = sdS + (pair * 2u + static_cast<uint32_t>(q64 & 1)) * 16384u +
                                  static_cast<uint32_t>(row_in_tile) * 128u;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const int piece = hf * 4 + j;
              st_shared_v4(rowa + (static_cast<uint32_t>(piece ^ (row_in_tile & 7)) << 4),
                           ds[4 * j], ds[4 * j + 1], ds[4 * j + 2], ds[4 * j + 3]);
            }
            tmem_st_wait();
            fence_proxy_async_smem();
          }
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(bar(SM_DONE + buf));
          AT_ADD(at_st, at_d);
          flush_stores();
          if ((q64 & 1) || q64 == n_q64 - 1) ++qtc;
        }
        // dV_kt / dK_kt are stored one sub-block later (flush_stores), when their MMAs have long
        // retired, instead of waiting for them here
        pend_kv = true;
        pend_kt = kt;
        pend_b = b;
        pend_h = h;
        pend_ktc = ktc;
        ++ktc;
      }
      pend_q = true;
      pend_it = it;
    }
    flush_stores();
#ifdef VITK_ATTN_TRACE
    if (lane == 0 && warp == 4 && blockIdx.x < 160) {
      long long* t = g_attn_trace[blockIdx.x];
      t[4] = clock64() - at_s0;
      t[5] = at_vec; t[6] = at_dsf; t[7] = at_sf; t[8] = at_tld; t[9] = at_math;
      t[10] = at_st;  // whole sub-block body from the TMEM load to the arrive (includes 8 and 9)
      t[11] = at_wkv; t[12] = at_skv; t[13] = at_wq; t[14] = at_sq;
    }
#endif
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

static size_t tc2_smem_bytes(int N, int H, bool with_dbias) {
  const int Nk = (N + 15) & ~15;
  return 4 * static_cast<size_t>(Nk) * 128 + 65536 + 32768 + 4096 + 256 + 1024 +
         (with_dbias ? static_cast<size_t>(3) * H * 64 * 4 : 0);
}

bool attention_bwd_tc2_fits(int N, int H, bool with_dbias) {
  return N <= 256 && tc2_smem_bytes(N, H, with_dbias) <= 232448;
}

int attention_bwd_tc2(const void* qkv, const void* ctx, const void* dctx, const float* lse,
                     void* dqkv, int B, int N, int H, int hd, cudaStream_t stream,
                     const DropParams* drop, float* dbias) {
  VITK_REQUIRE(qkv && ctx && dctx && lse && dqkv, "attention_bwd: null operand");
  VITK_REQUIRE(hd == 64 && N >= 1 && attention_bwd_tc2_fits(N, H, dbias != nullptr),
               "attention_bwd(tc2): needs head_dim 64 and a sequence whose tiles fit shared memory");
  const int Nk = (N + 15) & ~15;
  const int D = H * 64;
  const size_t smem = tc2_smem_bytes(N, H, dbias != nullptr);
  VITK_TRY(opt_in_smem<attn_bwd_tc2_kernel<false>>(232448, "attn_bwd_tc2_kernel<false>"));
  VITK_TRY(opt_in_smem<attn_bwd_tc2_kernel<true>>(232448, "attn_bwd_tc2_kernel<true>"));
  CUtensorMap tq, tdo, tq1, tdo1, tout;
  const int rows0 = Nk < 128 ? Nk : 128, rows1 = Nk > 128 ? Nk - 128 : rows0;
  VITK_TRY(make_row_map(&tq, qkv, B, N, 3 * D, 3 * D, rows0));
  VITK_TRY(make_row_map(&tdo, dctx, B, N, D, D, rows0));
  VITK_TRY(make_row_map(&tq1, qkv, B, N, 3 * D, 3 * D, rows1));
  VITK_TRY(make_row_map(&tdo1, dctx, B, N, D, D, rows1));
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
    attn_bwd_tc2_kernel<true><<<grid, kThreads, smem, stream>>>(tq, tdo, tq1, tdo1, tout, prm);
  else
    attn_bwd_tc2_kernel<false><<<grid, kThreads, smem, stream>>>(tq, tdo, tq1, tdo1, tout, prm);
  VITK_CHECK_LAUNCH("attn_bwd_tc2_kernel");
  return VITK_OK;
}

}  // namespace vitk

#ifdef VITK_ATTN_TRACE
extern "C" int vitk_debug_attn_bwd_trace(long long* out_host, int n) {
  if (n > 320 * 16) n = 320 * 16;
  return cudaMemcpyFromSymbol(out_host, vitk::g_attn_trace, sizeof(long long) * n) == cudaSuccess ? n : -1;
}
#endif
