// tcgen05 attention for long sequences (208 < N <= 640 tokens, hd = 64): the forward of
// softmax(q k^T / sqrt(hd)) v (reference train.py:543-549) when the keys of a head do not fit one
// MMA tile - ViT-B/16 at 384 px has 577 tokens (BASELINE.json configs[4]).
//
// One (image, head) per work item, persistent CTAs.  K and V of the item stay in shared memory
// (<= 2 x 80 KB), the query rows are processed in tiles of 128, the keys in blocks of 128, in ONE
// pass with a lazily updated reference maximum (no second sweep over the key blocks):
//     S_j = Q K_j^T;  m_j = row max of block j;
//     the reference m_ref moves up to m_j only when m_j exceeds it by more than 8 (in the base-2
//     exponent), and only then O and the partial row sums are rescaled by 2^((m_ref - m_j) c);
//     P_j = exp2((S_j - m_ref) c) <= 2^8 -> TMEM (bf16), O += P_j V_j, row sums
// O / l at the end is exact whatever reference was used.  After the first block of a q-tile the
// reference rarely moves, so the rescale (a TMEM read-modify-write of the 64 output columns that
// has to wait for the previous block's P V) is off the common path.
// Every (q-tile, key block) is a "unit"; unit u uses TMEM score region u % 3, so the score product
// of unit u+2 is in flight while the softmax warps work on unit u and P V of unit u-1 runs.
//
//   warp 0       TMA producer: K, V per item; Q tiles double-buffered
//   warp 1       score-product issuer (one elected lane): keeps up to three score tiles in flight
//   warp 3       issues P V of a unit as soon as its probabilities are written
//   warps 4-15   softmax: three independent sets of four warps (one per TMEM lane quarter), set s
//                owns score region s and therefore every third unit; thread == query row over the
//                whole 128-key block (two sweeps of four tcgen05.ld: block maximum, then
//                exponentials).  The sets run out of phase, so one set's tcgen05.ld / st latencies
//                hide under the other two's exponentials; the reference maximum of a row is handed
//                from the set of unit u to the set of unit u+1 through shared memory + an mbarrier
//   warps 16-19  output: O / rowsum -> bf16 -> smem slab -> TMA store; log-sum-exp rows
//
// TMEM (512 columns): score regions [0,128) [128,256) [256,384) | O [384,448).
#include <cuda_bf16.h>

#include "attention_kernels.cuh"
#include "common.h"
#include "ptx.cuh"

namespace vitk {
using namespace ptx;

namespace {

constexpr int kThreads3 = 20 * 32;
constexpr int kQTile3 = 128 * 128;  // bytes of one 128-row x 64-column bf16 Q tile
constexpr uint32_t kOCol3 = 384;
constexpr int kKeyBlock = 128;

struct Tc3Params {
  int B, N, H, Nk;     // Nk = N rounded up to 16
  int n_qt, n_kb;      // query tiles, key blocks
  int parts;           // q-tile ranges per (image, head)
  float scale;
  float* lse;
};

enum : int {
  kKFull = 0, kKFree = 1,   // K of the item landed / its last score product retired
  kVFull = 18, kVFree = 19, // V of the item landed / its last P V retired
  kQFull = 2,    // [2]
  kQFree = 4,    // [2]
  kSFull = 6,    // [3] score tile of region r complete
  kDone = 9,     // [3] softmax finished with region r (P written), the 4 warps of set r
  kLReady = 12,  // row sums of a q-tile published (12 warps)
  kOFull = 13, kOFree = 14,
  kRegFree = 15,  // [3] P V of the unit in region r has retired: region reusable, O up to date
  kDec = 20,     // [3 sets][4 lane quarters] reference maximum after this set's unit published
  kFinal = 32,   // [4 lane quarters] reference maximum of the finished q-tile published
  kNumBars3 = 36
};

#ifdef VITK_ATTN_TRACE
#define TR3(role, idx, k)                                                                  \
  do {                                                                                     \
    if (blockIdx.x == 0 && (idx) < 60 && p.lse != nullptr)                                 \
      reinterpret_cast<long long*>(p.lse)[(role) * 256 + (idx) * 4 + (k)] = clock64();     \
  } while (0)
#else
#define TR3(role, idx, k) do { } while (0)
#endif

__global__ void __launch_bounds__(kThreads3, 1)
attn_fwd_tc3_kernel(const __grid_constant__ CUtensorMap tm_q,    // box {64, 128, 1}
                    const __grid_constant__ CUtensorMap tm_kv,   // box {64, min(Nk, 256), 1}
                    const __grid_constant__ CUtensorMap tm_kv_tail,  // box {64, Nk % 256, 1}
                    const __grid_constant__ CUtensorMap tm_o,    // box {64, 32, 1}
                    const Tc3Params p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = smem_u32(smem_raw);
  const uint32_t base = (raw_addr + 1023u) & ~1023u;
  uint8_t* smem = smem_raw + (base - raw_addr);

  const int Nk = p.Nk, N = p.N;
  const uint32_t kv_bytes = static_cast<uint32_t>(Nk) * 128u;      // multiple of 2048
  const uint32_t sK = base, sV = sK + kv_bytes;
  const uint32_t sQ = sV + kv_bytes;                               // 2 x 16 KB
  const uint32_t staging_base = sQ + 2u * kQTile3;                 // 4 warps x 4 KB
  const uint32_t stat_base = staging_base + 4u * 4096u;
  // float [2 q-tile parities][4 (3 used) sets][128 rows] partial row sums, then [128] the running
  // reference maximum of each row (handed from unit to unit), then [2][128] final reference
  // maxima of a q-tile (row-sum conversion, log-sum-exp)
  float* l_smem = reinterpret_cast<float*>(smem + (stat_base - base));
  float* mref_smem = l_smem + 2 * 4 * 128;
  float* mrow_smem = mref_smem + 2 * 4 * 128;  // (spare room after the 128 running maxima)
  const uint32_t bar_base = stat_base + (2 * 4 * 128 * 2 + 2 * 128) * 4u;
  auto bar = [&](int i) { return bar_base + 8u * i; };
  volatile uint32_t* tmem_slot =
      reinterpret_cast<volatile uint32_t*>(smem + (bar_base - base) + 8 * kNumBars3);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  // Work item = (image, head, part): with fewer heads than SMs the q-tiles of a head are split into
  // `parts` ranges handled by different CTAs.
  const int parts = p.parts;
  const int num_items = p.B * p.H * parts;
  const int D = p.H * 64;
  const int n_qt = p.n_qt, n_kb = p.n_kb;
  auto qt_begin = [&](int part) { return (n_qt * part) / parts; };
  auto block_keys = [&](int j) { return min(kKeyBlock, Nk - j * kKeyBlock); };  // multiple of 16

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tm_q);
    prefetch_tmap(&tm_kv);
    prefetch_tmap(&tm_kv_tail);
    prefetch_tmap(&tm_o);
  }
  if (warp == 1 && lane == 0) {
    mbar_init(bar(kKFull), 1);
    mbar_init(bar(kKFree), 1);
    mbar_init(bar(kVFull), 1);
    mbar_init(bar(kVFree), 1);
    for (int b = 0; b < 2; ++b) {
      mbar_init(bar(kQFull + b), 1);
      mbar_init(bar(kQFree + b), 1);
    }
    for (int r = 0; r < 3; ++r) {
      mbar_init(bar(kSFull + r), 1);
      mbar_init(bar(kDone + r), 4);
      mbar_init(bar(kRegFree + r), 1);
    }
    mbar_init(bar(kLReady), 12);
    for (int i = 0; i < 12; ++i) mbar_init(bar(kDec + i), 1);
    for (int i = 0; i < 4; ++i) mbar_init(bar(kFinal + i), 1);
    mbar_init(bar(kOFull), 1);
    mbar_init(bar(kOFree), 4);
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

  if (warp < 4) {
    setmaxnreg_dec<40>();
    if (warp == 0) {
      // ======================= TMA producer =======================
      if (lane == 0) {
        int it = 0;
        uint32_t qc = 0;  // running q-tile counter -> Q buffer qc & 1
        for (int item = blockIdx.x; item < num_items; item += gridDim.x, ++it) {
          const int head = item / parts, part = item - head * parts;
          const int b = head / p.H, h = head - b * p.H;
          // K and V have their own barriers: K is free again once the item's last score product
          // has retired (early - the score issuer runs three units ahead), V once its last P V
          // has, so the next item's K arrives under this item's last softmax blocks and its V
          // under the next item's first one
          mbar_wait(bar(kKFree), (it & 1) ^ 1u);
          mbar_arrive_expect_tx(bar(kKFull), kv_bytes);
          for (int r0 = 0; r0 < Nk; r0 += 256) {   // TMA boxes hold at most 256 rows
            const CUtensorMap* tm = (Nk - r0 >= 256 || Nk < 256) ? &tm_kv : &tm_kv_tail;
            tma_load_3d(sK + r0 * 128u, tm, bar(kKFull), D + h * 64, r0, b);
          }
          mbar_wait(bar(kVFree), (it & 1) ^ 1u);
          mbar_arrive_expect_tx(bar(kVFull), kv_bytes);
          for (int r0 = 0; r0 < Nk; r0 += 256) {
            const CUtensorMap* tm = (Nk - r0 >= 256 || Nk < 256) ? &tm_kv : &tm_kv_tail;
            tma_load_3d(sV + r0 * 128u, tm, bar(kVFull), 2 * D + h * 64, r0, b);
          }
          for (int t = qt_begin(part); t < qt_begin(part + 1); ++t, ++qc) {
            const uint32_t buf = qc & 1u;
            mbar_wait(bar(kQFree + buf), ((qc >> 1) & 1) ^ 1u);
            mbar_arrive_expect_tx(bar(kQFull + buf), kQTile3);
            tma_load_3d(sQ + buf * kQTile3, &tm_q, bar(kQFull + buf), h * 64, t * 128, b);
          }
        }
      }
    } else if (warp == 1) {
      // ============ score-product issuer (whole warp converged, one elected lane issues) ========
      // A single issuing thread is the bottleneck of this kernel (descriptor arithmetic and ~100
      // cycles per tcgen05.mma issue: 20 score MMAs + 40 P V MMAs per q-tile), so the two product
      // kinds are issued by two warps.  This one runs up to three units ahead: region u % 3 is
      // free once unit u - 3 has been completed by warp 3 (`region_free`).
      int it = 0;
      uint32_t u = 0, r = 0, qc = 0;
      for (int item = blockIdx.x; item < num_items; item += gridDim.x, ++it) {
        const int part = item % parts;
        mbar_wait(bar(kKFull), it & 1);
        tc_fence_after();
        const int t_end = qt_begin(part + 1);
        for (int t = qt_begin(part); t < t_end; ++t, ++qc) {
          const uint32_t qbuf = qc & 1u;
          mbar_wait(bar(kQFull + qbuf), (qc >> 1) & 1);  // the Q tile has landed
          tc_fence_after();
          const uint64_t q_desc = make_desc_sw128(sQ + qbuf * kQTile3, 16, 1024);
          for (int j = 0; j < n_kb; ++j, ++u) {
            if (u >= 3u) {
              mbar_wait(bar(kRegFree + r), ((u / 3u) - 1u) & 1u);
              tc_fence_after();
            }
            TR3(2, u, 0);
            const uint32_t idesc_s = make_idesc_bf16(128, block_keys(j));
            const uint64_t k_desc = make_desc_sw128(sK + j * (kKeyBlock * 128u), 16, 1024);
            const bool last_of_qt = (j == n_kb - 1);
            if (elect_one_sync()) {
#pragma unroll
              for (int k = 0; k < 4; ++k)
                mma_bf16_ss(tmem_base + r * 128u, q_desc + 2u * k, k_desc + 2u * k, idesc_s,
                            k > 0 ? 1u : 0u);
              mma_commit(bar(kSFull + r));
              if (last_of_qt) mma_commit(bar(kQFree + qbuf));  // last reader of this Q tile
              if (last_of_qt && t == t_end - 1) mma_commit(bar(kKFree));  // last reader of K
            }
            __syncwarp();
            TR3(2, u, 1);
            r = (r == 2u) ? 0u : r + 1u;
          }
        }
      }
    } else if (warp == 3) {
      // ============ P V issuer ============
      const uint32_t idesc_pv = make_idesc_bf16(128, 64, 0, 1);  // B (= V) is MN-major
      uint32_t u = 0, r = 0, qc = 0;
      int it = 0;
      for (int item = blockIdx.x; item < num_items; item += gridDim.x, ++it) {
        const int part = item % parts;
        const int t_end = qt_begin(part + 1);
        mbar_wait(bar(kVFull), it & 1);
        for (int t = qt_begin(part); t < t_end; ++t, ++qc) {
          for (int j = 0; j < n_kb; ++j, ++u) {
            mbar_wait(bar(kDone + r), (u / 3u) & 1u);  // the probabilities of this unit are written
            TR3(0, u, 0);
            tc_fence_after();
            if (j == 0) {
              mbar_wait(bar(kOFree), (qc & 1u) ^ 1u);  // the previous O tile has been read out
              tc_fence_after();
            }
            const int nk = block_keys(j);
            // V rows of this key block (128 B each, 8-row swizzle atoms 1024 B apart); 16 keys
            // per MMA; P as bf16 pairs at the start of each 32-column chunk of the region
            const uint64_t v_desc = make_desc_sw128(sV + j * (kKeyBlock * 128u), kv_bytes, 1024);
            const bool last_of_item = (t == t_end - 1 && j == n_kb - 1);
            if (elect_one_sync()) {
              // fully unrolled and predicated: two instructions per MMA instead of a rolled
              // loop's eight (the issuing warp competes with five busy warps for issue slots)
#pragma unroll
              for (int ks = 0; ks < kKeyBlock / 16; ++ks)
                if (ks < nk / 16)
                  mma_bf16_ts(tmem_base + kOCol3,
                              tmem_base + r * 128u +
                                  static_cast<uint32_t>((ks >> 1) * 32 + (ks & 1) * 8),
                              v_desc + static_cast<uint64_t>(ks) * 128u, idesc_pv,
                              (j > 0 || ks > 0) ? 1u : 0u);
              mma_commit(bar(kRegFree + r));  // P consumed and O up to date when these retire
              if (j == n_kb - 1) mma_commit(bar(kOFull));
              if (last_of_item) mma_commit(bar(kVFree));  // last reader of V
            }
            __syncwarp();
            TR3(0, u, 1);
            r = (r == 2u) ? 0u : r + 1u;
          }
        }
      }
    }
  } else if (warp < 16) {
    setmaxnreg_inc<120>();
    // ============ softmax: set = score region, thread == query row over the whole key block =====
    const int set = (warp - 4) >> 2;  // owns region `set` and the units u with u % 3 == set
    const int q = warp & 3;           // TMEM lane quarter
    const float c = p.scale * kLog2e;
    const uint64_t cc = pack2(__float_as_uint(c), __float_as_uint(c));
    const int r_in_tile = q * 32 + lane;
    const uint32_t lane_off = static_cast<uint32_t>(q * 32) << 16;
    const uint32_t treg = tmem_base + lane_off + static_cast<uint32_t>(set) * 128u;
    const uint32_t prev_set = (set + 2) % 3;
    uint32_t u = 0, qc = 0;
    for (int item = blockIdx.x; item < num_items; item += gridDim.x) {
      const int part = item % parts;
      for (int t = qt_begin(part); t < qt_begin(part + 1); ++t, ++qc) {
        const int par = qc & 1;
        const bool warp_rows = t * 128 + q * 32 < N;
        float m_mine = -INFINITY;  // reference this thread's partial row sum is relative to
        uint64_t la = 0ull, lb = 0ull;
        for (int j = 0; j < n_kb; ++j, ++u) {
          if (u % 3u != static_cast<uint32_t>(set)) continue;
          mbar_wait(bar(kSFull + set), (u / 3u) & 1u);
          if (warp == 4 && lane == 0) TR3(1, u, 0);
          tc_fence_after();
          const int nk = block_keys(j);           // multiple of 16
          const int valid = min(nk, N - j * kKeyBlock);  // keys >= N are TMA zero fill
          const int n32 = nk >> 5;
          const bool tail16 = (nk & 31) != 0;
          // ---- sweep 1: block maximum of the row
          float m_blk = -INFINITY;
          if (warp_rows) {
            // two 32-column loads in flight per wait (the wait costs ~100 cycles whatever it covers)
            for (int ch = 0; ch < n32; ch += 2) {
              uint32_t v[2][32];
              const bool two = ch + 1 < n32;
              tmem_ld_32x32b_x32(treg + ch * 32, v[0]);
              if (two) tmem_ld_32x32b_x32(treg + (ch + 1) * 32, v[1]);
              tmem_ld_wait();
#pragma unroll
              for (int hh = 0; hh < 2; ++hh) {
                if (hh == 1 && !two) break;
                const int k0 = (ch + hh) * 32;
                if (k0 + 32 <= valid) {
                  float a0 = m_blk, a1 = -INFINITY, a2 = -INFINITY, a3 = -INFINITY;
#pragma unroll
                  for (int i = 0; i < 4; ++i) {
                    a0 = fmax3(a0, __uint_as_float(v[hh][8 * i]), __uint_as_float(v[hh][8 * i + 1]));
                    a1 = fmax3(a1, __uint_as_float(v[hh][8 * i + 2]), __uint_as_float(v[hh][8 * i + 3]));
                    a2 = fmax3(a2, __uint_as_float(v[hh][8 * i + 4]), __uint_as_float(v[hh][8 * i + 5]));
                    a3 = fmax3(a3, __uint_as_float(v[hh][8 * i + 6]), __uint_as_float(v[hh][8 * i + 7]));
                  }
                  m_blk = fmaxf(fmaxf(a0, a1), fmaxf(a2, a3));
                } else {
#pragma unroll
                  for (int i = 0; i < 32; ++i)
                    if (k0 + i < valid) m_blk = fmaxf(m_blk, __uint_as_float(v[hh][i]));
                }
              }
            }
            if (tail16) {
              uint32_t v[16];
              tmem_ld_32x32b_x16(treg + n32 * 32, v);
              tmem_ld_wait();
              const int k0 = n32 * 32;
#pragma unroll
              for (int i = 0; i < 16; ++i)
                if (k0 + i < valid) m_blk = fmaxf(m_blk, __uint_as_float(v[i]));
            }
          }
          // ---- reference maximum: taken over from the previous unit's set, moved lazily
          float m_ref = m_blk;
          // (the previous unit's set has finished with mref_smem, also across a q-tile boundary)
          if (u > 0u) mbar_wait(bar(kDec + prev_set * 4 + q), ((u - 1u) / 3u) & 1u);
          if (j > 0) {
            m_ref = mref_smem[r_in_tile];
            const bool resc = warp_rows && ((m_blk - m_ref) * c > 8.f);
            if (__any_sync(0xffffffffu, resc)) {
              // O += P V of the previous unit must have retired before O is touched
              mbar_wait(bar(kRegFree + prev_set), ((u - 1u) / 3u) & 1u);
              tc_fence_after();
              const float f = resc ? exp2f((m_ref - m_blk) * c) : 1.f;
#pragma unroll
              for (int h2 = 0; h2 < 2; ++h2) {
                uint32_t o[32];
                tmem_ld_32x32b_x32(tmem_base + lane_off + kOCol3 + h2 * 32, o);
                tmem_ld_wait();
#pragma unroll
                for (int i = 0; i < 32; ++i) o[i] = __float_as_uint(__uint_as_float(o[i]) * f);
                tmem_st_32x32b_x16(tmem_base + lane_off + kOCol3 + h2 * 32,
                                   *reinterpret_cast<uint32_t(*)[16]>(&o[0]));
                tmem_st_32x32b_x16(tmem_base + lane_off + kOCol3 + h2 * 32 + 16,
                                   *reinterpret_cast<uint32_t(*)[16]>(&o[16]));
              }
              tmem_st_wait();
              tc_fence_before();
            }
            if (resc) m_ref = m_blk;
          }
          mref_smem[r_in_tile] = m_ref;
          if (j == n_kb - 1) {
            // Every set has published its row sums of the previous q-tile: with fewer key blocks
            // than sets a set may have no unit in this q-tile, and without this wait the others
            // could lap it (kFinal / kLReady arrivals of two q-tiles would mix).
            if (qc > 0u) mbar_wait(bar(kLReady), (qc - 1u) & 1u);
            mrow_smem[par * 128 + r_in_tile] = m_ref;
          }
          __syncwarp();
          if (lane == 0) {
            mbar_arrive(bar(kDec + set * 4 + q));
            if (j == n_kb - 1) mbar_arrive(bar(kFinal + q));
          }
          // ---- this thread's partial row sum follows the reference
          if (m_mine != m_ref) {
            if (m_mine == -INFINITY) {
              la = lb = 0ull;
            } else {
              const float f = exp2f((m_mine - m_ref) * c);
              const uint64_t ff = pack2(__float_as_uint(f), __float_as_uint(f));
              la = fmul2(la, ff);
              lb = fmul2(lb, ff);
            }
            m_mine = m_ref;
          }
          // ---- sweep 2: p = 2^((s - m_ref) c), row sum, P -> TMEM (bf16 pairs at the start of
          //      each 32-column chunk, where the P V issuer expects them)
          if (warp_rows) {
            const float nm = -m_ref * c;
            const uint64_t nmc = pack2(__float_as_uint(nm), __float_as_uint(nm));
            for (int ch = 0; ch < n32; ++ch) {
              uint32_t v[32];
              tmem_ld_32x32b_x32(treg + ch * 32, v);
              tmem_ld_wait();
              const int k0 = ch * 32;
              uint32_t pk[16];
#pragma unroll
              for (int i = 0; i < 16; ++i) {
                float t0, t1;
                unpack2(ffma2(pack2(v[2 * i], v[2 * i + 1]), cc, nmc), t0, t1);
                float e0 = ex2_approx(t0);
                float e1 = ex2_approx(t1);
                if (k0 + 32 > valid) {
                  if (k0 + 2 * i >= valid) e0 = 0.f;
                  if (k0 + 2 * i + 1 >= valid) e1 = 0.f;
                }
                const uint64_t e = pack2(__float_as_uint(e0), __float_as_uint(e1));
                if (i & 1) lb = fadd2(lb, e); else la = fadd2(la, e);
                pk[i] = pack_bf16x2(e0, e1);
              }
              tmem_st_32x32b_x16(treg + ch * 32, pk);
            }
            if (tail16) {
              uint32_t v[16];
              tmem_ld_32x32b_x16(treg + n32 * 32, v);
              tmem_ld_wait();
              const int k0 = n32 * 32;
              uint32_t pk[8];
#pragma unroll
              for (int i = 0; i < 8; ++i) {
                float t0, t1;
                unpack2(ffma2(pack2(v[2 * i], v[2 * i + 1]), cc, nmc), t0, t1);
                float e0 = ex2_approx(t0);
                float e1 = ex2_approx(t1);
                if (k0 + 2 * i >= valid) e0 = 0.f;
                if (k0 + 2 * i + 1 >= valid) e1 = 0.f;
                const uint64_t e = pack2(__float_as_uint(e0), __float_as_uint(e1));
                if (i & 1) lb = fadd2(lb, e); else la = fadd2(la, e);
                pk[i] = pack_bf16x2(e0, e1);
              }
              tmem_st_32x32b_x8(treg + n32 * 32, pk);
            }
            tmem_st_wait();
          }
          tc_fence_before();
          __syncwarp();
          if (warp == 4 && lane == 0) TR3(1, u, 1);
          if (lane == 0) mbar_arrive(bar(kDone + set));
        }
        // ---- end of the q-tile: bring the partial row sum to the final reference and publish it
        mbar_wait(bar(kFinal + q), qc & 1u);
        {
          const float m_fin = mrow_smem[par * 128 + r_in_tile];
          float l0, l1, l2, l3;
          unpack2(la, l0, l1);
          unpack2(lb, l2, l3);
          float l = (l0 + l1) + (l2 + l3);
          if (m_mine == -INFINITY) l = 0.f;
          else if (m_mine != m_fin) l *= exp2f((m_mine - m_fin) * c);
          l_smem[(par * 4 + set) * 128 + r_in_tile] = l;
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(bar(kLReady));
      }
    }
  } else {
    setmaxnreg_dec<72>();
    // ======================= output: O / rowsum -> bf16 -> TMA store =======================
    const int q = warp & 3;
    const uint32_t o_addr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + kOCol3;
    const uint32_t slab = staging_base + static_cast<uint32_t>(warp - 16) * 4096u;
    uint32_t qc = 0;
    for (int item = blockIdx.x; item < num_items; item += gridDim.x) {
      const int head = item / parts, part = item - head * parts;
      const int b = head / p.H, h = head - b * p.H;
      for (int t = qt_begin(part); t < qt_begin(part + 1); ++t, ++qc) {
        const int par = qc & 1;
        const int row0 = t * 128 + q * 32;
        const bool rows = row0 < N;
        mbar_wait(bar(kLReady), qc & 1u);   // the q-tile's row statistics are in shared memory
        mbar_wait(bar(kOFull), qc & 1u);
        tc_fence_after();
        float l = 1.f, m = 0.f;
        uint32_t pk[32];
        if (rows) {
          const int r = q * 32 + lane;
          l = (l_smem[(par * 4 + 0) * 128 + r] + l_smem[(par * 4 + 1) * 128 + r]) +
              l_smem[(par * 4 + 2) * 128 + r];
          m = mrow_smem[par * 128 + r];
          const float inv_l = 1.f / l;
#pragma unroll
          for (int half = 0; half < 2; ++half) {
            uint32_t o[32];
            tmem_ld_32x32b_x32(o_addr + half * 32, o);
            tmem_ld_wait();
#pragma unroll
            for (int i = 0; i < 16; ++i)
              pk[half * 16 + i] = pack_bf16x2(__uint_as_float(o[2 * i]) * inv_l,
                                              __uint_as_float(o[2 * i + 1]) * inv_l);
          }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(bar(kOFree));
        if (rows) {
          const int r = row0 + lane;
#ifndef VITK_ATTN_TRACE
          if (p.lse != nullptr && r < N)
            p.lse[(static_cast<size_t>(b) * p.H + h) * N + r] = m * p.scale + logf(l);
#else
          (void)r; (void)m;
#endif
          if (lane == 0) tma_store_wait_read<0>();  // the previous slab has left smem
          __syncwarp();
          const uint32_t row = slab + static_cast<uint32_t>(lane) * 128u;
#pragma unroll
          for (int i = 0; i < 8; ++i)
            st_shared_v4(row + (static_cast<uint32_t>(i ^ (lane & 7)) << 4), pk[4 * i],
                         pk[4 * i + 1], pk[4 * i + 2], pk[4 * i + 3]);
          fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) {
            tma_store_3d(&tm_o, slab, h * 64, row0, b);  // rows >= N are clipped
            tma_store_commit();
          }
        }
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
}

}  // namespace

int attention_fwd_tc3(const void* qkv, void* ctx, float* lse, int B, int N, int H, int hd,
                      cudaStream_t stream) {
  VITK_REQUIRE(qkv && ctx, "attention: null operand");
  VITK_REQUIRE(hd == 64 && N >= 1 && N <= 640, "attention(tc3): needs head_dim 64 and N <= 640");
  VITK_REQUIRE(B > 0 && H > 0, "attention: bad shape B=%d H=%d", B, H);
  VITK_REQUIRE(device_cc() >= 100, "attention(tc3): requires an sm_100 device");
  const int Nk = (N + 15) & ~15;
  const int D = H * 64;
  const size_t smem = 2 * static_cast<size_t>(Nk) * 128 + 2 * kQTile3 + 4 * 4096 +
                      (2 * 4 * 128 * 2 + 2 * 128) * 4 + 8 * kNumBars3 + 64 + 1024;
  VITK_REQUIRE(smem <= 232448, "attention(tc3): shared memory budget exceeded");
  VITK_TRY(opt_in_smem<attn_fwd_tc3_kernel>(232448, "attn_fwd_tc3_kernel"));
  CUtensorMap tq, tkv, tkv_tail, to;
  const int kv_box = Nk < 256 ? Nk : 256;
  const int kv_tail = (Nk >= 256 && Nk % 256 != 0) ? Nk % 256 : kv_box;
  VITK_TRY(make_row_map(&tq, qkv, B, N, 3 * D, 3 * D, 128));
  VITK_TRY(make_row_map(&tkv, qkv, B, N, 3 * D, 3 * D, kv_box));
  VITK_TRY(make_row_map(&tkv_tail, qkv, B, N, 3 * D, 3 * D, kv_tail));
  VITK_TRY(make_row_map(&to, ctx, B, N, D, D, 32));
  Tc3Params prm;
  prm.B = B;
  prm.N = N;
  prm.H = H;
  prm.Nk = Nk;
  prm.n_qt = (N + 127) / 128;
  prm.n_kb = (Nk + kKeyBlock - 1) / kKeyBlock;
  prm.scale = 1.0f / sqrtf(static_cast<float>(hd));
  prm.lse = lse;
  int grid = sm_count();
  // With fewer heads than SMs the q-tiles of a head are split over several CTAs (K and V are then
  // loaded once per part, from L2).  With more heads than SMs a split only trades the round-robin
  // tail for extra un-overlapped K / V loads (measured neutral), so it stays off.
  prm.parts = 1;
  {
    const long long heads = static_cast<long long>(B) * H;
    if (heads < grid) {
      long long want = (grid + heads - 1) / heads;
      if (want > prm.n_qt) want = prm.n_qt;
      if (want > 4) want = 4;
      prm.parts = static_cast<int>(want);
    }
  }
  grid = persistent_grid(static_cast<long long>(B) * H * prm.parts);
  ProfileScope prof(PROF_ATTN, attention_flops(B, H, N, N, hd), stream);
  attn_fwd_tc3_kernel<<<grid, kThreads3, smem, stream>>>(tq, tkv, tkv_tail, to, prm);
  VITK_CHECK_LAUNCH("attn_fwd_tc3_kernel");
  return VITK_OK;
}

}  // namespace vitk
