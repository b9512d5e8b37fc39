// tcgen05 attention, software-pipelined across (image, head) items: the forward of
// softmax(q k^T / sqrt(hd)) v (reference train.py:543-549) for N <= 208 tokens, hd = 64.
//
// Same data path as attention_tc.cu (3-D TMA over the packed qkv activation, S and P in TMEM, V as an
// MN-major smem operand, ctx written by TMA) but organised around what bounds this kernel: the
// exponentials (16 MUFU results / clk / SM).  A lone warp per scheduler only sustains one MUFU per
// ~12-15 cycles (latency, fixed tcgen05.wait / st costs; tests/ubench_softmax_chunk.cu), so the
// softmax runs on 16 warps - four per scheduler - and everything else is moved off them:
//
//   warp 0       TMA producer: Q tile(s), K, V of item i+1 while item i is being processed
//   warp 1       MMA issuer (one elected lane).  Order per item: PV_0(i), S_0(i+1), PV_1(i), S_1(i+1):
//                the score MMA of the NEXT item is queued right behind the PV MMA that frees its TMEM
//                region (the tensor pipe executes one thread's MMAs in issue order)
//   warps 4-19   softmax, all sixteen on the same q-tile, the two q-tiles of an item in turn (while
//                they work on one tile the tensor pipe runs PV of the previous and S of the next
//                tile in the other TMEM region).  Warps 4q..4q+3 (q = 0..3) own one quarter of the
//                key columns each, thread == query row of that quarter.  Two sweeps over the row in
//                TMEM: max (quarters exchange it through smem + a 128-thread named barrier), then
//                exp2 / row sum / P -> TMEM as bf16 over the warp's own, already consumed S columns
//   warps 20-23  output: O (own TMEM columns, shared by both q-tiles) / rowsum -> bf16 -> smem slab
//                -> TMA store; also the log-sum-exp rows saved for the backward pass
//
// TMEM (512 columns): S_0 / P_0 [0, 224) | S_1 / P_1 [224, 448) | O [448, 512).
// Registers: 768 threads x 80 at launch, re-balanced with setmaxnreg to 40 / 88 (softmax) / 72.
#include <cuda_bf16.h>

#include "attention_kernels.cuh"
#include "common.h"
#include "dropout.cuh"
#include "ptx.cuh"

namespace vitk {
using namespace ptx;

namespace {

constexpr int kThreads2 = 24 * 32;
constexpr int kQTile = 128 * 128;  // bytes of one 128-row x 64-column bf16 Q tile
constexpr uint32_t kRegion = 224;  // TMEM columns per q-tile (S fp32, later P bf16)
constexpr uint32_t kOColumn = 448;

struct Tc2Params {
  int B, N, H, Nk, q_tiles;
  int descending;  // walk the (image, head) items from the last to the first
  DropParams drop; // attention-probability dropout (train.py:545); element = ((b H + h) N + i) Nk + j
  float scale;
  float* lse;
};

// Row maximum over COLS score columns starting at key k0 (4 independent chains of 3-input max).
template <int COLS>
__device__ __forceinline__ void chunk_max(const uint32_t (&v)[COLS], int k0, int N, float (&m)[4]) {
  if (k0 + COLS <= N) {
#pragma unroll
    for (int j = 0; j < COLS / 8; ++j) {
      m[0] = fmax3(m[0], __uint_as_float(v[8 * j]), __uint_as_float(v[8 * j + 1]));
      m[1] = fmax3(m[1], __uint_as_float(v[8 * j + 2]), __uint_as_float(v[8 * j + 3]));
      m[2] = fmax3(m[2], __uint_as_float(v[8 * j + 4]), __uint_as_float(v[8 * j + 5]));
      m[3] = fmax3(m[3], __uint_as_float(v[8 * j + 6]), __uint_as_float(v[8 * j + 7]));
    }
  } else {
    const int valid = N - k0;
#pragma unroll
    for (int j = 0; j < COLS; ++j)
      if (j < valid) m[j & 3] = fmaxf(m[j & 3], __uint_as_float(v[j]));
  }
}

// Second sweep, one chunk of COLS keys of one row, in place in the registers the TMEM load filled:
// p = 2^(s c - m c), row sum, P -> TMEM as bf16 pairs at column pcol.  MASKED is only instantiated
// for the last chunk of a row (keys >= N are TMA zero fill and must not count).
// DROP: the probabilities written for the PV product are dropped / rescaled (the row sum keeps the
// undropped values: dropout follows the softmax normalisation); row_pairs = pair index of key 0.
template <int COLS, bool MASKED, bool DROP>
__device__ __forceinline__ void exp_chunk(uint32_t (&v)[COLS], int k0, int N, uint64_t cc,
                                          uint64_t nmc, uint32_t pcol, uint64_t& la, uint64_t& lb,
                                          const DropParams& drop, uint32_t row_pairs) {
  const int valid = N - k0;  // only read when MASKED
  uint32_t pk[COLS / 2];
#pragma unroll
  for (int j = 0; j < COLS / 2; ++j) {
    float t0, t1;
    unpack2(ffma2(pack2(v[2 * j], v[2 * j + 1]), cc, nmc), t0, t1);
    float e0 = ex2_approx(t0);
    float e1 = ex2_approx(t1);
    if constexpr (MASKED) {
      if (2 * j >= valid) e0 = 0.f;
      if (2 * j + 1 >= valid) e1 = 0.f;
    }
    const uint64_t e = pack2(__float_as_uint(e0), __float_as_uint(e1));
    if (j & 1) lb = fadd2(lb, e); else la = fadd2(la, e);
    if constexpr (DROP) {
      const uint32_t bits = drop_bits(row_pairs + static_cast<uint32_t>(k0 / 2 + j), drop.key);
      e0 = drop_keep_lo(bits, drop.thresh) ? e0 * drop.scale : 0.f;
      e1 = drop_keep_hi(bits, drop.thresh) ? e1 * drop.scale : 0.f;
    }
    pk[j] = pack_bf16x2(e0, e1);
  }
  if constexpr (COLS == 32) tmem_st_32x32b_x16(pcol, pk);
  else tmem_st_32x32b_x8(pcol, pk);
}

template <int COLS, bool DROP>
__device__ __forceinline__ void exp_chunk_any(uint32_t (&v)[COLS], int k0, int N, uint64_t cc,
                                              uint64_t nmc, uint32_t pcol, uint64_t& la,
                                              uint64_t& lb, const DropParams& drop,
                                              uint32_t row_pairs) {
  if (k0 + COLS <= N) exp_chunk<COLS, false, DROP>(v, k0, N, cc, nmc, pcol, la, lb, drop, row_pairs);
  else exp_chunk<COLS, true, DROP>(v, k0, N, cc, nmc, pcol, la, lb, drop, row_pairs);
}

// Debug aid (build with -DVITK_ATTN_TRACE): CTA 0 records SM-clock timestamps of its first 8 items
// into the lse buffer, read back by tests/trace_attn.py to see how the roles overlap.
#ifdef VITK_ATTN_TRACE
#define TR(role, idx, k)                                                      \
  do {                                                                        \
    if (blockIdx.x == 0 && (idx) < 8 && p.lse != nullptr)                     \
      reinterpret_cast<long long*>(p.lse)[(role) * 64 + (idx) * 8 + (k)] = clock64(); \
  } while (0)
#else
#define TR(role, idx, k) do { } while (0)
#endif

// DROP: attention-probability dropout compiled in (separate instantiation; the inference kernel
// carries none of it).
template <bool DROP>
__global__ void __launch_bounds__(kThreads2, 1)
attn_fwd_tc2_kernel(const __grid_constant__ CUtensorMap tm_q,
                    const __grid_constant__ CUtensorMap tm_kv,
                    const __grid_constant__ CUtensorMap tm_o, const Tc2Params p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = smem_u32(smem_raw);
  const uint32_t base = (raw_addr + 1023u) & ~1023u;
  uint8_t* smem = smem_raw + (base - raw_addr);

  const int Nk = p.Nk;
  const uint32_t kv_bytes = static_cast<uint32_t>(Nk) * 128u;
  const uint32_t stage_bytes = 2u * kQTile + 2u * kv_bytes;
  const uint32_t staging_base = base + 2u * stage_bytes;  // 4 output warps x 2 slabs x 4 KB
  // row statistics, float [2 item parities][2 tiles][4 column quarters][128 rows]: maxima, sums
  const uint32_t m_base = staging_base + 8u * 4096u;
  const uint32_t l_base = m_base + 8192u;
  const uint32_t bar_base = l_base + 8192u;
  // Q/K and V of a stage are tracked separately: Q and K are dead as soon as the score MMAs of the
  // item have run - a whole item earlier than V - so their reload gets that much more lead time
  // over the HBM latency.
  auto qk_full = [&](int s) { return bar_base + 8u * s; };
  auto qk_empty = [&](int s) { return bar_base + 8u * (2 + s); };
  auto v_full = [&](int s) { return bar_base + 8u * (4 + s); };
  auto v_empty = [&](int s) { return bar_base + 8u * (6 + s); };
  auto s_full = [&](int t) { return bar_base + 8u * (8 + t); };
  auto p_full = [&](int t) { return bar_base + 8u * (10 + t); };
  const uint32_t o_full = bar_base + 8u * 12;
  const uint32_t o_free = bar_base + 8u * 13;
  volatile uint32_t* tmem_slot =
      reinterpret_cast<volatile uint32_t*>(smem + (bar_base - base) + 8 * 14);
  float* m_smem = reinterpret_cast<float*>(smem + (m_base - base));
  float* l_smem = reinterpret_cast<float*>(smem + (l_base - base));
  auto stat_idx = [](int par, int t, int cq, int row) { return ((par * 2 + t) * 4 + cq) * 128 + row; };

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int num_items = p.B * p.H;
  const int D = p.H * 64;
  const int q_tiles = p.q_tiles;
  // key columns of the four softmax quarters: multiples of 16 (whole PV MMA steps), the first
  // `rem` quarters one step wider
  const int steps = Nk >> 4;
  const int qbase = steps >> 2, qrem = steps & 3;
  auto quarter_begin = [&](int cq) { return 16 * (cq * qbase + (cq < qrem ? cq : qrem)); };

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tm_q);
    prefetch_tmap(&tm_kv);
    prefetch_tmap(&tm_o);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < 2; ++s) {
      mbar_init(qk_full(s), 1);
      mbar_init(qk_empty(s), 1);
      mbar_init(v_full(s), 1);
      mbar_init(v_empty(s), 1);
      mbar_init(s_full(s), 1);
      mbar_init(p_full(s), 16);
    }
    mbar_init(o_full, 1);
    mbar_init(o_free, 4);
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

  // 768 threads x 80 registers at launch; the producer / issuer warpgroup hands most of its share to
  // the four softmax warpgroups: 128 x (40 + 4 x 88 + 72) = 58 K <= the 60 K allocated at launch.
  if (warp < 4) {
    setmaxnreg_dec<40>();
    if (warp == 0) {
      // ======================= TMA producer =======================
      if (lane == 0) {
        int it = 0;
        for (int item = blockIdx.x; item < num_items; item += gridDim.x, ++it) {
          const int stage = it & 1;
          const uint32_t phase = (it >> 1) & 1;
          const int item_id = p.descending ? num_items - 1 - item : item;
          const int b = item_id / p.H, h = item_id - b * p.H;
          const uint32_t sq = base + stage * stage_bytes;
          const uint32_t sk = sq + 2u * kQTile;
          const uint32_t sv = sk + kv_bytes;
          mbar_wait(qk_empty(stage), phase ^ 1u);
          mbar_arrive_expect_tx(qk_full(stage), q_tiles * kQTile + kv_bytes);
          for (int t = 0; t < q_tiles; ++t)
            tma_load_3d(sq + t * kQTile, &tm_q, qk_full(stage), h * 64, t * 128, b);
          tma_load_3d(sk, &tm_kv, qk_full(stage), D + h * 64, 0, b);
          mbar_wait(v_empty(stage), phase ^ 1u);
          mbar_arrive_expect_tx(v_full(stage), kv_bytes);
          tma_load_3d(sv, &tm_kv, v_full(stage), 2 * D + h * 64, 0, b);
        }
      }
    } else if (warp == 1) {
      // ================= MMA issuer (whole warp converged, one elected lane issues) =============
      const uint32_t idesc_s = make_idesc_bf16(128, Nk);
      const uint32_t idesc_pv = make_idesc_bf16(128, 64, 0, 1);  // B (= V) is MN-major
      auto issue_scores = [&](int stage, int t) {
        const uint32_t sq = base + stage * stage_bytes + t * kQTile;
        const uint32_t sk = base + stage * stage_bytes + 2u * kQTile;
        const uint64_t q_desc = make_desc_sw128(sq, 16, 1024);
        const uint64_t k_desc = make_desc_sw128(sk, 16, 1024);
        const uint32_t d_s = tmem_base + static_cast<uint32_t>(t) * kRegion;
        if (elect_one_sync()) {
#pragma unroll
          for (int k = 0; k < 4; ++k)
            mma_bf16_ss(d_s, q_desc + 2u * k, k_desc + 2u * k, idesc_s, k > 0 ? 1u : 0u);
          mma_commit(s_full(t));
          if (t == q_tiles - 1) mma_commit(qk_empty(stage));  // last reader of this stage's Q and K
        }
        __syncwarp();
      };
      int it = 0;
      uint32_t oc = 0;  // O tiles produced so far
      if (static_cast<int>(blockIdx.x) < num_items) {
        mbar_wait(qk_full(0), 0);
        tc_fence_after();
        for (int t = 0; t < q_tiles; ++t) issue_scores(0, t);
      }
      for (int item = blockIdx.x; item < num_items; item += gridDim.x, ++it) {
        const int stage = it & 1;
        const uint32_t ph = it & 1;
        const bool has_next = item + static_cast<int>(gridDim.x) < num_items;
        const uint32_t sv = base + stage * stage_bytes + 2u * kQTile + kv_bytes;
        // V: rows = keys (128 B each, 8-row swizzle atoms 1024 B apart); 16 keys per MMA
        const uint64_t v_desc = make_desc_sw128(sv, kv_bytes, 1024);
        for (int t = 0; t < q_tiles; ++t) {
          if (t == 0) mbar_wait(v_full(stage), (it >> 1) & 1);
          mbar_wait(p_full(t), ph);
          TR(0, it, t * 4 + 0);
          mbar_wait(o_free, (oc & 1u) ^ 1u);  // the previous O tile has been read out
          TR(0, it, t * 4 + 1);
          tc_fence_after();
          const uint32_t region = tmem_base + static_cast<uint32_t>(t) * kRegion;
          if (elect_one_sync()) {
            // P of a column quarter starts at the quarter's own first S column.  Fully unrolled and
            // predicated (a quarter holds at most 4 MMA steps): the issuing warp shares its
            // scheduler with five busy warps, so every instruction of a rolled loop costs several
            // issue slots of latency - unrolled, an MMA is two instructions instead of eight.
#pragma unroll
            for (int cq = 0; cq < 4; ++cq) {
              const int kb = quarter_begin(cq);
              const int nsteps = (quarter_begin(cq + 1) - kb) >> 4;
#pragma unroll
              for (int i = 0; i < 4; ++i)
                if (i < nsteps)
                  mma_bf16_ts(tmem_base + kOColumn, region + static_cast<uint32_t>(kb + i * 8),
                              v_desc + static_cast<uint64_t>((kb >> 4) + i) * 128u, idesc_pv,
                              (cq > 0 || i > 0) ? 1u : 0u);
            }
            mma_commit(o_full);
            if (t == q_tiles - 1) mma_commit(v_empty(stage));  // last reader of this stage's V
          }
          __syncwarp();
          TR(0, it, t * 4 + 3);
          ++oc;
          if (has_next) {
            if (t == 0) {
              mbar_wait(qk_full(stage ^ 1), ((it + 1) >> 1) & 1);
              tc_fence_after();
            }
            issue_scores(stage ^ 1, t);  // overwrites S_t / P_t behind PV_t (in-order tensor pipe)
          }
          TR(0, it, t * 4 + 2);
        }
      }
    }
  } else if (warp < 20) {
    setmaxnreg_inc<88>();
    // ================= softmax (thread == one column quarter of one query row) ================
    const int cq = (warp - 4) >> 2;  // column quarter
    const int q = warp & 3;          // TMEM lane quarter
    const float c = p.scale * kLog2e;
    const int N = p.N;
    const int kbeg = quarter_begin(cq);
    const int cols = quarter_begin(cq + 1) - kbeg;  // multiple of 16, <= 64
    const int n32 = cols >> 5;
    const bool tail16 = (cols & 16) != 0;
    const uint64_t cc = pack2(__float_as_uint(c), __float_as_uint(c));
    const int bar_id = 1 + q;  // joins the four column quarters of one lane quarter
    int it = 0;
    for (int item = blockIdx.x; item < num_items; item += gridDim.x, ++it) {
      const int par = it & 1;
      const int item_id = p.descending ? num_items - 1 - item : item;
      for (int t = 0; t < q_tiles; ++t) {
        const bool warp_rows = t * 128 + q * 32 < N;
        // pair index of key 0 of this thread's row in the dropout index space
        const uint32_t row_pairs =
            (static_cast<uint32_t>(item_id) * static_cast<uint32_t>(N) +
             static_cast<uint32_t>(t * 128 + q * 32 + lane)) * static_cast<uint32_t>(Nk >> 1);
        const uint32_t region =
            tmem_base + (static_cast<uint32_t>(q * 32) << 16) + static_cast<uint32_t>(t) * kRegion;
        const uint32_t pbase = region + kbeg;  // P of this quarter overwrites its own S columns
        mbar_wait(s_full(t), it & 1);
        if (q == 0 && cq == 0 && lane == 0) TR(1 + t, it, 0);
        tc_fence_after();
        if (warp_rows) {
          uint32_t v32[32];
          uint32_t(&v16)[16] = *reinterpret_cast<uint32_t(*)[16]>(&v32[0]);
          // ---- sweep 1: maximum over this quarter of the row, then across the quarters
          float mx[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
          for (int ch = 0; ch < n32; ++ch) {
            tmem_ld_32x32b_x32(region + kbeg + ch * 32, v32);
            tmem_ld_wait();
            chunk_max<32>(v32, kbeg + ch * 32, N, mx);
          }
          if (tail16) {
            tmem_ld_32x32b_x16(region + kbeg + n32 * 32, v16);
            tmem_ld_wait();
            chunk_max<16>(v16, kbeg + n32 * 32, N, mx);
          }
          const int r = q * 32 + lane;
          m_smem[stat_idx(par, t, cq, r)] = fmaxf(fmaxf(mx[0], mx[1]), fmaxf(mx[2], mx[3]));
          named_bar_sync(bar_id, 128);
          const float m = fmaxf(fmaxf(m_smem[stat_idx(par, t, 0, r)], m_smem[stat_idx(par, t, 1, r)]),
                                fmaxf(m_smem[stat_idx(par, t, 2, r)], m_smem[stat_idx(par, t, 3, r)]));
          // ---- sweep 2: p = 2^((s - m) c), partial row sum, P -> TMEM
          const float nm = -m * c;
          const uint64_t nmc = pack2(__float_as_uint(nm), __float_as_uint(nm));
          uint64_t la = 0ull, lb = 0ull;
          for (int ch = 0; ch < n32; ++ch) {
            tmem_ld_32x32b_x32(region + kbeg + ch * 32, v32);
            tmem_ld_wait();
            exp_chunk_any<32, DROP>(v32, kbeg + ch * 32, N, cc, nmc, pbase + ch * 16, la, lb, p.drop,
                              row_pairs);
          }
          if (tail16) {
            tmem_ld_32x32b_x16(region + kbeg + n32 * 32, v16);
            tmem_ld_wait();
            exp_chunk_any<16, DROP>(v16, kbeg + n32 * 32, N, cc, nmc, pbase + n32 * 16, la, lb, p.drop,
                              row_pairs);
          }
          float l0, l1, l2, l3;
          unpack2(la, l0, l1);
          unpack2(lb, l2, l3);
          l_smem[stat_idx(par, t, cq, r)] = (l0 + l1) + (l2 + l3);
          tmem_st_wait();
        }
        tc_fence_before();
        __syncwarp();
        if (q == 0 && cq == 0 && lane == 0) TR(1 + t, it, 1);
        if (lane == 0) mbar_arrive(p_full(t));
      }
    }
  } else {
    setmaxnreg_dec<72>();
    // ======================= output: O / rowsum -> bf16 -> TMA store =======================
    const int q = warp & 3;
    const int N = p.N;
    const uint32_t o_addr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + kOColumn;
    const uint32_t stg = staging_base + static_cast<uint32_t>(warp - 20) * 8192u;
    uint32_t oc = 0;
    int buf = 0;
    int it = 0;
    if (static_cast<int>(blockIdx.x) < num_items) mbar_wait(p_full(0), 0);
    for (int item = blockIdx.x; item < num_items; item += gridDim.x, ++it) {
      const int item_id = p.descending ? num_items - 1 - item : item;
          const int b = item_id / p.H, h = item_id - b * p.H;
      const bool has_next = item + static_cast<int>(gridDim.x) < num_items;
      const int par = it & 1;
      for (int t = 0; t < q_tiles; ++t) {
        const int row0 = t * 128 + q * 32;
        const bool rows = row0 < N;
        mbar_wait(o_full, oc & 1u);
        ++oc;
        if (q == 0 && lane == 0) TR(3, it, t * 4 + 0);
        tc_fence_after();
        // the row statistics were published before p_full(t), which this warp has already observed
        float l = 1.f, m = 0.f;
        uint32_t pk[32];
        if (rows) {
          const int r = q * 32 + lane;
          l = (l_smem[stat_idx(par, t, 0, r)] + l_smem[stat_idx(par, t, 1, r)]) +
              (l_smem[stat_idx(par, t, 2, r)] + l_smem[stat_idx(par, t, 3, r)]);
          m = fmaxf(fmaxf(m_smem[stat_idx(par, t, 0, r)], m_smem[stat_idx(par, t, 1, r)]),
                    fmaxf(m_smem[stat_idx(par, t, 2, r)], m_smem[stat_idx(par, t, 3, r)]));
          const float inv_l = 1.f / l;
#pragma unroll
          for (int half = 0; half < 2; ++half) {
            uint32_t o[32];
            tmem_ld_32x32b_x32(o_addr + half * 32, o);
            tmem_ld_wait();
#pragma unroll
            for (int j = 0; j < 16; ++j)
              pk[half * 16 + j] = pack_bf16x2(__uint_as_float(o[2 * j]) * inv_l,
                                              __uint_as_float(o[2 * j + 1]) * inv_l);
          }
        }
        // The statistics of the NEXT O tile are observed before this one is released, so p_full
        // can never run two phases ahead of this warp (its producer chain passes through o_free).
        if (t + 1 < q_tiles) mbar_wait(p_full(t + 1), it & 1);
        else if (has_next) mbar_wait(p_full(0), (it + 1) & 1);
        tc_fence_before();
        __syncwarp();
        if (q == 0 && lane == 0) TR(3, it, t * 4 + 1);
        if (lane == 0) mbar_arrive(o_free);
        if (rows) {
#ifndef VITK_ATTN_TRACE
          const int r = row0 + lane;
          if (p.lse != nullptr && r < N)
            p.lse[(static_cast<size_t>(b) * p.H + h) * N + r] = m * p.scale + logf(l);
#endif
          if (lane == 0) tma_store_wait_read<1>();  // the slab used two tiles ago has left smem
          __syncwarp();
          const uint32_t slab = stg + static_cast<uint32_t>(buf) * 4096u;
          const uint32_t row = slab + static_cast<uint32_t>(lane) * 128u;
#pragma unroll
          for (int j = 0; j < 8; ++j)
            st_shared_v4(row + (static_cast<uint32_t>(j ^ (lane & 7)) << 4), pk[4 * j],
                         pk[4 * j + 1], pk[4 * j + 2], pk[4 * j + 3]);
          fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) {
            tma_store_3d(&tm_o, slab, h * 64, row0, b);  // rows >= N are clipped
            tma_store_commit();
          }
          buf ^= 1;
        }
        if (q == 0 && lane == 0) TR(3, it, t * 4 + 2);
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

int attention_fwd_tc2(const void* qkv, void* ctx, float* lse, int B, int N, int H, int hd,
                      cudaStream_t stream, const DropParams* drop) {
  VITK_REQUIRE(qkv && ctx, "attention: null operand");
  VITK_REQUIRE(hd == 64 && N >= 1 && N <= 208, "attention(tc2): needs head_dim 64 and N <= 208");
  VITK_REQUIRE(B > 0 && H > 0, "attention: bad shape B=%d H=%d", B, H);
  VITK_REQUIRE(device_cc() >= 100, "attention(tc2): requires an sm_100 device");
  const int Nk = (N + 15) & ~15;
  const int D = H * 64;
  const size_t smem =
      2 * (2 * static_cast<size_t>(kQTile) + 2 * static_cast<size_t>(Nk) * 128) + 8 * 4096 + 16384 +
      256 + 1024;
  VITK_REQUIRE(smem <= 232448, "attention(tc2): shared memory budget exceeded");
  VITK_TRY(opt_in_smem<attn_fwd_tc2_kernel<false>>(232448, "attn_fwd_tc2_kernel<false>"));
  VITK_TRY(opt_in_smem<attn_fwd_tc2_kernel<true>>(232448, "attn_fwd_tc2_kernel<true>"));
  CUtensorMap tq, tkv, to;
  VITK_TRY(make_row_map(&tq, qkv, B, N, 3 * D, 3 * D, 128));
  VITK_TRY(make_row_map(&tkv, qkv, B, N, 3 * D, 3 * D, Nk));
  VITK_TRY(make_row_map(&to, ctx, B, N, D, D, 32));
  Tc2Params prm;
  prm.B = B;
  prm.N = N;
  prm.H = H;
  prm.Nk = Nk;
  prm.q_tiles = (N + 127) / 128;
  prm.scale = 1.0f / sqrtf(static_cast<float>(hd));
  prm.lse = lse;
  prm.descending = sweep_next();
  if (drop != nullptr) prm.drop = *drop;
  VITK_REQUIRE(prm.drop.thresh == 0u || static_cast<long long>(B) * H * N * Nk < (1ll << 32),
               "attention: dropout index space exceeds 32 bits");
  const int grid = persistent_grid(B * H);
  ProfileScope prof(PROF_ATTN, attention_flops(B, H, N, N, hd), stream);
  if (prm.drop.thresh != 0u)
    attn_fwd_tc2_kernel<true><<<grid, kThreads2, smem, stream>>>(tq, tkv, to, prm);
  else
    attn_fwd_tc2_kernel<false><<<grid, kThreads2, smem, stream>>>(tq, tkv, to, prm);
  VITK_CHECK_LAUNCH("attn_fwd_tc2_kernel");
  return VITK_OK;
}

}  // namespace vitk
