// tcgen05 attention for one key block: ctx = softmax(q k^T / sqrt(hd)) v per (image, head) when all
// keys of a head fit one MMA tile (N <= 256 tokens: ViT-B/L at 224 px have 197/198), hd = 64.
// Reference semantics: train.py:543-549 (scale AFTER the product, softmax over keys, no mask).
//
// Persistent CTAs loop over (image, head) items.  Per item:
//   TMA (3-D maps over the packed [B, N, 3D] qkv activation; rows >= N zero-filled):
//       Q tile(s) [128 x 64], K [Nk x 64], V [Nk x 64]  -> 128B-swizzled smem, 2-stage ring
//   MMA  S_t = Q_t K^T        tcgen05.mma, A/B from smem (K-major), D = 128 x Nk fp32 in TMEM
//   softmax warpgroup t (thread == query row): two sweeps over the row in TMEM (max; exp2/sum),
//       P written back to TMEM as packed bf16 over the dead S columns
//   MMA  O_t = P_t V          tcgen05.mma, A from TMEM, B = V from smem (MN-major), D in TMEM
//   epilogue: O_t / rowsum -> bf16 -> swizzled smem slab -> TMA store (3-D map clips rows >= N)
// The [B,H,N,N] score tensor never exists in HBM; q/k/v are read in place from the packed qkv
// buffer (no permute copies) and ctx is written directly in [B, N, H*hd] order.
#include <cuda_bf16.h>

#include "attention_kernels.cuh"
#include "common.h"
#include "ptx.cuh"

namespace vitk {
using namespace ptx;

namespace {

constexpr int kTcThreads = 12 * 32;  // warp 0 TMA, 1 MMA, 2 TMEM alloc, 4-7 / 8-11 softmax groups
constexpr int kQTileBytes = 128 * 128;
constexpr int kRegionCols = 256;  // TMEM columns per q-tile: S [0,Nk) -> P [0,Nk/2), O [128,192)
constexpr int kOCol = 128;

struct TcParams {
  int B, N, H, Nk, q_tiles;
  float scale;
  float* lse;
};

__global__ void __launch_bounds__(kTcThreads, 1)
attn_fwd_tc_kernel(const __grid_constant__ CUtensorMap tm_q, const __grid_constant__ CUtensorMap tm_kv,
                   const __grid_constant__ CUtensorMap tm_o, const TcParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = smem_u32(smem_raw);
  const uint32_t base = (raw_addr + 1023u) & ~1023u;
  uint8_t* smem = smem_raw + (base - raw_addr);

  const int Nk = p.Nk;
  const uint32_t kv_bytes = static_cast<uint32_t>(Nk) * 128u;
  const uint32_t stage_bytes = 2u * kQTileBytes + 2u * kv_bytes;
  const uint32_t staging_base = base + 2u * stage_bytes;  // 8 warps x 4 KB
  const uint32_t bar_base = staging_base + 8u * 4096u;
  auto kv_full = [&](int s) { return bar_base + 8u * s; };
  auto kv_empty = [&](int s) { return bar_base + 8u * (2 + s); };
  auto s_full = [&](int t) { return bar_base + 8u * (4 + t); };
  auto p_full = [&](int t) { return bar_base + 8u * (6 + t); };
  auto o_full = [&](int t) { return bar_base + 8u * (8 + t); };
  auto o_free = [&](int t) { return bar_base + 8u * (10 + t); };
  volatile uint32_t* tmem_slot =
      reinterpret_cast<volatile uint32_t*>(smem + (bar_base - base) + 8 * 12);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int num_items = p.B * p.H;
  const int D = p.H * 64;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tm_q);
    prefetch_tmap(&tm_kv);
    prefetch_tmap(&tm_o);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < 2; ++s) {
      mbar_init(kv_full(s), 1);
      mbar_init(kv_empty(s), 1);
      mbar_init(s_full(s), 1);
      mbar_init(p_full(s), 4);
      mbar_init(o_full(s), 1);
      mbar_init(o_free(s), 4);
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
        const int stage = it & 1;
        const uint32_t phase = (it >> 1) & 1;
        const int b = item / p.H, h = item - b * p.H;
        mbar_wait(kv_empty(stage), phase ^ 1u);
        const uint32_t sq = base + stage * stage_bytes;
        const uint32_t sk = sq + 2u * kQTileBytes;
        const uint32_t sv = sk + kv_bytes;
        mbar_arrive_expect_tx(kv_full(stage), p.q_tiles * kQTileBytes + 2u * kv_bytes);
        for (int t = 0; t < p.q_tiles; ++t)
          tma_load_3d(sq + t * kQTileBytes, &tm_q, kv_full(stage), h * 64, t * 128, b);
        tma_load_3d(sk, &tm_kv, kv_full(stage), D + h * 64, 0, b);
        tma_load_3d(sv, &tm_kv, kv_full(stage), 2 * D + h * 64, 0, b);
      }
    }
  } else if (warp == 1) {
    // ======================= MMA issuer =======================
    if (lane == 0) {
      const uint32_t idesc_s = make_idesc_bf16(128, Nk);
      const uint32_t idesc_pv = make_idesc_bf16(128, 64, 0, 1);  // B (= V) is MN-major
      int it = 0;
      for (int item = blockIdx.x; item < num_items; item += gridDim.x, ++it) {
        const int stage = it & 1;
        const uint32_t kv_phase = (it >> 1) & 1;
        const uint32_t ph = it & 1;
        const uint32_t sq = base + stage * stage_bytes;
        const uint32_t sk = sq + 2u * kQTileBytes;
        const uint32_t sv = sk + kv_bytes;
        mbar_wait(kv_full(stage), kv_phase);
        tc_fence_after();
        const uint64_t k_desc = make_desc_sw128(sk, 16, 1024);
        for (int t = 0; t < p.q_tiles; ++t) {
          mbar_wait(o_free(t), ph ^ 1u);  // previous item's O_t (aliasing S_t) has been read
          tc_fence_after();
          const uint64_t q_desc = make_desc_sw128(sq + t * kQTileBytes, 16, 1024);
          const uint32_t d_s = tmem_base + static_cast<uint32_t>(t * kRegionCols);
#pragma unroll
          for (int k = 0; k < 4; ++k)
            mma_bf16_ss(d_s, q_desc + 2u * k, k_desc + 2u * k, idesc_s, k > 0 ? 1u : 0u);
          mma_commit(s_full(t));
        }
        for (int t = 0; t < p.q_tiles; ++t) {
          mbar_wait(p_full(t), ph);
          tc_fence_after();
          const uint32_t region = tmem_base + static_cast<uint32_t>(t * kRegionCols);
          // V: rows = keys (128 B each, 8-row swizzle atoms 1024 B apart); 16 keys per MMA
          const uint64_t v_desc = make_desc_sw128(sv, kv_bytes, 1024);
          for (int ks = 0; ks < Nk / 16; ++ks)
            mma_bf16_ts(region + kOCol, region + static_cast<uint32_t>(ks * 8),
                        v_desc + static_cast<uint64_t>(ks) * 128u, idesc_pv, ks > 0 ? 1u : 0u);
          mma_commit(o_full(t));
        }
        mma_commit(kv_empty(stage));  // smem stage reusable once every MMA above has retired
      }
    }
  } else if (warp >= 4) {
    // ======================= softmax + output (thread == query row) =======================
    const int t = (warp - 4) >> 2;  // q-tile of this warpgroup
    const int q = warp & 3;         // TMEM lane quarter
    const float c = p.scale * kLog2e;
    const int N = p.N;
    const int row_in_img0 = t * 128 + q * 32;  // first row of this warp
    const bool warp_active = (t < p.q_tiles);
    const bool warp_rows = warp_active && (row_in_img0 < N);
    const uint32_t region = tmem_base + (static_cast<uint32_t>(q * 32) << 16) +
                            static_cast<uint32_t>(t * kRegionCols);
    const uint32_t slab = staging_base + static_cast<uint32_t>(warp - 4) * 4096u;
    const int n32 = Nk >> 5;         // full 32-key chunks
    const bool tail16 = (Nk & 31) != 0;
    int it = 0;
    if (warp_active) {
      for (int item = blockIdx.x; item < num_items; item += gridDim.x, ++it) {
        const uint32_t ph = it & 1;
        const int b = item / p.H, h = item - b * p.H;
        mbar_wait(s_full(t), ph);
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
          const int r = row_in_img0 + lane;
          if (p.lse != nullptr && r < N)
            p.lse[(static_cast<size_t>(b) * p.H + h) * N + r] = m * p.scale + logf(l);
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(p_full(t));

        // ---- O_t = P_t V is ready: normalise, convert, store
        mbar_wait(o_full(t), ph);
        tc_fence_after();
        if (warp_rows) {
          uint32_t o0[32], o1[32];
          tmem_ld_32x32b_x32(region + kOCol, o0);
          tmem_ld_32x32b_x32(region + kOCol + 32, o1);
          tmem_ld_wait();
          uint32_t pk[32];
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            pk[j] = pack_bf16x2(__uint_as_float(o0[2 * j]) * inv_l,
                                __uint_as_float(o0[2 * j + 1]) * inv_l);
            pk[16 + j] = pack_bf16x2(__uint_as_float(o1[2 * j]) * inv_l,
                                     __uint_as_float(o1[2 * j + 1]) * inv_l);
          }
          if (lane == 0) tma_store_wait_read<0>();  // previous item's slab has left smem
          __syncwarp();
          const uint32_t row = slab + static_cast<uint32_t>(lane) * 128u;
#pragma unroll
          for (int j = 0; j < 8; ++j)
            st_shared_v4(row + (static_cast<uint32_t>(j ^ (lane & 7)) << 4), pk[4 * j],
                         pk[4 * j + 1], pk[4 * j + 2], pk[4 * j + 3]);
          fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) {
            tma_store_3d(&tm_o, slab, h * 64, row_in_img0, b);  // rows >= N are clipped
            tma_store_commit();
          }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(o_free(t));
      }
      if (lane == 0) tma_store_wait<0>();
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

}  // namespace

int attention_fwd_tc(const void* qkv, void* ctx, float* lse, int B, int N, int H, int hd,
                     cudaStream_t stream) {
  VITK_REQUIRE(qkv && ctx, "attention: null operand");
  VITK_REQUIRE(hd == 64 && N >= 1 && N <= 256, "attention(tc): needs head_dim 64 and N <= 256");
  VITK_REQUIRE(device_cc() >= 100, "attention(tc): requires an sm_100 device");
  const int Nk = (N + 15) & ~15;
  const int D = H * 64;
  const size_t smem = 2 * (2 * kQTileBytes + 2 * static_cast<size_t>(Nk) * 128) + 8 * 4096 + 256 + 1024;
  VITK_REQUIRE(smem <= 232448, "attention(tc): shared memory budget exceeded");
  VITK_TRY(opt_in_smem<attn_fwd_tc_kernel>(232448, "attn_fwd_tc_kernel"));
  CUtensorMap tq, tkv, to;
  VITK_TRY(make_row_map(&tq, qkv, B, N, 3 * D, 3 * D, 128));
  VITK_TRY(make_row_map(&tkv, qkv, B, N, 3 * D, 3 * D, Nk));
  VITK_TRY(make_row_map(&to, ctx, B, N, D, D, 32));
  TcParams prm;
  prm.B = B;
  prm.N = N;
  prm.H = H;
  prm.Nk = Nk;
  prm.q_tiles = (N + 127) / 128;
  prm.scale = 1.0f / sqrtf(static_cast<float>(hd));
  prm.lse = lse;
  const int grid = persistent_grid(B * H);
  ProfileScope prof(PROF_ATTN, attention_flops(B, H, N, N, hd), stream);
  attn_fwd_tc_kernel<<<grid, kTcThreads, smem, stream>>>(tq, tkv, to, prm);
  VITK_CHECK_LAUNCH("attn_fwd_tc_kernel");
  return VITK_OK;
}

}  // namespace vitk
