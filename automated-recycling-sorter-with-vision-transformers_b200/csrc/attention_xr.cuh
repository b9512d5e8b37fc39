// Device and host helpers shared by the ragged-head_dim separate-source attention kernels
// (attention_xr.cu forward, attention_xr_bwd.cu backward).  A head's columns start at element
// h * hd of a row, so for head_dim 50 its byte offset is only 4-byte aligned (2-byte for an odd
// head_dim).  A TMA box must start 16-byte aligned, so operands arrive by TMA only when hd is a
// multiple of 8 and are staged by thread loads otherwise; results always leave through thread
// stores of exactly hd columns at the widest access the addresses allow.
#pragma once
#include <cuda_bf16.h>

#include "ptx.cuh"

namespace vitk {
namespace xr {

// head_dim padded to the MMA k-step / N granule
__host__ __device__ constexpr int pad16(int v) { return (v + 15) & ~15; }

// Zeroes columns [hd, hdp) of an operand staged by TMA as 64-column 128B-swizzled boxes of
// `box_bytes` each (rows of 128 bytes, 16-byte chunk c of row r stored at chunk c ^ (r & 7)).
// Those columns hold the next head's values; the contraction over the head dimension must not
// see them.  The caller issues fence.proxy.async before the tensor core reads the tile.
__device__ __forceinline__ void zero_pad_cols(uint32_t base, uint32_t box_bytes, int rows, int hd,
                                              int hdp, int t, int nt) {
  const int pad = hdp - hd;
  const unsigned short z = 0;
  for (int i = t; i < rows * pad; i += nt) {
    const int r = i / pad, col = hd + (i - r * pad);
    const uint32_t a = base + static_cast<uint32_t>(col >> 6) * box_bytes +
                       static_cast<uint32_t>(r) * 128u +
                       ((static_cast<uint32_t>((col & 63) >> 3) ^ static_cast<uint32_t>(r & 7)) << 4) +
                       static_cast<uint32_t>(col & 7) * 2u;
    asm volatile("st.shared.u16 [%0], %1;" ::"r"(a), "h"(z) : "memory");
  }
}

// A TMA box must start on a 16-byte boundary of the row, which h * hd is only when hd is a
// multiple of 8.  Otherwise the operands are staged by the threads of a warp: rows [0, rows) x
// columns [0, hdp) of the same swizzled 64-column-box layout a TMA load writes, read from global
// in pieces of the widest width the head's offset allows (8, 4 or 2 bytes), columns >= hd and
// rows >= nvalid written as zeros.  The caller issues fence.proxy.async before the tensor core
// reads the tile.
__device__ __forceinline__ void load_tile(uint32_t base, uint32_t box_bytes,
                                          const __nv_bfloat16* src, long long ld, int rows,
                                          int nvalid, int hd, int hdp, int t, int nt) {
  const int w = (hd % 4 == 0) ? 4 : (hd % 2 == 0) ? 2 : 1;  // elements per piece
  const int upr = hdp / w;                                  // pieces per row
  for (int i = t; i < rows * upr; i += nt) {
    const int r = i / upr, col = (i - r * upr) * w;
    const bool ok = r < nvalid && col < hd;
    const __nv_bfloat16* g = src + r * ld + col;
    const uint32_t a = base + static_cast<uint32_t>(col >> 6) * box_bytes +
                       static_cast<uint32_t>(r) * 128u +
                       ((static_cast<uint32_t>((col & 63) >> 3) ^ static_cast<uint32_t>(r & 7)) << 4) +
                       static_cast<uint32_t>(col & 7) * 2u;
    if (w == 4) {
      const uint2 v = ok ? __ldg(reinterpret_cast<const uint2*>(g)) : make_uint2(0u, 0u);
      asm volatile("st.shared.v2.b32 [%0], {%1, %2};" ::"r"(a), "r"(v.x), "r"(v.y) : "memory");
    } else if (w == 2) {
      const uint32_t v = ok ? __ldg(reinterpret_cast<const unsigned int*>(g)) : 0u;
      asm volatile("st.shared.b32 [%0], %1;" ::"r"(a), "r"(v) : "memory");
    } else {
      const unsigned short v = ok ? __ldg(reinterpret_cast<const unsigned short*>(g)) : 0;
      asm volatile("st.shared.u16 [%0], %1;" ::"r"(a), "h"(v) : "memory");
    }
  }
}

// Columns [c0, c0 + 16) of one output row (c0 a multiple of 16), as bf16, at most up to column
// hd.  vw (1, 2, 4 or 8 elements) divides hd and the row's address and pitch allow accesses of
// 2 * vw bytes (xr::store_width).
__device__ __forceinline__ void store_cols16(__nv_bfloat16* row, int c0, int hd, int vw,
                                             const float (&v)[16]) {
  const int n = hd - c0;
  if (n <= 0) return;
  __nv_bfloat16* dst = row + c0;
  if (vw == 8) {
#pragma unroll
    for (int j = 0; j < 2; ++j)
      if (8 * j < n)
        *reinterpret_cast<uint4*>(dst + 8 * j) =
            make_uint4(ptx::pack_bf16x2(v[8 * j], v[8 * j + 1]), ptx::pack_bf16x2(v[8 * j + 2], v[8 * j + 3]),
                       ptx::pack_bf16x2(v[8 * j + 4], v[8 * j + 5]), ptx::pack_bf16x2(v[8 * j + 6], v[8 * j + 7]));
  } else if (vw == 4) {
#pragma unroll
    for (int j = 0; j < 4; ++j)
      if (4 * j < n)
        *reinterpret_cast<uint2*>(dst + 4 * j) =
            make_uint2(ptx::pack_bf16x2(v[4 * j], v[4 * j + 1]), ptx::pack_bf16x2(v[4 * j + 2], v[4 * j + 3]));
  } else if (vw == 2) {
#pragma unroll
    for (int j = 0; j < 8; ++j)
      if (2 * j < n) *reinterpret_cast<uint32_t*>(dst + 2 * j) = ptx::pack_bf16x2(v[2 * j], v[2 * j + 1]);
  } else {
#pragma unroll
    for (int j = 0; j < 16; ++j)
      if (j < n) dst[j] = __float2bfloat16_rn(v[j]);
  }
}

// Widest store (elements) that keeps every row start h * hd of an output aligned: vw divides
// hd, the pitch, the image stride (ignored for a single image) and the base address.
inline int store_width(const void* p, long long img, int ld, int hd, int B) {
  for (int w = 8; w > 1; w >>= 1)
    if (hd % w == 0 && ld % w == 0 && (B == 1 || img % w == 0) &&
        reinterpret_cast<uintptr_t>(p) % (2u * w) == 0)
      return w;
  return 1;
}

}  // namespace xr
}  // namespace vitk
