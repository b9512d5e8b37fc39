// Host-side plumbing shared by every translation unit of libvitk: error reporting that never
// throws across the C ABI, launch accounting, device properties, TMA descriptor encoding,
// workspace carving.
#pragma once
#include <cstddef>
#include <cstdint>
#include <cstdio>
#include <cuda.h>
#include <cuda_runtime.h>

#include "../../include/vitk.h"

namespace vitk {

// Error codes are the VITK_* macros of include/vitk.h.

// printf-style; stores into a thread-local buffer, returns `code`.
int set_error(int code, const char* fmt, ...);
const char* last_error();

#define VITK_CHECK_CUDA(expr)                                                              \
  do {                                                                                     \
    cudaError_t _e = (expr);                                                               \
    if (_e != cudaSuccess)                                                                 \
      return ::vitk::set_error(VITK_ERR_CUDA, "%s failed: %s (%s:%d)", #expr,      \
                               cudaGetErrorString(_e), __FILE__, __LINE__);                \
  } while (0)

#define VITK_CHECK_LAUNCH(name)                                                            \
  do {                                                                                     \
    cudaError_t _e = cudaGetLastError();                                                   \
    if (_e != cudaSuccess)                                                                 \
      return ::vitk::set_error(VITK_ERR_CUDA, "launch of %s failed: %s", name,     \
                               cudaGetErrorString(_e));                                    \
    ::vitk::count_launch();                                                                \
  } while (0)

#define VITK_REQUIRE(cond, ...)                                                            \
  do {                                                                                     \
    if (!(cond)) return ::vitk::set_error(VITK_ERR_INVALID, __VA_ARGS__);          \
  } while (0)

#define VITK_TRY(expr)                 \
  do {                                 \
    int _rc = (expr);                  \
    if (_rc != 0) return _rc;          \
  } while (0)

void count_launch();
long long launch_count();

inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// True when p (null counts as aligned) is a multiple of `bytes`: the host-side check in front of
// kernels that move 8- or 16-byte vectors.
inline bool is_aligned(const void* p, uintptr_t bytes) {
  return (reinterpret_cast<uintptr_t>(p) & (bytes - 1)) == 0;
}

// Lays buffers out in a caller-provided workspace, one after the other in the order they are
// taken, each at a 1024-byte aligned offset.  A null base hands out null pointers and only counts
// the bytes (the workspace-size queries).
struct Carver {
  char* base;
  size_t off = 0;
  explicit Carver(void* b) : base(static_cast<char*>(b)) {}
  void* take(size_t n) {
    void* p = base ? base + off : nullptr;
    off += align_up(n, 1024);
    return p;
  }
};

// Optional per-kernel-class timing (bench.py's roofline leg): when enabled, every launcher brackets
// its kernel with CUDA events on the launching stream.  Off by default (zero overhead).
enum ProfKind : int { PROF_GEMM = 0, PROF_ATTN = 1, PROF_LN = 2, PROF_PATCH = 3, PROF_OTHER = 4,
                      PROF_OPT = 5, PROF_NKINDS = 6 };
bool profile_enabled();
void profile_enable(bool on);
// Sums (and clears) the recorded intervals: per kind milliseconds, work units (FLOPs for GEMM and
// attention, bytes for the HBM-bound kernels) and launch counts. Synchronises the recorded events.
int profile_collect(double* ms, double* work, long long* launches, int nkinds);

struct ProfileScope {
  ProfileScope(int kind, double work, cudaStream_t stream);
  ~ProfileScope();
  int idx_;
  cudaStream_t stream_;
};

// Sweep direction of the row-ordered kernels (LayerNorm rows, GEMM row tiles, attention items).
// Inside a SweepAlternation scope consecutive launches alternate between ascending and descending
// order, so every kernel starts on the rows its producer wrote LAST - the part of a 77-310 MB
// intermediate that is still resident in the 126 MB L2.  Outside a scope everything is ascending.
struct SweepAlternation {
  SweepAlternation();
  ~SweepAlternation();
};
int sweep_next();  // direction for the kernel being launched: 0 ascending, 1 descending

// Cached per current device, minus the SMs set aside with reserve_sms (persistent kernels size
// their grids with it: a data-parallel backward leaves a few SMs to the NCCL kernels it overlaps).
int sm_count();
void reserve_sms(int n);
int device_cc();  // e.g. 100
// Grid of a persistent kernel over `items` work items: one CTA per SM, fewer when items run out.
inline int persistent_grid(long long items) {
  const int sms = sm_count();
  return items < sms ? static_cast<int>(items) : sms;
}

// Lets `Kernel` launch with up to `bytes` of dynamic shared memory.  cudaFuncSetAttribute runs on
// the first call for each kernel in the process; later calls report its result.
cudaError_t set_max_dynamic_smem(const void* kernel, int bytes);
int smem_opt_in_failed(cudaError_t e, const char* kernel_name);
template <auto Kernel>
int opt_in_smem(int bytes, const char* kernel_name) {
  static const cudaError_t e = set_max_dynamic_smem(reinterpret_cast<const void*>(Kernel), bytes);
  return e == cudaSuccess ? VITK_OK : smem_opt_in_failed(e, kernel_name);
}

// FLOPs of softmax(q k^T) v over B * H heads (two products of 2 * Nq * Nk * hd each); the
// backward recomputes the scores and forms four more products: 10 instead of 4.
inline double attention_flops(int B, int H, int Nq, int Nk, int hd, bool backward = false) {
  return (backward ? 10.0 : 4.0) * B * H * static_cast<double>(Nq) * Nk * hd;
}

// 2-D bf16 (or any 2-byte / 4-byte element) row-major tensor map: dims {inner, outer},
// row pitch in bytes, box {box_inner, box_outer}, 128-byte swizzle. Cached by value.
int make_tmap_2d(CUtensorMap* out, const void* base, int elem_bytes, uint64_t inner,
                 uint64_t outer, uint64_t pitch_bytes, uint32_t box_inner, uint32_t box_outer,
                 bool swizzle128 = true);

// 3-D variant: dims {inner, rows, batch}, pitches (bytes) of the rows and batch dimensions, box
// {box_inner, box_rows, 1}. Rows beyond `rows` are zero-filled on load and clipped on store, which
// keeps per-image token tiles from touching the neighbouring image.
int make_tmap_3d(CUtensorMap* out, const void* base, int elem_bytes, uint64_t inner, uint64_t rows,
                 uint64_t batch, uint64_t row_pitch_bytes, uint64_t batch_pitch_bytes,
                 uint32_t box_inner, uint32_t box_rows);

// Per-image row map: bf16 [B][rows][row_elems], rows `pitch` elements apart and images
// `img_stride` elements apart (rows * pitch when negative); box of 64 elements (128 bytes,
// swizzled) by `box_rows` rows.
int make_row_map(CUtensorMap* out, const void* base, int B, int rows, int row_elems, long long pitch,
                 int box_rows, long long img_stride = -1);

}  // namespace vitk
