#include "common.h"

#include <cstdarg>
#include <cstring>
#include <atomic>
#include <mutex>
#include <vector>

namespace vitk {

static thread_local char g_err[1024] = "";
static std::atomic<long long> g_launches{0};

int set_error(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}
const char* last_error() { return g_err; }

void count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }
long long launch_count() { return g_launches.load(std::memory_order_relaxed); }

// ---- optional profiling -----------------------------------------------------------------------
struct ProfRec {
  cudaEvent_t start, stop;
  int kind;
  double work;
};
static std::mutex g_prof_mu;
static std::vector<ProfRec> g_prof;
static std::atomic<bool> g_prof_on{false};

bool profile_enabled() { return g_prof_on.load(std::memory_order_relaxed); }
void profile_enable(bool on) { g_prof_on.store(on); }

ProfileScope::ProfileScope(int kind, double work, cudaStream_t stream) : idx_(-1), stream_(stream) {
  if (!profile_enabled()) return;
  ProfRec r;
  r.kind = kind;
  r.work = work;
  if (cudaEventCreate(&r.start) != cudaSuccess || cudaEventCreate(&r.stop) != cudaSuccess) return;
  cudaEventRecord(r.start, stream);
  std::lock_guard<std::mutex> lk(g_prof_mu);
  g_prof.push_back(r);
  idx_ = static_cast<int>(g_prof.size()) - 1;
}
ProfileScope::~ProfileScope() {
  if (idx_ < 0) return;
  std::lock_guard<std::mutex> lk(g_prof_mu);
  cudaEventRecord(g_prof[idx_].stop, stream_);
}

int profile_collect(double* ms, double* work, long long* launches, int nkinds) {
  std::lock_guard<std::mutex> lk(g_prof_mu);
  for (int k = 0; k < nkinds; ++k) ms[k] = work[k] = 0.0, launches[k] = 0;
  for (ProfRec& r : g_prof) {
    float t = 0.f;
    cudaError_t e = cudaEventSynchronize(r.stop);
    if (e == cudaSuccess) e = cudaEventElapsedTime(&t, r.start, r.stop);
    cudaEventDestroy(r.start);
    cudaEventDestroy(r.stop);
    if (e != cudaSuccess) {
      g_prof.clear();
      return set_error(VITK_ERR_CUDA, "profile_collect: %s", cudaGetErrorString(e));
    }
    if (r.kind >= 0 && r.kind < nkinds) {
      ms[r.kind] += t;
      work[r.kind] += r.work;
      launches[r.kind] += 1;
    }
  }
  g_prof.clear();
  return VITK_OK;
}

static std::mutex g_dev_mu;
static int g_sm_count[64];
static int g_cc[64];
static bool g_dev_init[64];

static void init_dev(int dev) {
  std::lock_guard<std::mutex> lk(g_dev_mu);
  if (g_dev_init[dev]) return;
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, dev) == cudaSuccess) {
    g_sm_count[dev] = prop.multiProcessorCount;
    g_cc[dev] = prop.major * 10 + prop.minor;
  }
  g_dev_init[dev] = true;
}
namespace {
thread_local int t_sweep_depth = 0;
thread_local int t_sweep_dir = 0;
}  // namespace
SweepAlternation::SweepAlternation() {
  if (t_sweep_depth++ == 0) t_sweep_dir = 0;
}
SweepAlternation::~SweepAlternation() { --t_sweep_depth; }
int sweep_next() {
  if (t_sweep_depth == 0) return 0;
  const int d = t_sweep_dir;
  t_sweep_dir ^= 1;
  return d;
}

static int g_sm_reserve = 0;
void reserve_sms(int n) { g_sm_reserve = n < 0 ? 0 : n; }
int sm_count() {
  int dev = 0;
  cudaGetDevice(&dev);
  if (!g_dev_init[dev]) init_dev(dev);
  const int n = g_sm_count[dev] - g_sm_reserve;
  return n < 2 ? 2 : n;
}
int device_cc() {
  int dev = 0;
  cudaGetDevice(&dev);
  if (!g_dev_init[dev]) init_dev(dev);
  return g_cc[dev];
}

cudaError_t set_max_dynamic_smem(const void* kernel, int bytes) {
  return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
}
int smem_opt_in_failed(cudaError_t e, const char* kernel_name) {
  return set_error(VITK_ERR_CUDA, "cudaFuncSetAttribute(%s) failed: %s", kernel_name,
                   cudaGetErrorString(e));
}

// cuTensorMapEncodeTiled is a driver entry point; resolve it through the runtime so libvitk does
// not link against libcuda (only stubs exist on the build box).
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*,
                                  const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                  const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn g_encode = nullptr;
static std::once_flag g_encode_once;

static EncodeTiledFn get_encode() {
  std::call_once(g_encode_once, [] {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) ==
            cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      g_encode = reinterpret_cast<EncodeTiledFn>(fn);
  });
  return g_encode;
}

int make_tmap_2d(CUtensorMap* out, const void* base, int elem_bytes, uint64_t inner,
                 uint64_t outer, uint64_t pitch_bytes, uint32_t box_inner, uint32_t box_outer,
                 bool swizzle128) {
  EncodeTiledFn enc = get_encode();
  if (!enc) return set_error(VITK_ERR_CUDA, "cuTensorMapEncodeTiled entry point not available");
  if ((reinterpret_cast<uintptr_t>(base) & 15) != 0 || (pitch_bytes & 15) != 0)
    return set_error(VITK_ERR_INVALID,
                     "TMA operand must be 16-byte aligned (base %p, pitch %llu bytes)", base,
                     (unsigned long long)pitch_bytes);
  if (box_inner * (uint32_t)elem_bytes > 128 && swizzle128)
    return set_error(VITK_ERR_INVALID, "128B-swizzled TMA box inner extent exceeds 128 bytes");
  if (box_outer > 256 || box_inner > 256)
    return set_error(VITK_ERR_INVALID, "TMA box extent exceeds 256");
  CUtensorMapDataType dt;
  switch (elem_bytes) {
    case 2: dt = CU_TENSOR_MAP_DATA_TYPE_BFLOAT16; break;
    case 4: dt = CU_TENSOR_MAP_DATA_TYPE_FLOAT32; break;
    default: return set_error(VITK_ERR_INVALID, "unsupported TMA element size %d", elem_bytes);
  }
  cuuint64_t dims[2] = {inner, outer};
  cuuint64_t strides[1] = {pitch_bytes};
  cuuint32_t box[2] = {box_inner, box_outer};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(out, dt, 2, const_cast<void*>(base), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE,
                   swizzle128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_NONE,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS)
    return set_error(VITK_ERR_CUDA,
                     "cuTensorMapEncodeTiled failed (%d): base %p dims {%llu,%llu} pitch %llu box "
                     "{%u,%u}",
                     (int)r, base, (unsigned long long)inner, (unsigned long long)outer,
                     (unsigned long long)pitch_bytes, box_inner, box_outer);
  return VITK_OK;
}

int make_tmap_3d(CUtensorMap* out, const void* base, int elem_bytes, uint64_t inner, uint64_t rows,
                 uint64_t batch, uint64_t row_pitch_bytes, uint64_t batch_pitch_bytes,
                 uint32_t box_inner, uint32_t box_rows) {
  EncodeTiledFn enc = get_encode();
  if (!enc) return set_error(VITK_ERR_CUDA, "cuTensorMapEncodeTiled entry point not available");
  if ((reinterpret_cast<uintptr_t>(base) & 15) != 0 || (row_pitch_bytes & 15) != 0 ||
      (batch_pitch_bytes & 15) != 0)
    return set_error(VITK_ERR_INVALID, "TMA operand must be 16-byte aligned");
  if (box_inner * (uint32_t)elem_bytes != 128 || box_rows > 256 || box_rows == 0)
    return set_error(VITK_ERR_INVALID, "bad 3-D TMA box {%u,%u}", box_inner, box_rows);
  CUtensorMapDataType dt;
  switch (elem_bytes) {
    case 2: dt = CU_TENSOR_MAP_DATA_TYPE_BFLOAT16; break;
    case 4: dt = CU_TENSOR_MAP_DATA_TYPE_FLOAT32; break;
    default: return set_error(VITK_ERR_INVALID, "unsupported TMA element size %d", elem_bytes);
  }
  cuuint64_t dims[3] = {inner, rows, batch};
  cuuint64_t strides[2] = {row_pitch_bytes, batch_pitch_bytes};
  cuuint32_t box[3] = {box_inner, box_rows, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = enc(out, dt, 3, const_cast<void*>(base), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS)
    return set_error(VITK_ERR_CUDA, "cuTensorMapEncodeTiled(3d) failed (%d)", (int)r);
  return VITK_OK;
}

int make_row_map(CUtensorMap* out, const void* base, int B, int rows, int row_elems, long long pitch,
                 int box_rows, long long img_stride) {
  if (img_stride < 0) img_stride = static_cast<long long>(rows) * pitch;
  return make_tmap_3d(out, base, 2, row_elems, rows, B, static_cast<uint64_t>(pitch) * 2,
                      static_cast<uint64_t>(img_stride) * 2, 64, box_rows);
}

}  // namespace vitk
