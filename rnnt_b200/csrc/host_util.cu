#include "host_util.h"

#include <stdarg.h>
#include <stdio.h>
#include <string.h>

#include <mutex>
#include <vector>

namespace rb {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
const char* get_error() { return g_err; }

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (fn) return fn;
  void* p = nullptr;
  cudaDriverEntryPointQueryResult qres;
  cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres);
  if (e != cudaSuccess || qres != cudaDriverEntryPointSuccess || p == nullptr) return nullptr;
  fn = reinterpret_cast<EncodeTiledFn>(p);
  return fn;
}

int make_tmap_2d(CUtensorMap* out, const void* gptr, int elem_bytes, uint64_t inner, uint64_t outer,
                 uint64_t row_stride_bytes, uint32_t box_inner, uint32_t box_outer) {
  EncodeTiledFn fn = get_encode_fn();
  RB_REQUIRE(fn != nullptr, -20, "cuTensorMapEncodeTiled entry point not available");
  RB_REQUIRE(elem_bytes == 2 || elem_bytes == 4, -21, "tensor map: unsupported element size %d", elem_bytes);
  RB_REQUIRE((reinterpret_cast<uintptr_t>(gptr) & 15) == 0 && (row_stride_bytes & 15) == 0, -22,
             "tensor map: base %p / row stride %llu must be 16-byte aligned", gptr,
             (unsigned long long)row_stride_bytes);
  RB_REQUIRE(box_inner * elem_bytes == 128 && box_outer <= 256, -23, "tensor map: box %ux%u unsupported",
             box_inner, box_outer);
  cuuint64_t dims[2] = {inner, outer};
  cuuint64_t strides[1] = {row_stride_bytes};
  cuuint32_t box[2] = {box_inner, box_outer};
  cuuint32_t estr[2] = {1, 1};
  CUtensorMapDataType dt = elem_bytes == 2 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32;
  CUresult r = fn(out, dt, 2, const_cast<void*>(gptr), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  RB_REQUIRE(r == CUDA_SUCCESS, -24, "cuTensorMapEncodeTiled failed with CUresult %d (inner %llu outer %llu)",
             (int)r, (unsigned long long)inner, (unsigned long long)outer);
  return 0;
}

int device_sm_count() {
  static int cached[64] = {0};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
  if (cached[dev] == 0) {
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
    cached[dev] = n;
  }
  return cached[dev];
}

int pair_kernel_setup(const void* kernel, int threads, size_t smem, int* pairs) {
  RB_CUDA_CHECK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
  // keyed on (device, kernel); a handful of kernels -> linear scan
  struct Entry { int dev; const void* fn; int pairs; };
  static std::mutex mu;
  static std::vector<Entry> cache;
  int dev = 0;
  const int fallback = device_sm_count() / 2;
  *pairs = fallback;
  if (cudaGetDevice(&dev) != cudaSuccess) return 0;
  {
    std::lock_guard<std::mutex> lk(mu);
    for (const Entry& e : cache)
      if (e.dev == dev && e.fn == kernel) {
        *pairs = e.pairs;
        return 0;
      }
  }
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(2 * fallback);
  cfg.blockDim = dim3(threads);
  cfg.dynamicSmemBytes = smem;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr; cfg.numAttrs = 1;
  int n = 0;
  if (cudaOccupancyMaxActiveClusters(&n, kernel, &cfg) != cudaSuccess || n <= 0) {
    cudaGetLastError();
    n = fallback;
  }
  *pairs = n < fallback ? n : fallback;
  std::lock_guard<std::mutex> lk(mu);
  cache.push_back({dev, kernel, *pairs});
  return 0;
}

namespace {
struct ProfRec { int family; cudaEvent_t start, end; };
std::mutex g_prof_mu;
bool g_prof_on = false;
std::vector<ProfRec> g_prof_recs;
}  // namespace

ProfScope::ProfScope(int family, cudaStream_t stream) : family_(family), stream_(stream) {
  std::lock_guard<std::mutex> lk(g_prof_mu);
  on_ = g_prof_on;
  if (on_) {
    cudaEventCreate(&start_);
    cudaEventRecord(start_, stream_);
  }
}
ProfScope::~ProfScope() {
  if (!on_) return;
  cudaEvent_t end;
  cudaEventCreate(&end);
  cudaEventRecord(end, stream_);
  std::lock_guard<std::mutex> lk(g_prof_mu);
  g_prof_recs.push_back({family_, start_, end});
}
int prof_begin() {
  std::lock_guard<std::mutex> lk(g_prof_mu);
  for (auto& r : g_prof_recs) { cudaEventDestroy(r.start); cudaEventDestroy(r.end); }
  g_prof_recs.clear();
  g_prof_on = true;
  return 0;
}
int prof_end(float* ms, long long* launches) {
  std::lock_guard<std::mutex> lk(g_prof_mu);
  g_prof_on = false;
  for (int i = 0; i < kProfFamilies; ++i) { ms[i] = 0.f; launches[i] = 0; }
  int rc = 0;
  for (auto& r : g_prof_recs) {
    cudaError_t e = cudaEventSynchronize(r.end);
    float t = 0.f;
    if (e == cudaSuccess) e = cudaEventElapsedTime(&t, r.start, r.end);
    if (e != cudaSuccess) { set_error("profile: %s", cudaGetErrorString(e)); rc = static_cast<int>(e); }
    ms[r.family] += t;
    launches[r.family] += 1;
    cudaEventDestroy(r.start);
    cudaEventDestroy(r.end);
  }
  g_prof_recs.clear();
  return rc;
}

}  // namespace rb
