// Host-side helpers: error reporting and TMA tensor-map construction (driver entry point resolved at
// run time through cudart, so the library has no link-time dependency on libcuda).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace rb {

void set_error(const char* fmt, ...);
const char* get_error();

#define RB_CUDA_CHECK(expr)                                                                   \
  do {                                                                                        \
    cudaError_t _e = (expr);                                                                  \
    if (_e != cudaSuccess) {                                                                  \
      rb::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
      return static_cast<int>(_e);                                                            \
    }                                                                                         \
  } while (0)

#define RB_REQUIRE(cond, code, ...)  \
  do {                               \
    if (!(cond)) {                   \
      rb::set_error(__VA_ARGS__);    \
      return (code);                 \
    }                                \
  } while (0)

// 2D row-major tensor [outer][inner] of 2-byte (fp16) or 4-byte (f32) elements, 128-byte swizzle,
// box = box_inner x box_outer elements.  OOB box parts are zero-filled on load and dropped on store.
int make_tmap_2d(CUtensorMap* out, const void* gptr, int elem_bytes, uint64_t inner, uint64_t outer,
                 uint64_t row_stride_bytes, uint32_t box_inner, uint32_t box_outer);

int device_sm_count();
// Sets `kernel`'s maximum dynamic shared memory to `smem` bytes and stores in *pairs the number of its 2-CTA clusters
// (CTA pairs, one CTA per SM) that can be co-resident on the current device; the persistent pair kernels launch at most
// that many.  Returns 0 or the CUDA error of setting the attribute.
int pair_kernel_setup(const void* kernel, int threads, size_t smem, int* pairs);

// Opt-in per-kernel-family timing (CUDA events on the launch stream) and launch counting; used by bench.py to
// compute the live roofline numbers.  Off by default: the hot path then records nothing.
enum ProfFamily { kProfPrep = 0, kProfJointF = 1, kProfLattice = 2, kProfJointG = 3, kProfDh = 4, kProfDw = 5,
                  kProfDb = 6, kProfOther = 7, kProfFamilies = 8 };
struct ProfScope {
  ProfScope(int family, cudaStream_t stream);
  ~ProfScope();
  int family_;
  cudaStream_t stream_;
  cudaEvent_t start_ = nullptr;
  bool on_ = false;
};
int prof_begin();
int prof_end(float* ms, long long* launches);

}  // namespace rb
