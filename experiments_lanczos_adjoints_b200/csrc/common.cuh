// Shared helpers for libb200lanczos (sm_100a only).
#pragma once

#include <cuda_runtime.h>

#include <atomic>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <string>

#include "../../include/b200_lanczos.h"

namespace bl {

// ---- error plumbing -----------------------------------------------------------------
void set_error(const std::string& msg);
extern std::atomic<uint64_t> g_launches;

#define BL_CUDA(expr)                                                                   \
  do {                                                                                  \
    cudaError_t _e = (expr);                                                            \
    if (_e != cudaSuccess) {                                                            \
      ::bl::set_error(std::string(#expr) + ": " + cudaGetErrorString(_e));              \
      return BL_ECUDA;                                                                  \
    }                                                                                   \
  } while (0)

#define BL_CHECK(expr)        \
  do {                        \
    int _rc = (expr);         \
    if (_rc != BL_OK) return _rc; \
  } while (0)

#define BL_REQUIRE(cond, msg)                         \
  do {                                                \
    if (!(cond)) {                                    \
      ::bl::set_error(std::string("invalid argument: ") + (msg)); \
      return BL_EINVAL;                               \
    }                                                 \
  } while (0)

// Count a launch and surface launch-time errors.
#define BL_LAUNCHED()                         \
  do {                                        \
    ::bl::g_launches.fetch_add(1, std::memory_order_relaxed); \
    BL_CUDA(cudaGetLastError());              \
  } while (0)

inline cudaStream_t as_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }
inline size_t dtype_size(int dtype) { return dtype == BL_F32 ? 4 : 8; }
inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

int sm_count();

// Optional per-launch event bracket (bl_profile_begin/end).  No-ops unless profiling is on.
bool prof_enabled();
void prof_start(int cls, double bytes, cudaStream_t s);
void prof_stop(cudaStream_t s);
struct ProfScope {
  cudaStream_t s;
  bool on;
  ProfScope(int cls, double bytes, cudaStream_t stream) : s(stream), on(prof_enabled()) {
    if (on) prof_start(cls, bytes, s);
  }
  ~ProfScope() {
    if (on) prof_stop(s);
  }
};

// ---- device-side helpers ----------------------------------------------------------------
template <typename T>
struct Vec;  // 16-byte vector of T
template <>
struct Vec<float> {
  using type = float4;
  static constexpr int N = 4;
};
template <>
struct Vec<double> {
  using type = double2;
  static constexpr int N = 2;
};

__device__ __forceinline__ void vec_unpack(const float4& v, float (&a)[4]) {
  a[0] = v.x; a[1] = v.y; a[2] = v.z; a[3] = v.w;
}
__device__ __forceinline__ void vec_unpack(const double2& v, double (&a)[2]) {
  a[0] = v.x; a[1] = v.y;
}
__device__ __forceinline__ float4 vec_pack(const float (&a)[4]) {
  return make_float4(a[0], a[1], a[2], a[3]);
}
__device__ __forceinline__ double2 vec_pack(const double (&a)[2]) {
  return make_double2(a[0], a[1]);
}

// Streaming 128-bit load that does not allocate in L1 (basis rows are read once per pass).
__device__ __forceinline__ float4 ld_stream(const float4* p) {
  float4 v;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
               : "l"(p));
  return v;
}
__device__ __forceinline__ double2 ld_stream(const double2* p) {
  double2 v;
  asm volatile("ld.global.nc.L1::no_allocate.v2.f64 {%0,%1}, [%2];"
               : "=d"(v.x), "=d"(v.y)
               : "l"(p));
  return v;
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Block-wide sum of one double per thread; result valid in thread 0.  `smem` >= 32 doubles.
__device__ __forceinline__ double block_sum(double v, double* smem) {
  v = warp_sum(v);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  __syncthreads();
  if (lane == 0) smem[warp] = v;
  __syncthreads();
  double r = 0.0;
  if (warp == 0) {
    const int nw = (blockDim.x + 31) >> 5;
    r = lane < nw ? smem[lane] : 0.0;
    r = warp_sum(r);
  }
  return r;
}

// "Last block done" election among `blocks` blocks that share `counter`: returns true in every thread of the
// block that finishes last.  Partials written by all blocks before the call are visible to the elected block.
__device__ __forceinline__ bool last_block_done(unsigned int* counter, unsigned int blocks) {
  __shared__ bool is_last;
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned int prev = atomicAdd(counter, 1u);
    is_last = (prev == blocks - 1);
    if (is_last) *counter = 0u;  // re-arm for the next launch on the same stream
  }
  __syncthreads();
  if (is_last) __threadfence();
  return is_last;
}
// ... among all blocks of the grid
__device__ __forceinline__ bool last_block_done(unsigned int* counter) {
  return last_block_done(counter, gridDim.x * gridDim.y);
}

}  // namespace bl
