// Shared helpers for libmovierec_b200 (sm_100a).  Internal header; the public ABI is
// include/movierec_b200.h.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "movierec_b200.h"

namespace mr {

constexpr int kWarp = 32;
constexpr int kB200Sms = 148;  // B200: 2 dies x 74 SMs; grids are sized from the live SM count

// ---- error plumbing (thread-local message, no global mutable state) --------------------------
void set_error(const char* fmt, ...);
int cuda_fail(cudaError_t e, const char* what);

#define MR_REQUIRE(cond, ...)         \
  do {                                \
    if (!(cond)) {                    \
      mr::set_error(__VA_ARGS__);     \
      return MR_ERR_INVALID;          \
    }                                 \
  } while (0)

#define MR_CUDA(call)                                       \
  do {                                                      \
    cudaError_t e__ = (call);                               \
    if (e__ != cudaSuccess) return mr::cuda_fail(e__, #call); \
  } while (0)

#define MR_LAUNCH_CHECK(name)                                  \
  do {                                                         \
    cudaError_t e__ = cudaGetLastError();                      \
    if (e__ != cudaSuccess) return mr::cuda_fail(e__, name);   \
    mr::count_launch();                                        \
  } while (0)

// Opt-in, thread-local profiling (mr_profile_begin / mr_profile_end): CUDA events recorded on the
// caller's stream at phase boundaries, and a count of this library's kernel launches.
void count_launch();
void prof_mark(int phase, cudaStream_t st);  // phase < 0 closes the current interval

int sm_count();  // cached per thread; <0 on error

inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// Bump allocator over the caller's workspace (256-byte aligned slices).
struct Carver {
  char* base;
  size_t off;
  explicit Carver(void* p) : base(static_cast<char*>(p)), off(0) {}
  template <typename T>
  T* take(size_t count) {
    T* p = reinterpret_cast<T*>(base + off);
    off += align_up(count * sizeof(T), 256);
    return p;
  }
};

// ---- device helpers --------------------------------------------------------------------------
#ifdef __CUDACC__

__device__ __forceinline__ float4 ldg4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }

// Streaming 128-bit load that does not allocate in L1 (rows that are read once per tile).
__device__ __forceinline__ float4 ld_stream4(const float* p) {
  float4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0, %1, %2, %3}, [%4];"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
               : "l"(p));
  return r;
}

// One element of the dense optimizer sweeps (legacy-Keras Adam, SGD, the l2 gradient term) with every rounding
// spelled out.  Left to itself the compiler contracts a * b + c into FMAs differently in each loop, so the vector and
// scalar paths of the flat sweep and the data-parallel exchange kernel used to differ in the last bit; with these
// they compute the same bits for the same inputs.
__device__ __forceinline__ void adam_step(float& p, float g, float& m, float& v, float lr_t, float b1, float b2,
                                          float eps) {
  m = __fmaf_rn(b1, m, __fmul_rn(1.f - b1, g));
  v = __fmaf_rn(b2, v, __fmul_rn(__fmul_rn(1.f - b2, g), g));
  p = __fsub_rn(p, __fdiv_rn(__fmul_rn(lr_t, m), __fadd_rn(__fsqrt_rn(v), eps)));
}
__device__ __forceinline__ float sgd_step(float p, float g, float lr) { return __fmaf_rn(-lr, g, p); }
__device__ __forceinline__ float plus_l2(float g, float p, float c2) { return __fmaf_rn(c2, p, g); }  // g + 2 l2 p

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

__device__ __forceinline__ int warp_sum_int(int v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Logistic and the logits form of binary cross-entropy (SURVEY App. A-3):
// bce = max(z,0) - z*y + log1p(exp(-|z|)).
__device__ __forceinline__ float sigmoidf_stable(float z) {
  if (z >= 0.f) return 1.f / (1.f + expf(-z));
  float e = expf(z);
  return e / (1.f + e);
}
__device__ __forceinline__ float bce_logits(float z, float y) {
  return fmaxf(z, 0.f) - z * y + log1pf(expf(-fabsf(z)));
}

// Order key for ranking: NaN ranks last (SURVEY App. A-7).
__device__ __forceinline__ float rank_key(float s) { return isnan(s) ? -INFINITY : s; }

#endif  // __CUDACC__

// ---- kernels' host launchers (one per .cu) ----------------------------------------------------
struct TrainPlan;  // neumf_train.cu

}  // namespace mr
