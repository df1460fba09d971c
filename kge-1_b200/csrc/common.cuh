// Shared device/host helpers for the kgeb200 C-ABI library (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <math.h>
#include "../../include/kgeb200.h"

#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ < 1000)
#error "kgeb200 is written for sm_100a (B200) only"
#endif

namespace kgeb {

// thread-local last error text, returned by kgeb_last_error()
void set_error(const char* fmt, ...);
int cuda_status(cudaError_t e, const char* what);

#define KGEB_REQUIRE(cond, ...)                 \
  do {                                          \
    if (!(cond)) {                              \
      kgeb::set_error(__VA_ARGS__);             \
      return KGEB_ERR_ARG;                      \
    }                                           \
  } while (0)

#define KGEB_LAUNCH_CHECK(what)                                  \
  do {                                                           \
    cudaError_t e__ = cudaGetLastError();                        \
    if (e__ != cudaSuccess) return kgeb::cuda_status(e__, what); \
  } while (0)

__device__ __forceinline__ int64_t load_index(const void* idx, int idx64, int64_t i) {
  if (idx == nullptr) return i;
  return idx64 ? reinterpret_cast<const int64_t*>(idx)[i]
               : static_cast<int64_t>(reinterpret_cast<const int32_t*>(idx)[i]);
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

__device__ __forceinline__ float sgnf(float x) { return (x > 0.f) ? 1.f : ((x < 0.f) ? -1.f : 0.f); }

// Branch-free transcendental forms (MUFU ex2 / lg2 / rcp; ~1e-6 relative error) so that the compiler can keep
// many independent element chains in flight in the tile epilogues:
//   softplus(x) = max(x,0) + log(1 + exp(-|x|)) ;  sigmoid(x) = 1 / (1 + exp(-x))  (exp overflow -> 1/inf = 0)
__device__ __forceinline__ float softplusf(float x) { return fmaxf(x, 0.f) + __logf(1.f + __expf(-fabsf(x))); }
__device__ __forceinline__ float sigmoidf(float x) { return __fdividef(1.f, 1.f + __expf(-x)); }

constexpr int kNumSMs = 148;  // B200

// Adagrad applied by the flush of the dense table-gradient tile kernel (kgeb_fused_bwd_update; tc_bwd.cu)
struct TableUpdate {
  float* w;                 // [n_ent, d] fp32 master rows of the shard
  float* state;             // [n_ent, d] Adagrad sum of squares
  void* mirror;             // [n_ent, d] bf16 mirror (= the tile operand)
  const int32_t* slot_of;   // [n_ent]: >= 0 = row also gets sparse gradient rows this step: parked in gbuf[slot]
  float* gbuf;              // [slots, d]
  const int* skip;          // optional device word: non-zero = abandon the step, touch nothing
  float clr, eps;
  const float* clr_dev;     // optional device word: the rate of this step, read in place of clr (_sched entry)
};

inline cudaStream_t as_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }

}  // namespace kgeb
