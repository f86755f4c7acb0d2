// common.cuh — shared helpers for libnib.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>
#include "../../include/nib.h"

namespace nib {

void set_error(const char* fmt, ...);
int check_device();  // NIB_OK or NIB_ENODEVICE (cached)

#define NIB_CUDA(expr)                                                                 \
  do {                                                                                 \
    cudaError_t _e = (expr);                                                           \
    if (_e != cudaSuccess) {                                                           \
      nib::set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e)); \
      return _e == cudaErrorMemoryAllocation ? NIB_ENOMEM : NIB_ECUDA;                 \
    }                                                                                  \
  } while (0)

#define NIB_REQUIRE(cond, ...)                                                         \
  do {                                                                                 \
    if (!(cond)) {                                                                     \
      nib::set_error(__VA_ARGS__);                                                     \
      return NIB_EINVAL;                                                               \
    }                                                                                  \
  } while (0)

#define NIB_DEVICE_OR_FAIL()                                                           \
  do {                                                                                 \
    int _d = nib::check_device();                                                      \
    if (_d != NIB_OK) return _d;                                                       \
  } while (0)

#define NIB_LAUNCH_CHECK()                                                             \
  do {                                                                                 \
    cudaError_t _e = cudaGetLastError();                                               \
    if (_e != cudaSuccess) {                                                           \
      nib::set_error("%s:%d: kernel launch -> %s", __FILE__, __LINE__, cudaGetErrorString(_e)); \
      return NIB_ECUDA;                                                                \
    }                                                                                  \
  } while (0)

static inline int ceil_div(int a, int b) { return (a + b - 1) / b; }
static inline long long ceil_div_ll(long long a, long long b) { return (a + b - 1) / b; }

// number of SMs of the current device (148 on B200); cached.
int num_sms();

// Per-(use, device, stream) library scratch of at least `bytes` (allocated with max(bytes, min_bytes) when it has to
// grow).  Never shared between streams; see api.cu.
enum ScratchSlot { SCRATCH_GP_DINV = 0, SCRATCH_GP_TRSV, SCRATCH_GP_COLREDUCE, SCRATCH_GP_SCALARS, SCRATCH_HEAT_WSEG,
                   SCRATCH_TIES, SCRATCH_BBOX, SCRATCH_GP_KB };
int stream_scratch(int slot, cudaStream_t st, size_t bytes, size_t min_bytes, void** out);

template <typename T> struct Elem;
template <> struct Elem<float> {
  static __device__ __forceinline__ float ld(const float* p) { return *p; }
  static __device__ __forceinline__ void st(float* p, float v) { *p = v; }
};
template <> struct Elem<__nv_bfloat16> {
  static __device__ __forceinline__ float ld(const __nv_bfloat16* p) { return __bfloat162float(*p); }
  static __device__ __forceinline__ void st(__nv_bfloat16* p, float v) { *p = __float2bfloat16_rn(v); }
};

}  // namespace nib
