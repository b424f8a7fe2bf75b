// common.cuh -- shared host/device helpers for librpcc_b200 (sm_100a).
//
// Arithmetic contract: every translation unit is compiled with -fmad=false, IEEE division and
// square root, no flush-to-zero, so a float expression here rounds exactly like the reference's
// baseline-x86-64 C++ (no FMA).  The two places where the reference's own CUDA kernels fuse
// (FPS distance, chamfer distance) call __fmaf_rn explicitly.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/rpcc_b200.h"

namespace rpcc {

void set_error(const char* fmt, ...);
void count_launch(int n = 1);
int check_cuda(cudaError_t e, const char* what);

inline cudaStream_t as_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }

#define RPCC_CUDA(call)                                              \
  do {                                                               \
    int _rc = ::rpcc::check_cuda((call), #call);                     \
    if (_rc != RPCC_OK) return _rc;                                  \
  } while (0)

#define RPCC_LAUNCH_CHECK(name)                                      \
  do {                                                               \
    ::rpcc::count_launch();                                          \
    int _rc = ::rpcc::check_cuda(cudaGetLastError(), name);          \
    if (_rc != RPCC_OK) return _rc;                                  \
  } while (0)

#define RPCC_REQUIRE(cond, msg)                                      \
  do {                                                               \
    if (!(cond)) {                                                   \
      ::rpcc::set_error("%s: %s", __func__, msg);                    \
      return RPCC_ERR_ARG;                                           \
    }                                                                \
  } while (0)

int sm_count();
int scratch_pool(cudaMemPool_t* out);   // library-owned stream-ordered pool of the current device

// streaming (read-once) loads / L2-coherent loads
__device__ __forceinline__ float4 ld_stream_f4(const float4* p) {
  float4 v;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
  return v;
}
__device__ __forceinline__ float ld_stream_f(const float* p) {
  float v;
  asm volatile("ld.global.nc.L1::no_allocate.f32 %0, [%1];" : "=f"(v) : "l"(p));
  return v;
}

// torch (2.11, CUDA) float32 reduction of a size-3 innermost dimension: two lanes per output,
// lane 0 accumulates elements 0 and 2, lane 1 element 1, then lane0 + lane1
// (ATen/native/cuda/Reduce.cuh; pinned on the GPU box by tests/test_torch_semantics.py).
__host__ __device__ __forceinline__ float torch_sum3(float t0, float t1, float t2) {
  return (t0 + t2) + t1;
}

__device__ __forceinline__ unsigned lanemask_lt() {
  unsigned m;
  asm("mov.u32 %0, %%lanemask_lt;" : "=r"(m));
  return m;
}

}  // namespace rpcc
