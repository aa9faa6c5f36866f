// Host-side helpers shared by the C-ABI translation units: error reporting that
// never throws across the ABI, TMA tensor-map encoding through the driver entry
// point (no link-time dependency on libcuda), launch bookkeeping.
#pragma once

#include <cuda.h>
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/xclip_b200.h"

namespace xclip {

void set_error(const char* fmt, ...);
int fail(int code, const char* fmt, ...);

int num_sms();

// cudaFuncSetAttribute(MaxDynamicSharedMemorySize) once per (device, kernel): the attribute is
// per device, so a process driving several GPUs must set it on each of them
int ensure_dynamic_smem(const void* kernel, int bytes);

// counts kernel launches made by this library (bench.py reports it as gpu_launches)
void count_launch(int n = 1);

// rank-2 bf16 tensor map, SWIZZLE_128B, zero OOB fill.  inner = contiguous dim.
int encode_2d_bf16(CUtensorMap* out, const void* ptr, uint64_t inner, uint64_t outer,
                   uint64_t outer_stride_elems, uint32_t box_inner, uint32_t box_outer);
// rank-3 bf16 tensor map (inner, mid, outer) with strides in elements for mid/outer.
int encode_3d_bf16(CUtensorMap* out, const void* ptr, uint64_t inner, uint64_t mid,
                   uint64_t outer, uint64_t mid_stride_elems, uint64_t outer_stride_elems,
                   uint32_t box_inner, uint32_t box_mid);

}  // namespace xclip

#define XCLIP_REQUIRE(cond, ...)                                          \
  do {                                                                    \
    if (!(cond)) return ::xclip::fail(XCLIP_ERR_INVALID, __VA_ARGS__);    \
  } while (0)

#define XCLIP_CUDA(expr)                                                                \
  do {                                                                                  \
    cudaError_t _e = (expr);                                                            \
    if (_e != cudaSuccess)                                                              \
      return ::xclip::fail(XCLIP_ERR_CUDA, "%s failed: %s (%s:%d)", #expr,             \
                           cudaGetErrorString(_e), __FILE__, __LINE__);                 \
  } while (0)

#define XCLIP_LAUNCH_CHECK(name)                                                        \
  do {                                                                                  \
    cudaError_t _e = cudaGetLastError();                                                \
    if (_e != cudaSuccess)                                                              \
      return ::xclip::fail(XCLIP_ERR_CUDA, "launch of %s failed: %s", name,             \
                           cudaGetErrorString(_e));                                     \
    ::xclip::count_launch();                                                            \
  } while (0)
