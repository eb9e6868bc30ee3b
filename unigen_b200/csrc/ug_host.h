// Host-side helpers shared by the C-ABI translation units: error reporting, launch counting,
// TMA descriptor encoding through the driver entry point (no link-time dependency on libcuda).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <cstdarg>
#include <cstdio>

#include "../../include/unigen_b200.h"

namespace ug {

void set_error(const char* fmt, ...);
void count_launch(int n = 1);
int num_sms();
int current_device_slot();  // cudaGetDevice() clamped to [0, 64): index into per-device caches

// cudaFuncAttributeMaxDynamicSharedMemorySize is a per-device (per-context) attribute: opt in once per device the kernel is
// launched on, not once per process (a process may drive cuda:1 after cuda:0).
template <typename Kernel>
int ensure_dynamic_smem(Kernel kern, int bytes, bool (&done)[64], const char* name) {
  const int dev = current_device_slot();
  if (done[dev]) return UG_OK;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
  if (e != cudaSuccess) {
    set_error("%s: cudaFuncSetAttribute(smem=%d) failed: %s", name, bytes, cudaGetErrorString(e));
    return UG_ERR_CUDA;
  }
  done[dev] = true;
  return UG_OK;
}

// Encode a (up to 4-D) bf16 tiled tensor map with 128-byte swizzle. dims/box innermost-first; strides in
// BYTES for dims 1..rank-1. Returns UG_OK or an error status (message set).
int encode_tmap_bf16(CUtensorMap* map, const void* base, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                     const uint32_t* box);
// Same with any element type (the fp8 GEMM's operands are UINT8 maps: one e4m3 per byte, 128 elements per swizzle row).
int encode_tmap(CUtensorMap* map, CUtensorMapDataType dtype, const void* base, int rank, const uint64_t* dims,
                const uint64_t* strides_bytes, const uint32_t* box);

#define UG_CHECK_ARG(cond, ...)      \
  do {                               \
    if (!(cond)) {                   \
      ug::set_error(__VA_ARGS__);    \
      return UG_ERR_INVALID;         \
    }                                \
  } while (0)

#define UG_CHECK_LAUNCH(name)                                                        \
  do {                                                                               \
    cudaError_t e__ = cudaGetLastError();                                            \
    if (e__ != cudaSuccess) {                                                        \
      ug::set_error("%s: launch failed: %s", name, cudaGetErrorString(e__));         \
      return UG_ERR_CUDA;                                                            \
    }                                                                                \
    ug::count_launch();                                                              \
  } while (0)

}  // namespace ug
