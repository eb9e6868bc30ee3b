#include "ug_host.h"

#include <cstring>
#include <mutex>

namespace ug {

static thread_local char g_err[512] = "";
static thread_local int64_t g_launches = 0;

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
void count_launch(int n) { g_launches += n; }

int current_device_slot() {
  int dev = 0;
  cudaGetDevice(&dev);
  return (dev < 0 || dev >= 64) ? 0 : dev;
}

int num_sms() {
  static int cached[64] = {0};
  const int dev = current_device_slot();
  if (cached[dev] == 0) {
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
    cached[dev] = n;
  }
  return cached[dev];
}

typedef CUresult (*encode_fn_t)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static encode_fn_t get_encode_fn() {
  static encode_fn_t fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres);
    if (e == cudaSuccess && qres == cudaDriverEntryPointSuccess) fn = reinterpret_cast<encode_fn_t>(p);
  });
  return fn;
}

int encode_tmap(CUtensorMap* map, CUtensorMapDataType dtype, const void* base, int rank, const uint64_t* dims,
                const uint64_t* strides_bytes, const uint32_t* box) {
  encode_fn_t fn = get_encode_fn();
  if (!fn) {
    set_error("cuTensorMapEncodeTiled driver entry point not available");
    return UG_ERR_CUDA;
  }
  if ((reinterpret_cast<uintptr_t>(base) & 15) != 0) {
    set_error("TMA base pointer %p is not 16-byte aligned", base);
    return UG_ERR_INVALID;
  }
  cuuint64_t gdims[5];
  cuuint64_t gstrides[4];
  cuuint32_t gbox[5], estr[5];
  for (int i = 0; i < rank; ++i) {
    gdims[i] = dims[i];
    gbox[i] = box[i];
    estr[i] = 1;
    if (i > 0) {
      gstrides[i - 1] = strides_bytes[i - 1];
      if (gstrides[i - 1] % 16 != 0) {
        set_error("TMA stride %llu (dim %d) is not a multiple of 16 bytes", (unsigned long long)gstrides[i - 1], i);
        return UG_ERR_INVALID;
      }
    }
  }
  CUresult r = fn(map, dtype, (cuuint32_t)rank, const_cast<void*>(base), gdims, gstrides,
                  gbox, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                  CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed (CUresult %d): rank %d dims [%llu,%llu,%llu] box [%u,%u,%u]", (int)r, rank,
              (unsigned long long)dims[0], (unsigned long long)(rank > 1 ? dims[1] : 0),
              (unsigned long long)(rank > 2 ? dims[2] : 0), box[0], rank > 1 ? box[1] : 0, rank > 2 ? box[2] : 0);
    return UG_ERR_CUDA;
  }
  return UG_OK;
}

int encode_tmap_bf16(CUtensorMap* map, const void* base, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                     const uint32_t* box) {
  return encode_tmap(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, base, rank, dims, strides_bytes, box);
}

}  // namespace ug

extern "C" {

const char* ug_last_error(void) { return ug::g_err; }
int ug_abi_version(void) { return UG_ABI_VERSION; }
int64_t ug_launch_count(void) { return ug::g_launches; }
void ug_reset_launch_count(void) { ug::g_launches = 0; }

int ug_device_check(void) {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) {
    ug::set_error("no CUDA device: %s", cudaGetErrorString(e));
    return UG_ERR_NO_DEVICE;
  }
  int major = 0, minor = 0;
  cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev);
  cudaDeviceGetAttribute(&minor, cudaDevAttrComputeCapabilityMinor, dev);
  if (major != 10) {
    ug::set_error("device %d is sm_%d%d; libunigen_b200 only carries sm_100a code", dev, major, minor);
    return UG_ERR_NO_DEVICE;
  }
  if (!ug::get_encode_fn()) {
    ug::set_error("cuTensorMapEncodeTiled driver entry point not available");
    return UG_ERR_CUDA;
  }
  return UG_OK;
}

}  // extern "C"
