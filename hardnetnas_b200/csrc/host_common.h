// Host-side helpers shared by the C-ABI translation units: error reporting and TMA descriptor
// construction (cuTensorMapEncodeTiled resolved through the runtime, so the library links against
// cudart only and loads on machines without a driver).
#pragma once

#include <cuda.h>
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/hardnet_b200.h"

namespace hn {

char* error_buffer();  // thread-local, 512 bytes

inline void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(error_buffer(), 512, fmt, ap);
  va_end(ap);
}

#define HN_CUDA(expr)                                                                         \
  do {                                                                                        \
    cudaError_t e__ = (expr);                                                                 \
    if (e__ != cudaSuccess) {                                                                 \
      ::hn::set_error("%s:%d %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(e__));  \
      return HN_ERR_CUDA;                                                                     \
    }                                                                                         \
  } while (0)

#define HN_REQUIRE(cond, ...)        \
  do {                               \
    if (!(cond)) {                   \
      ::hn::set_error(__VA_ARGS__);  \
      return HN_ERR_INVALID;         \
    }                                \
  } while (0)

#define HN_TRY(expr)            \
  do {                          \
    int s__ = (expr);           \
    if (s__ != HN_OK) return s__; \
  } while (0)

// 16-bit element tiled tensor map. dims[0] is the contiguous dimension; strides_bytes has rank-1 entries
// (dims 1..rank-1). swizzle_bytes is 32 / 64 / 128 (and must equal box[0] * 2) or 0 for a dense, unswizzled box.
int make_tmap_16bit(CUtensorMap* tm, const void* base, int rank, const uint64_t* dims,
                    const uint64_t* strides_bytes, const uint32_t* box, int swizzle_bytes);
// The same for 1-byte elements (swizzle_bytes = box[0]).
int make_tmap_8bit(CUtensorMap* tm, const void* base, int rank, const uint64_t* dims,
                   const uint64_t* strides_bytes, const uint32_t* box, int swizzle_bytes);

int device_sm_count(int* out);

// cudaFuncAttributeMaxDynamicSharedMemorySize is a per-device setting: remember per kernel instantiation (one static
// DeviceOnce per call site) on which devices it has been raised, so one process may drive several GPUs.
struct DeviceOnce {
  unsigned long long done[2] = {0, 0};   // up to 128 devices
  bool first_time() {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 128) return true;
    const unsigned long long bit = 1ull << (dev & 63);
    if (done[dev >> 6] & bit) return false;
    done[dev >> 6] |= bit;
    return true;
  }
};

// Number of kernels this library has launched (reported by bench.py as gpu_launches).
void count_launch(int n = 1);
long long launch_count();

}  // namespace hn
