#include "host_common.h"

#include <atomic>
#include <mutex>

namespace hn {

char* error_buffer() {
  static thread_local char buf[512] = {0};
  return buf;
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn resolve_encode() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess) {
      fn = reinterpret_cast<EncodeTiledFn>(p);
    }
  });
  return fn;
}

static int make_tmap(CUtensorMap* tm, CUtensorMapDataType dtype, const void* base, int rank, const uint64_t* dims,
                     const uint64_t* strides_bytes, const uint32_t* box, int swizzle_bytes) {
  EncodeTiledFn fn = resolve_encode();
  if (!fn) {
    set_error("cuTensorMapEncodeTiled is not available (no CUDA driver?)");
    return HN_ERR_CUDA;
  }
  cuuint64_t gdim[5];
  cuuint64_t gstr[4];
  cuuint32_t bdim[5];
  cuuint32_t estr[5];
  for (int i = 0; i < rank; ++i) {
    gdim[i] = dims[i];
    bdim[i] = box[i];
    estr[i] = 1;
    if (i > 0) gstr[i - 1] = strides_bytes[i - 1];
  }
  const CUtensorMapSwizzle sw = swizzle_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B
                                : swizzle_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B
                                : swizzle_bytes == 32 ? CU_TENSOR_MAP_SWIZZLE_32B
                                                      : CU_TENSOR_MAP_SWIZZLE_NONE;
  CUresult r = fn(tm, dtype, static_cast<cuuint32_t>(rank), const_cast<void*>(base), gdim,
                  gstr, bdim, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed with CUresult %d (rank %d, dims %llu %llu box %u %u swizzle %d)",
              static_cast<int>(r), rank, (unsigned long long)dims[0], (unsigned long long)(rank > 1 ? dims[1] : 0),
              box[0], rank > 1 ? box[1] : 0, swizzle_bytes);
    return HN_ERR_CUDA;
  }
  return HN_OK;
}

int make_tmap_16bit(CUtensorMap* tm, const void* base, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                    const uint32_t* box, int swizzle_bytes) {
  // FLOAT16 vs BFLOAT16 only matters for OOB NaN fill, which is not used: tiles are moved as raw 16-bit.
  return make_tmap(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, base, rank, dims, strides_bytes, box, swizzle_bytes);
}

int make_tmap_8bit(CUtensorMap* tm, const void* base, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                   const uint32_t* box, int swizzle_bytes) {
  // raw bytes (e4m3 operand rows): out-of-bounds boxes are zero-filled as for the 16-bit maps
  return make_tmap(tm, CU_TENSOR_MAP_DATA_TYPE_UINT8, base, rank, dims, strides_bytes, box, swizzle_bytes);
}

static std::atomic<long long> g_launch_count{0};
void count_launch(int n) { g_launch_count.fetch_add(n, std::memory_order_relaxed); }
long long launch_count() { return g_launch_count.load(); }

int device_sm_count(int* out) {
  int dev = 0;
  HN_CUDA(cudaGetDevice(&dev));
  HN_CUDA(cudaDeviceGetAttribute(out, cudaDevAttrMultiProcessorCount, dev));
  return HN_OK;
}

}  // namespace hn

extern "C" const char* hn_last_error(void) { return hn::error_buffer(); }
extern "C" int hn_version(void) { return 100; }
extern "C" long long hn_launch_count(void) { return hn::launch_count(); }
