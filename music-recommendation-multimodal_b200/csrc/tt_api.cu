// Host-side plumbing shared by every launcher: thread-local error string, the
// TMA tensor-map encoder (driver entry point resolved at run time so the library
// has no link-time dependency on libcuda), device properties.
#include <stdarg.h>
#include <stdio.h>
#include <string.h>

#include "../../include/tt_b200.h"
#include "tt_common.cuh"

namespace tt {

static thread_local char g_err[512] = "";

void set_last_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int cuda_fail(cudaError_t e, const char* what) {
  set_last_error("CUDA error %d (%s) at %s", static_cast<int>(e), cudaGetErrorString(e), what);
  return TT_ERR_CUDA;
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*,
                                  const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                  const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (fn) return fn;
  void* p = nullptr;
  cudaDriverEntryPointQueryResult q;
  cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q);
  if (e != cudaSuccess || q != cudaDriverEntryPointSuccess || p == nullptr) return nullptr;
  fn = reinterpret_cast<EncodeTiledFn>(p);
  return fn;
}

int make_tmap_bf16(CUtensorMap* out, const void* base, int rank, const uint64_t* dims,
                   const uint64_t* strides_bytes, const uint32_t* box) {
  return make_tmap(out, base, rank, dims, strides_bytes, box, /*fp32=*/0, /*swizzle_bytes=*/128);
}

int make_tmap(CUtensorMap* out, const void* base, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
              const uint32_t* box, int fp32, int swizzle_bytes) {
  EncodeTiledFn fn = get_encode_fn();
  if (!fn) {
    set_last_error("cuTensorMapEncodeTiled entry point unavailable (no CUDA driver?)");
    return TT_ERR_CUDA;
  }
  if ((reinterpret_cast<uintptr_t>(base) & 15) != 0) {
    set_last_error("TMA base pointer must be 16-byte aligned");
    return TT_ERR_INVALID;
  }
  cuuint64_t gdim[5];
  cuuint64_t gstr[5];
  cuuint32_t gbox[5];
  cuuint32_t estr[5];
  for (int i = 0; i < rank; ++i) {
    gdim[i] = dims[i];
    gbox[i] = box[i];
    estr[i] = 1;
    if (i > 0) {
      gstr[i - 1] = strides_bytes[i - 1];
      if (gstr[i - 1] % 16 != 0) {
        set_last_error("TMA stride %d (%llu bytes) not a multiple of 16", i,
                       (unsigned long long)gstr[i - 1]);
        return TT_ERR_INVALID;
      }
    }
  }
  const CUtensorMapSwizzle sw = swizzle_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B
                               : swizzle_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B
                               : swizzle_bytes == 32 ? CU_TENSOR_MAP_SWIZZLE_32B : CU_TENSOR_MAP_SWIZZLE_NONE;
  CUresult r = fn(out, fp32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16,
                  static_cast<cuuint32_t>(rank),
                  const_cast<void*>(base), gdim, gstr, gbox, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  sw, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_last_error("cuTensorMapEncodeTiled failed: CUresult %d (rank %d dims %llu,%llu,%llu)",
                   static_cast<int>(r), rank, (unsigned long long)dims[0],
                   (unsigned long long)(rank > 1 ? dims[1] : 0),
                   (unsigned long long)(rank > 2 ? dims[2] : 0));
    return TT_ERR_CUDA;
  }
  return TT_OK;
}

int num_sms() {
  static int n = 0;
  if (n) return n;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return 148;
  int v = 0;
  if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || v <= 0)
    return 148;
  n = v;
  return n;
}

}  // namespace tt

extern "C" {

const char* tt_last_error(void) { return tt::g_err; }

int tt_version(void) { return TT_B200_VERSION; }

int tt_num_sms(void) { return tt::num_sms(); }

}  // extern "C"
