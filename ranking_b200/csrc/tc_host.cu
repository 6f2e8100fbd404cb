// Host helpers shared by the tensor-core GEMM engines and the scorer planners (tc_host.h).
#include "common.cuh"
#include "tc_host.h"

namespace tfr {

typedef CUresult (*EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*,
                             const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                             const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                             CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeFn get_encode_fn() {
  static EncodeFn fn = nullptr;
  if (fn) return fn;
  void* p = nullptr;
  cudaDriverEntryPointQueryResult qres;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) !=
          cudaSuccess ||
      qres != cudaDriverEntryPointSuccess)
    return nullptr;
  fn = reinterpret_cast<EncodeFn>(p);
  return fn;
}

int encode_tmap_2d(CUtensorMap* tm, CUtensorMapDataType dtype, const void* ptr, uint64_t inner,
                   uint64_t outer, uint64_t ld_bytes, uint32_t box_inner, uint32_t box_outer,
                   CUtensorMapSwizzle swizzle) {
  EncodeFn fn = get_encode_fn();
  if (!fn) {
    set_error("cuTensorMapEncodeTiled is not available from the CUDA driver");
    return TFR_CUDA_ERROR;
  }
  cuuint64_t dims[2] = {inner, outer};
  cuuint64_t strides[1] = {ld_bytes};
  cuuint32_t box[2] = {box_inner, box_outer};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(tm, dtype, 2, const_cast<void*>(ptr), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed with CUresult %d (ptr %p dtype %d inner %llu outer "
              "%llu ld %llu B box %u x %u)", (int)r, ptr, (int)dtype, (unsigned long long)inner,
              (unsigned long long)outer, (unsigned long long)ld_bytes, box_inner, box_outer);
    return TFR_CUDA_ERROR;
  }
  return TFR_OK;
}

int num_sms() {
  static int n = 0;
  if (n == 0) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess ||
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0)
      n = 148;
  }
  return n;
}

}  // namespace tfr
