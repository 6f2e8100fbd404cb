// Host helpers shared by the tensor-core GEMM engines and the scorer planners.
#pragma once

#include <cuda.h>
#include <stdint.h>

namespace tfr {

// TMA descriptor of a 2-D row-major tensor [outer][inner] of `dtype` elements with a row
// pitch of `ld_bytes`, box {box_inner, box_outer} elements.  Returns a tfr_status.
int encode_tmap_2d(CUtensorMap* tm, CUtensorMapDataType dtype, const void* ptr, uint64_t inner,
                   uint64_t outer, uint64_t ld_bytes, uint32_t box_inner, uint32_t box_outer,
                   CUtensorMapSwizzle swizzle);

// SM count of the current device, queried once per process.  148 (a B200) when no device
// answers, so that workspace sizes can still be planned on a machine without a GPU.
int num_sms();

}  // namespace tfr
