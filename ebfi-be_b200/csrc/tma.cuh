// tma.cuh — tiled TMA tensor maps: host-side encoding (cuTensorMapEncodeTiled fetched through the statically linked
// runtime, so libebfi_b200.so does not link libcuda) and the device-side 3-D load.
#pragma once
#include <cuda.h>        // CUtensorMap types only
#include "common.cuh"
#include "umma.cuh"

#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <type_traits>

namespace tma {

// tensor-map element type of an activation type T (float | __nv_bfloat16 | __half)
template <typename T> constexpr CUtensorMapDataType elem_type()
{
    if constexpr (std::is_same_v<T, float>) return CU_TENSOR_MAP_DATA_TYPE_FLOAT32;
    else if constexpr (std::is_same_v<T, __half>) return CU_TENSOR_MAP_DATA_TYPE_FLOAT16;
    else {
        static_assert(std::is_same_v<T, __nv_bfloat16>, "activation type");
        return CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
    }
}

// 3-D tensor of `elem_bytes`-sized elements, dims fastest -> slowest = {d0, d1, d2}, byte strides of d1 and d2
// (multiples of 16); box = the tile one copy moves; out-of-range elements are read as zero. Returns an EBFI_* code.
int encode_3d(CUtensorMap &tm, const void *base, CUtensorMapDataType dtype, const uint64_t (&dims)[3],
              const uint64_t (&strides)[2], const uint32_t (&box)[3]);

#ifdef __CUDACC__
// global -> shared tile copy, completes (with its byte count) on `bar`
__device__ __forceinline__ void load_3d(void *smem_dst, const CUtensorMap *tmap, int c0, int c1, int c2, uint64_t *bar)
{
    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
                 ::"r"(umma::smem_u32(smem_dst)), "l"(tmap), "r"(c0), "r"(c1), "r"(c2), "r"(umma::smem_u32(bar))
                 : "memory");
}
#endif

}  // namespace tma
