// voxel.cuh -- the one definition of pcl::VoxelGrid's voxel index (utilities.hpp:38-63, SURVEY App. B.1), shared by the
// sub-map voxel grid (assemble.cu: k_voxel_keys) and the global map (map.cu: k_map_keys).  Both translation units are
// compiled -fmad=false, like the oracle (orc_voxelize), so the keys are the same bits everywhere.
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include "internal.cuh"

namespace b200 {

// grid of the fp32 bounding box [lo, hi] at 1/L = inv_leaf
__device__ __forceinline__ VoxelGridDev voxel_grid(const float lo[3], const float hi[3], float inv_leaf) {
  VoxelGridDev g;
  g.cells = 1;
#pragma unroll
  for (int d = 0; d < 3; d++) {
    g.min_b[d] = (int)floorf(lo[d] * inv_leaf);
    g.div_b[d] = (int)floorf(hi[d] * inv_leaf) - g.min_b[d] + 1;
    g.cells *= (long long)((hi[d] - lo[d]) * inv_leaf) + 1;
  }
  return g;
}

// PCL: "Leaf size is too small ... Integer indices would overflow" -> the input is returned as it is
__device__ __forceinline__ bool voxel_grid_overflows(const VoxelGridDev& g) { return g.cells > 2147483647LL; }

// idx = ijk0 + ijk1*dx + ijk2*dx*dy with ijk = floor(p * (1/L)) - float(min_b)
__device__ __forceinline__ uint32_t voxel_key(const float4& p, float inv_leaf, const VoxelGridDev& g) {
  const int i0 = (int)(floorf(p.x * inv_leaf) - (float)g.min_b[0]);
  const int i1 = (int)(floorf(p.y * inv_leaf) - (float)g.min_b[1]);
  const int i2 = (int)(floorf(p.z * inv_leaf) - (float)g.min_b[2]);
  return (uint32_t)(i0 + i1 * g.div_b[0] + i2 * g.div_b[0] * g.div_b[1]);
}

}  // namespace b200
