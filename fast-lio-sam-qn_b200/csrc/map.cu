// map.cu -- the corrected global map on the device: transformPcd of every keyframe by its corrected pose, merged in
// keyframe order, then ONE pcl::VoxelGrid over the result (fast_lio_sam_qn.cpp:302-316 /corrected_map, :398-411
// <seq>_map.pcd, :435-449 result.pcd; voxelizePcd = utilities.hpp:38-63).  Compiled -fmad=false like assemble.cu, so the
// points, the keys and the centroids are the bits the FMA-free oracle computes.
//
// The sub-map path (assemble.cu) batches many jobs of <= MAXSEG keyframes and voxelises each with one block; a map is
// one job over the whole store (83 M points for KITTI-05 at 30k points per keyframe), so every phase here is tiled over
// the whole device:
//   k_map_transform   one block per (keyframe, 2048-point tile) from a host-built table; pose in shared memory;
//                     merged float4 records + per-block fp32 min/max partials
//   k_map_grid        one block: partials -> bbox -> VoxelGrid parameters, PCL's int32 guard, key width
//   k_map_keys        voxel index per point (voxel.cuh, the same helper k_voxel_keys uses)
//   radix sort        launch_radix_sort: 3 x 8-bit digits when the grid needs <= 24 bits, else 3 x 11 bits
//   k_map_heads<0>    run heads counted per tile of sorted keys
//   k_map_scan        one block: exclusive scan of the tile counts -> voxel count
//   k_map_heads<1>    run heads scattered to their voxel slot; the records are gathered into sorted order
//   k_map_centroid    one thread per voxel, fp32 running sums in sorted (= ascending merged index) order
#include "internal.cuh"
#include "voxel.cuh"

namespace b200 {

int launch_radix_sort(const CloudDev* d_clouds, int count, int max_n, int key_bits, cudaStream_t s);
int radix_sort_result_buf(int key_bits);

// merged[dst + j] = float(pose * double(p)) with the intensity carried along (the expression of k_assemble)
__global__ void __launch_bounds__(MAP_THREADS) k_map_transform(const MapBlock* blocks, const double* poses, float4* merged,
                                                               float* partials) {
  const MapBlock b = blocks[blockIdx.x];
  __shared__ double T[12];
  __shared__ float red[MAP_THREADS / 32][6];
  if (threadIdx.x < 12) T[threadIdx.x] = poses[16 * (size_t)b.kf + threadIdx.x];
  __syncthreads();
  float mn[3] = {INFINITY, INFINITY, INFINITY}, mx[3] = {-INFINITY, -INFINITY, -INFINITY};
  float4* out = merged + b.dst;
#pragma unroll 4
  for (int j = threadIdx.x; j < b.n; j += MAP_THREADS) {
    const float4 p = b.src[j];
    const double x = p.x, y = p.y, z = p.z;
    float4 o;
    o.x = (float)(T[0] * x + T[1] * y + T[2] * z + T[3]);
    o.y = (float)(T[4] * x + T[5] * y + T[6] * z + T[7]);
    o.z = (float)(T[8] * x + T[9] * y + T[10] * z + T[11]);
    o.w = p.w;
    out[j] = o;
    mn[0] = fminf(mn[0], o.x); mx[0] = fmaxf(mx[0], o.x);
    mn[1] = fminf(mn[1], o.y); mx[1] = fmaxf(mx[1], o.y);
    mn[2] = fminf(mn[2], o.z); mx[2] = fmaxf(mx[2], o.z);
  }
#pragma unroll
  for (int d = 0; d < 3; d++)
    for (int o = 16; o > 0; o >>= 1) {
      mn[d] = fminf(mn[d], __shfl_xor_sync(0xffffffffu, mn[d], o));
      mx[d] = fmaxf(mx[d], __shfl_xor_sync(0xffffffffu, mx[d], o));
    }
  const int w = threadIdx.x >> 5;
  if ((threadIdx.x & 31) == 0) {
#pragma unroll
    for (int d = 0; d < 3; d++) {
      red[w][d] = mn[d];
      red[w][3 + d] = mx[d];
    }
  }
  __syncthreads();
  if (threadIdx.x < 6) {
    float v = red[0][threadIdx.x];
    for (int k = 1; k < MAP_THREADS / 32; k++) v = threadIdx.x < 3 ? fminf(v, red[k][threadIdx.x]) : fmaxf(v, red[k][threadIdx.x]);
    partials[6 * (size_t)blockIdx.x + threadIdx.x] = v;
  }
}

// One block of 1020 threads (170 groups of 6: thread t always reads component t % 6, coalesced over the partials).
__global__ void __launch_bounds__(1024) k_map_grid(const float* partials, int nblocks, float inv_leaf, MapInfo* info) {
  constexpr int G = 170;
  __shared__ float part[6 * G];
  const int t = threadIdx.x, comp = t % 6;
  if (t < 6 * G) {
    float v = comp < 3 ? INFINITY : -INFINITY;
    for (size_t i = t; i < 6 * (size_t)nblocks; i += 6 * G) v = comp < 3 ? fminf(v, partials[i]) : fmaxf(v, partials[i]);
    part[t] = v;
  }
  __syncthreads();
  __shared__ float box[6];
  if (t < 6) {
    float v = part[t];
    for (int k = 1; k < G; k++) v = t < 3 ? fminf(v, part[6 * k + t]) : fmaxf(v, part[6 * k + t]);
    box[t] = v;
  }
  __syncthreads();
  if (t == 0) {
    const VoxelGridDev g = voxel_grid(box, box + 3, inv_leaf);
    MapInfo m;
    m.grid = g;
    m.overflow = voxel_grid_overflows(g) ? 1 : 0;
    // keys lie in [0, div_b0 * div_b1 * div_b2): the width the sort has to cover
    const unsigned long long range = (unsigned long long)g.div_b[0] * (unsigned long long)g.div_b[1] * (unsigned long long)g.div_b[2];
    m.key_bits = range <= 1ull ? 1 : min(32, 64 - __clzll((long long)(range - 1ull)));
    m.voxels = 0;
    m.pad = 0;
    *info = m;
  }
}

__global__ void __launch_bounds__(MAP_THREADS) k_map_keys(const float4* merged, int n, float inv_leaf, const MapInfo* info,
                                                          uint32_t* keys, uint32_t* vals) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  keys[i] = voxel_key(merged[i], inv_leaf, info->grid);
  vals[i] = (uint32_t)i;
}

// Run heads of the sorted keys, per tile of MAP_TILE keys.  Warp w owns [base + w*256, +256): round r, lane l -> key
// r*32 + l, so (warp, round, lane) order is key order and the slots below ascend with the key index.
// SCATTER = false: tile_cnt[tile] = heads in the tile.  SCATTER = true: heads[tile_off[tile] + rank] = i, and the records
// of the tile are gathered into sorted order (the centroid loop then streams them: its loads do not wait on each other).
template <bool SCATTER>
__global__ void __launch_bounds__(MAP_THREADS) k_map_heads(const uint32_t* keys, const uint32_t* vals, const float4* merged, int n,
                                                           int* tile_cnt, const int* tile_off, int* heads, float4* sorted) {
  constexpr int NW = MAP_THREADS / 32, ROUNDS = MAP_TILE / MAP_THREADS;
  __shared__ int wsum[NW];
  const int base = blockIdx.x * MAP_TILE;
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t lt = (1u << lane) - 1u;
  unsigned bal[ROUNDS];
  int wcount = 0;
#pragma unroll
  for (int r = 0; r < ROUNDS; r++) {
    const int i = base + w * (32 * ROUNDS) + r * 32 + lane;
    const bool head = i < n && (i == 0 || keys[i] != keys[i - 1]);
    bal[r] = __ballot_sync(0xffffffffu, head);
    wcount += __popc(bal[r]);
  }
  if (lane == 0) wsum[w] = wcount;
  __syncthreads();
  if (!SCATTER) {
    if (threadIdx.x == 0) {
      int tot = 0;
      for (int k = 0; k < NW; k++) tot += wsum[k];
      tile_cnt[blockIdx.x] = tot;
    }
    return;
  }
  int pos = tile_off[blockIdx.x];
  for (int k = 0; k < w; k++) pos += wsum[k];
#pragma unroll
  for (int r = 0; r < ROUNDS; r++) {
    const int i = base + w * (32 * ROUNDS) + r * 32 + lane;
    if ((bal[r] >> lane) & 1u) heads[pos + __popc(bal[r] & lt)] = i;
    pos += __popc(bal[r]);
  }
#pragma unroll
  for (int r = 0; r < ROUNDS; r++) {
    const int i = base + r * MAP_THREADS + threadIdx.x;
    if (i < n) sorted[i] = merged[vals[i]];
  }
}

// Exclusive scan of the tile counts (one block; each thread scans a contiguous run of tiles); heads[voxels] = n closes the
// last run.
__global__ void __launch_bounds__(1024) k_map_scan(const int* tile_cnt, int ntiles, int n, int* tile_off, int* heads, MapInfo* info) {
  __shared__ int wtot[32];
  const int t = threadIdx.x, lane = t & 31, w = t >> 5;
  const int per = (ntiles + 1023) / 1024, a = min(ntiles, t * per), b = min(ntiles, a + per);
  int run = 0;
  for (int k = a; k < b; k++) run += tile_cnt[k];
  int incl = run;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int v = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += v;
  }
  if (lane == 31) wtot[w] = incl;
  __syncthreads();
  if (w == 0) {
    const int v = wtot[lane];
    int wi = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int u = __shfl_up_sync(0xffffffffu, wi, o);
      if (lane >= o) wi += u;
    }
    wtot[lane] = wi - v;
  }
  __syncthreads();
  int off = wtot[w] + incl - run;
  for (int k = a; k < b; k++) {
    tile_off[k] = off;
    off += tile_cnt[k];
  }
  if (t == 1023) {
    info->voxels = off;
    heads[off] = n;
  }
}

// pcl::VoxelGrid's centroid: fp32 running sums of x, y, z, intensity in sorted order, divided by the count
__global__ void __launch_bounds__(MAP_THREADS) k_map_centroid(const int* heads, const float4* sorted, int nv, float4* out) {
  const int v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= nv) return;
  const int a = heads[v], b = heads[v + 1];
  float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
#pragma unroll 8
  for (int j = a; j < b; j++) {
    const float4 p = sorted[j];
    s0 += p.x; s1 += p.y; s2 += p.z; s3 += p.w;
  }
  const float c = (float)(b - a);
  out[v] = make_float4(s0 / c, s1 / c, s2 / c, s3 / c);
}

// phase 1: merged records, bounding box, grid parameters (info)
int launch_map_transform(const MapBlock* d_blocks, int nblocks, const double* d_poses, float inv_leaf, float4* d_merged,
                         float* d_partials, MapInfo* d_info, cudaStream_t s) {
  k_map_transform<<<nblocks, MAP_THREADS, 0, s>>>(d_blocks, d_poses, d_merged, d_partials);
  k_map_grid<<<1, 1024, 0, s>>>(d_partials, nblocks, inv_leaf, d_info);
  return 2;
}

// phase 2: keys, sort, run heads and the gathered records; d_sort: descriptor whose n/keys/vals/hist are the sort's buffers
// (hist zeroed: radix_sort_ws_bytes(n, key_bits)).  key_bits: 24 or less, or 32.
int launch_map_sort_heads(const float4* d_merged, int n, float inv_leaf, MapInfo* d_info, const CloudDev* d_sort, const CloudDev& sort,
                          int key_bits, int* d_tile_cnt, int* d_tile_off, int* d_heads, float4* d_sorted, cudaStream_t s) {
  int l = 0;
  k_map_keys<<<(n + MAP_THREADS - 1) / MAP_THREADS, MAP_THREADS, 0, s>>>(d_merged, n, inv_leaf, d_info, sort.keys[0], sort.vals[0]); l++;
  l += launch_radix_sort(d_sort, 1, n, key_bits, s);
  const int kb = radix_sort_result_buf(key_bits);
  const int ntiles = (n + MAP_TILE - 1) / MAP_TILE;
  k_map_heads<false><<<ntiles, MAP_THREADS, 0, s>>>(sort.keys[kb], sort.vals[kb], d_merged, n, d_tile_cnt, nullptr, nullptr, nullptr); l++;
  k_map_scan<<<1, 1024, 0, s>>>(d_tile_cnt, ntiles, n, d_tile_off, d_heads, d_info); l++;
  k_map_heads<true><<<ntiles, MAP_THREADS, 0, s>>>(sort.keys[kb], sort.vals[kb], d_merged, n, nullptr, d_tile_off, d_heads, d_sorted); l++;
  return l;
}

// phase 3: one centroid per voxel
int launch_map_centroids(const int* d_heads, const float4* d_sorted, int nv, float4* d_out, cudaStream_t s) {
  k_map_centroid<<<(nv + MAP_THREADS - 1) / MAP_THREADS, MAP_THREADS, 0, s>>>(d_heads, d_sorted, nv, d_out);
  return 1;
}

}  // namespace b200
