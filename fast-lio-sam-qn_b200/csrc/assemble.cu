// assemble.cu -- the steps either side of the registration path (SURVEY.md §8(f), "next" rows), device-resident:
//   k_fetch_closest   LoopClosure::fetchClosestKeyframeIdx           fast_lio_sam_qn/src/loop_closure.cpp:34-56
//   k_assemble        transformPcd per keyframe + sub-map merge       loop_closure.cpp:58-106, utilities.hpp:164-175
//   k_voxel_*         voxelizePcd = pcl::VoxelGrid (centroid of all fields, leaf L)   utilities.hpp:38-63, SURVEY App. B.1
// Keyframe clouds stay on the device from the moment they are added, so a loop-closure attempt moves no point data
// over PCIe: candidate search, cloud assembly, voxel grid, index build and registration all start from HBM.
#include "internal.cuh"
#include "voxel.cuh"

namespace b200 {

int launch_radix_sort(const CloudDev* d_clouds, int count, int max_n, int key_bits, cudaStream_t s);
int radix_sort_result_buf(int key_bits);

// one warp per query keyframe q (treated as the LATEST keyframe: candidates are idx < q)
__global__ void __launch_bounds__(256) k_fetch_closest(const double* pos, const double* stamp, const int* queries, int count, double radius,
                                                        double tdiff_thr, int* out) {
  const int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (w >= count) return;
  const int q = queries[w];
  const double qx = pos[3 * q], qy = pos[3 * q + 1], qz = pos[3 * q + 2], qt = stamp[q];
  double best = radius * 3.0;
  int bi = -1;
  for (int idx = lane; idx < q; idx += 32) {
    const double dx = pos[3 * idx] - qx, dy = pos[3 * idx + 1] - qy, dz = pos[3 * idx + 2] - qz;
    const double dist = sqrt(dx * dx + dy * dy + dz * dz);
    if (radius > dist && tdiff_thr < (qt - stamp[idx]) && dist < best) {  // strictly closer: lowest idx survives ties
      best = dist;
      bi = idx;
    }
  }
  for (int o = 16; o > 0; o >>= 1) {
    const double ob = __shfl_xor_sync(0xffffffffu, best, o);
    const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
    if (oi >= 0 && (bi < 0 || ob < best || (ob == best && oi < bi))) {
      best = ob;
      bi = oi;
    }
  }
  if (lane == 0) out[w] = bi;
}

__global__ void k_assemble_init(const AssembleJob* jobs) {
  const AssembleJob& J = jobs[blockIdx.x];
  if (threadIdx.x < 3) J.bbox[threadIdx.x] = f2ord(INFINITY);
  else if (threadIdx.x < 6) J.bbox[threadIdx.x] = f2ord(-INFINITY);
  if (threadIdx.x == 6) {
    J.counters[0] = 0;  // number of voxels
    J.counters[1] = 0;  // overflow flag
  }
}

// merged[i] = float(pose_corrected * double(p)) with the intensity carried along; also the fp32 bounding box
__global__ void __launch_bounds__(256) k_assemble(const AssembleJob* jobs, const KeyframeDev* kfs, const double* poses) {
  const AssembleJob& J = jobs[blockIdx.y];
  float mn[3] = {INFINITY, INFINITY, INFINITY}, mx[3] = {-INFINITY, -INFINITY, -INFINITY};
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < J.total; i += gridDim.x * blockDim.x) {
    int sgm = 0;
    while (sgm + 1 < J.nseg && i >= J.seg_off[sgm + 1]) sgm++;
    const int kf = J.seg_kf[sgm];
    const float4 p = kfs[kf].pts[i - J.seg_off[sgm]];
    const double* T = poses + 16 * (size_t)kf;
    const double x = p.x, y = p.y, z = p.z;
    float4 o;
    o.x = (float)(T[0] * x + T[1] * y + T[2] * z + T[3]);
    o.y = (float)(T[4] * x + T[5] * y + T[6] * z + T[7]);
    o.z = (float)(T[8] * x + T[9] * y + T[10] * z + T[11]);
    o.w = p.w;
    J.merged[i] = o;
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
  if ((threadIdx.x & 31) == 0 && blockIdx.x * blockDim.x < J.total) {
#pragma unroll
    for (int d = 0; d < 3; d++) {
      atomicMin(&J.bbox[d], f2ord(mn[d]));
      atomicMax(&J.bbox[3 + d], f2ord(mx[d]));
    }
  }
}

// pcl::VoxelGrid first pass: the voxel index of every point (voxel.cuh)
__global__ void __launch_bounds__(256) k_voxel_keys(const AssembleJob* jobs, float inv_leaf) {
  const AssembleJob& J = jobs[blockIdx.y];
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= J.total) return;
  float lo[3], hi[3];
#pragma unroll
  for (int d = 0; d < 3; d++) {
    lo[d] = ord2f(J.bbox[d]);
    hi[d] = ord2f(J.bbox[3 + d]);
  }
  const VoxelGridDev g = voxel_grid(lo, hi, inv_leaf);
  if (voxel_grid_overflows(g)) {
    if (i == 0) J.counters[1] = 1;
    J.sort.keys[0][i] = (uint32_t)i;
    J.sort.vals[0][i] = (uint32_t)i;
    return;
  }
  J.sort.keys[0][i] = voxel_key(J.merged[i], inv_leaf, g);
  J.sort.vals[0][i] = (uint32_t)i;
}

// ordered compaction of the run heads (one block per job); heads[v] = first sorted slot of voxel v
__global__ void __launch_bounds__(1024) k_voxel_heads(const AssembleJob* jobs, int kbuf) {
  const AssembleJob& J = jobs[blockIdx.x];
  __shared__ int wsum[32];
  __shared__ int carry;
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  const uint32_t* keys = J.sort.keys[kbuf];
  for (int base = 0; base < J.total; base += 1024) {
    const int i = base + threadIdx.x;
    const int head = (i < J.total && (i == 0 || keys[i] != keys[i - 1])) ? 1 : 0;
    int incl = head;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int t = __shfl_up_sync(0xffffffffu, incl, o);
      if ((threadIdx.x & 31) >= o) incl += t;
    }
    if ((threadIdx.x & 31) == 31) wsum[threadIdx.x >> 5] = incl;
    __syncthreads();
    if (threadIdx.x < 32) {
      const int w = wsum[threadIdx.x];
      int wi = w;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, wi, o);
        if (threadIdx.x >= o) wi += t;
      }
      wsum[threadIdx.x] = wi - w;
    }
    __syncthreads();
    const int pos = carry + wsum[threadIdx.x >> 5] + incl - head;
    if (head) J.heads[pos] = i;
    __syncthreads();
    if (threadIdx.x == 1023) carry = pos + head;
    __syncthreads();
  }
  if (threadIdx.x == 0) J.counters[0] = carry;
}

// centroid of x, y, z, intensity per voxel: fp32 running sums in sorted (= ascending point index) order
__global__ void __launch_bounds__(256) k_voxel_centroid(const AssembleJob* jobs, int kbuf) {
  const AssembleJob& J = jobs[blockIdx.y];
  const int v = blockIdx.x * blockDim.x + threadIdx.x;
  const int nv = J.counters[0];
  if (v >= nv) return;
  const int a = J.heads[v], b = v + 1 < nv ? J.heads[v + 1] : J.total;
  const uint32_t* vals = J.sort.vals[kbuf];
  float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
  for (int j = a; j < b; j++) {
    const float4 p = J.merged[vals[j]];
    s0 += p.x; s1 += p.y; s2 += p.z; s3 += p.w;
  }
  const float c = (float)(b - a);
  J.out[v] = make_float4(s0 / c, s1 / c, s2 / c, s3 / c);
}

// PosePcd ingest (fast_lio_sam_qn/include/pose_pcd.hpp:37-39): FAST-LIO publishes the scan in the WORLD frame; the keyframe keeps
// it in the LiDAR frame: pcd_ = transformPcd(tmp_pcd, pose_eig_.inverse()) -- double math, float result, intensity carried.
// raw: (x, y, z, intensity) records `stride` floats apart (device copy of the message payload).
__global__ void __launch_bounds__(256) k_ingest_world(const float* raw, int stride, int n, const double* Tinv, float4* out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float* p = raw + (size_t)i * stride;
  const double x = p[0], y = p[1], z = p[2];
  float4 o;
  o.x = (float)(Tinv[0] * x + Tinv[1] * y + Tinv[2] * z + Tinv[3]);
  o.y = (float)(Tinv[4] * x + Tinv[5] * y + Tinv[6] * z + Tinv[7]);
  o.z = (float)(Tinv[8] * x + Tinv[9] * y + Tinv[10] * z + Tinv[11]);
  o.w = stride >= 8 ? p[4] : p[3];  // pcl::PointXYZI keeps the intensity in its second 16-byte lane
  out[i] = o;
}

// strided (x, y, z, ..., intensity at float 3 or, for pcl::PointXYZI's 32-byte records, float 4) -> packed float4
__global__ void __launch_bounds__(256) k_pack_xyzi(const float* raw, int stride, int n, float4* out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float* p = raw + (size_t)i * stride;
  out[i] = make_float4(p[0], p[1], p[2], stride >= 8 ? p[4] : p[3]);
}
void launch_pack_xyzi(const float* d_raw, int stride, int n, float4* d_out, cudaStream_t s) {
  k_pack_xyzi<<<(n + 255) / 256, 256, 0, s>>>(d_raw, stride, n, d_out);
}

void launch_ingest_world(const float* d_raw, int stride, int n, const double* d_Tinv, float4* d_out, cudaStream_t s) {
  k_ingest_world<<<(n + 255) / 256, 256, 0, s>>>(d_raw, stride, n, d_Tinv, d_out);
}

int launch_fetch_closest(const double* d_pos, const double* d_stamp, const int* d_queries, int count, double radius, double tdiff,
                         int* d_out, cudaStream_t s) {
  k_fetch_closest<<<(count * 32 + 255) / 256, 256, 0, s>>>(d_pos, d_stamp, d_queries, count, radius, tdiff, d_out);
  return 1;
}

// d_sort: CloudDev descriptors whose n/keys/vals/hist alias the jobs' sort fields
int launch_assemble_voxelize(const AssembleJob* d_jobs, const CloudDev* d_sort, int count, int max_total, const KeyframeDev* d_kfs,
                             const double* d_poses, float inv_leaf, cudaStream_t s) {
  int l = 0;
  k_assemble_init<<<count, 32, 0, s>>>(d_jobs); l++;
  k_assemble<<<dim3(min((max_total + 255) / 256, 1184), count), 256, 0, s>>>(d_jobs, d_kfs, d_poses); l++;
  k_voxel_keys<<<dim3((max_total + 255) / 256, count), 256, 0, s>>>(d_jobs, inv_leaf); l++;
  l += launch_radix_sort(d_sort, count, max_total, 32, s);  // voxel indices use up to 31 bits: 3 passes of 11 bits
  const int kbuf = radix_sort_result_buf(32);
  k_voxel_heads<<<count, 1024, 0, s>>>(d_jobs, kbuf); l++;
  k_voxel_centroid<<<dim3((max_total + 255) / 256, count), 256, 0, s>>>(d_jobs, kbuf); l++;
  return l;
}

}  // namespace b200
