// index_build.cu -- batched spatial-index build (replaces the serial nanoflann kd-tree build,
// third_party/nano_gicp/include/nano_gicp/impl/nanoflann_impl.hpp:1199-1211, 867-1012, which the
// reference runs twice per pair plus PCL's hidden third FLANN build, SURVEY.md §3.4).
//
// B200-first design: instead of a serial top-down pointer tree, every cloud becomes a
// Morton-sorted point array with a linear BVH on top (Karras 2012 radix tree, built with one
// thread per node, no recursion).  All clouds of a batch are built together: blockIdx.y is the
// cloud.  Seven launches per batch (round 1 needed eighteen):
//   k_bbox            per-block min/max partials (no atomics, no init kernel)
//   k_morton_ghist    partials -> bbox -> 30-bit Morton keys + the digit histograms of ALL sort passes
//   k_sort_pass x3    stable LSD radix sort, 10 bits per pass, ONE kernel per pass: tile-local ranks, decoupled
//                     look-back across the tiles of a cloud for the global offsets (no separate histogram / scan
//                     kernels), scatter; the last pass writes the sorted float4 points and the rank array directly
//   k_lbvh_topology   Karras radix tree, one thread per node
//   k_lbvh_aabb       bottom-up boxes: the work items (collapsed-leaf roots and lone points, ~1 in 6 candidates) are
//                     compacted inside each block so that climbing warps are fully populated; a child writes its box
//                     and its reference straight into its half of the parent's traversal record
// The sort is stable, so the layout -- and with it every later reduction order -- is deterministic.
// A mid-count split over the same Morton order was measured first and discarded: ranges that
// straddle octant boundaries give huge overlapping boxes (195 node + 71 leaf visits per 15-NN
// query vs 29 + 7 with prefix splits on the 100k KITTI-shaped scan).
#include "internal.cuh"

namespace b200 {

// ------------------------------------------------------------------------------------
// bounding box: per-block partials, reduced again by every block of the next kernel
// ------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_bbox(const CloudDev* clouds) {
  const CloudDev& c = clouds[blockIdx.y];
  float mn[3] = {INFINITY, INFINITY, INFINITY}, mx[3] = {-INFINITY, -INFINITY, -INFINITY};
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < c.n; i += gridDim.x * blockDim.x) {
    const float* p = c.raw + (size_t)i * c.raw_stride;
#pragma unroll
    for (int d = 0; d < 3; d++) {
      float v = p[d];
      mn[d] = fminf(mn[d], v);
      mx[d] = fmaxf(mx[d], v);
    }
  }
#pragma unroll
  for (int d = 0; d < 3; d++)
    for (int o = 16; o > 0; o >>= 1) {
      mn[d] = fminf(mn[d], __shfl_xor_sync(0xffffffffu, mn[d], o));
      mx[d] = fmaxf(mx[d], __shfl_xor_sync(0xffffffffu, mx[d], o));
    }
  __shared__ float red[8][6];
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
    for (int k = 1; k < 8; k++) v = threadIdx.x < 3 ? fminf(v, red[k][threadIdx.x]) : fmaxf(v, red[k][threadIdx.x]);
    c.bbox[6 * blockIdx.x + threadIdx.x] = v;  // partial of block blockIdx.x (empty blocks write +-inf)
  }
}

__device__ __forceinline__ uint32_t expand10(uint32_t v) {
  v &= 0x3FFu;
  v = (v | (v << 16)) & 0x030000FFu;
  v = (v | (v << 8)) & 0x0300F00Fu;
  v = (v | (v << 4)) & 0x030C30C3u;
  v = (v | (v << 2)) & 0x09249249u;
  return v;
}

// ------------------------------------------------------------------------------------
// stable LSD radix sort with one kernel per pass
// ------------------------------------------------------------------------------------
// Work memory of one sort (CloudDev::hist, ZERO-INITIALISED by the caller), in 32-bit words:
//   [0, P*R)                  global digit histograms of the P passes (R = 2^BITS bins)
//   [P*R, P*R + 32)           tile tickets, one per pass
//   [P*R + 32 + p*T*R ...)    look-back words of pass p: T tiles x R digits, (flag << 30) | count
constexpr int SORT_PASSES = 3;
constexpr uint32_t LB_AGG = 1u << 30, LB_INC = 2u << 30, LB_MASK = (1u << 30) - 1u;

__host__ __device__ inline int sort_tiles(int n) { return (n + SORT_TILE - 1) / SORT_TILE; }
template <int BITS>
__host__ __device__ inline size_t sort_ws_words(int n) {
  return (size_t)SORT_PASSES * (1 << BITS) + 32 + (size_t)SORT_PASSES * sort_tiles(n) * (1 << BITS);
}
// Keys of at most 24 bits (the global map's voxel indices, map.cu) take 3 passes of 8 bits: a look-back table of 256
// instead of 2048 words per tile.
constexpr int SORT8_MAX_BITS = 24;
size_t radix_sort_ws_bytes(int n, int key_bits) {
  if (key_bits <= SORT8_MAX_BITS) return 4 * sort_ws_words<8>(n);
  return 4 * (key_bits <= 30 ? sort_ws_words<10>(n) : sort_ws_words<11>(n));
}
int radix_sort_result_buf(int) { return SORT_PASSES & 1; }

// block-wide accumulation of the digit histograms of all passes (shared by the fused Morton kernel and k_sort_ghist)
template <int BITS>
struct GHist {
  static constexpr int R = 1 << BITS;
  uint32_t* h;  // [SORT_PASSES * R] shared memory
  __device__ void clear() {
    for (int j = threadIdx.x; j < SORT_PASSES * R; j += blockDim.x) h[j] = 0;
  }
  __device__ void add(uint32_t key) {
#pragma unroll
    for (int p = 0; p < SORT_PASSES; p++) atomicAdd(&h[p * R + ((key >> (p * BITS)) & (R - 1))], 1u);
  }
  __device__ void flush(uint32_t* ws) {
    for (int j = threadIdx.x; j < SORT_PASSES * R; j += blockDim.x) {
      const uint32_t v = h[j];
      if (v) atomicAdd(&ws[j], v);
    }
  }
};

// bbox partials -> Morton keys (cubic cells) + sort histograms.  Grid: (tiles of SORT_TILE points, cloud).
__global__ void __launch_bounds__(SORT_THREADS) k_morton_ghist(const CloudDev* clouds, int bbox_blocks) {
  const CloudDev& c = clouds[blockIdx.y];
  const int base = blockIdx.x * SORT_TILE;
  if (base >= c.n) return;
  __shared__ uint32_t sh[SORT_PASSES * 1024];
  __shared__ float s_box[6];
  GHist<10> gh{sh};
  gh.clear();
  {  // every block reduces the (few hundred) partials of its cloud again: cheaper than an atomic or a third kernel
    float v = threadIdx.x % 6 < 3 ? INFINITY : -INFINITY;
    const int comp = threadIdx.x % 6, lane6 = threadIdx.x / 6;  // 42 groups of 6 threads
    if (threadIdx.x < 252)
      for (int b = lane6; b < bbox_blocks; b += 42) {
        const float x = c.bbox[6 * b + comp];
        v = comp < 3 ? fminf(v, x) : fmaxf(v, x);
      }
    __shared__ float part[252];
    if (threadIdx.x < 252) part[threadIdx.x] = v;
    __syncthreads();
    if (threadIdx.x < 6) {
      float r = part[threadIdx.x];
      for (int k = 1; k < 42; k++) r = threadIdx.x < 3 ? fminf(r, part[6 * k + threadIdx.x]) : fmaxf(r, part[6 * k + threadIdx.x]);
      s_box[threadIdx.x] = r;
    }
    __syncthreads();
  }
  const float lo0 = s_box[0], lo1 = s_box[1], lo2 = s_box[2];
  const float ext = fmaxf(fmaxf(s_box[3] - lo0, s_box[4] - lo1), s_box[5] - lo2);
  const float scale = ext > 0.f ? 1023.0f / ext : 0.f;  // cubic cells: one scale for all axes
#pragma unroll
  for (int j = 0; j < SORT_ITEMS; j++) {
    const int i = base + j * SORT_THREADS + threadIdx.x;
    if (i < c.n) {
      const float* p = c.raw + (size_t)i * c.raw_stride;
      const uint32_t q0 = (uint32_t)min(max((int)((p[0] - lo0) * scale), 0), 1023);
      const uint32_t q1 = (uint32_t)min(max((int)((p[1] - lo1) * scale), 0), 1023);
      const uint32_t q2 = (uint32_t)min(max((int)((p[2] - lo2) * scale), 0), 1023);
      const uint32_t key = (expand10(q2) << 2) | (expand10(q1) << 1) | expand10(q0);
      c.keys[0][i] = key;
      c.vals[0][i] = (uint32_t)i;
      gh.add(key);
    }
  }
  __syncthreads();
  gh.flush(c.hist);
}

// digit histograms of keys that some other kernel produced (voxel grid, descriptor norm codes)
template <int BITS>
__global__ void __launch_bounds__(SORT_THREADS) k_sort_ghist(const CloudDev* clouds) {
  const CloudDev& c = clouds[blockIdx.y];
  const int base = blockIdx.x * SORT_TILE;
  if (base >= c.n) return;
  extern __shared__ uint32_t sh_dyn[];
  GHist<BITS> gh{sh_dyn};
  gh.clear();
  __syncthreads();
#pragma unroll
  for (int j = 0; j < SORT_ITEMS; j++) {
    const int i = base + j * SORT_THREADS + threadIdx.x;
    if (i < c.n) gh.add(c.keys[0][i]);
  }
  __syncthreads();
  gh.flush(c.hist);
}

// One pass: reads keys/vals[pass & 1], writes [(pass + 1) & 1].  GATHER (last pass of the index build): instead of the
// value array the kernel writes the sorted points (w = original index) and the inverse permutation.
template <int BITS, bool GATHER>
__global__ void __launch_bounds__(SORT_THREADS) k_sort_pass(const CloudDev* clouds, int pass) {
  constexpr int R = 1 << BITS, NW = SORT_THREADS / 32, DPT = R / SORT_THREADS;  // digits per thread
  const CloudDev& c = clouds[blockIdx.y];
  const int ntiles = sort_tiles(c.n);
  if ((int)blockIdx.x >= ntiles) return;
  __shared__ unsigned short cnt[NW][R];  // per-warp digit counts, then exclusive offsets inside the tile (<= SORT_TILE)
  __shared__ uint32_t gbase[R];          // first output slot of (digit, this tile)
  __shared__ uint32_t wtot[NW];
  __shared__ int s_tile;
  uint32_t* ws = c.hist;
  uint32_t* look = ws + SORT_PASSES * R + 32 + (size_t)pass * ntiles * R;
  if (threadIdx.x == 0) s_tile = (int)atomicAdd(&ws[SORT_PASSES * R + pass], 1u);  // tiles start in ticket order: look-back cannot deadlock
  for (int j = threadIdx.x; j < NW * R; j += SORT_THREADS) (&cnt[0][0])[j] = 0;
  __syncthreads();
  const int tile = s_tile;
  const int base = tile * SORT_TILE;
  const uint32_t* keys = c.keys[pass & 1];
  const uint32_t* vals = c.vals[pass & 1];
  uint32_t* okeys = c.keys[(pass + 1) & 1];
  uint32_t* ovals = c.vals[(pass + 1) & 1];
  const int shift = pass * BITS;
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t lt = (1u << lane) - 1u;
  // warp w owns the contiguous run [base + w*32*ITEMS, +32*ITEMS): round r, lane l -> key r*32+l,
  // so (warp, round, lane) order == key order and the ranks below are stable.
  uint32_t key[SORT_ITEMS], val[SORT_ITEMS], rk[SORT_ITEMS];
#pragma unroll
  for (int r = 0; r < SORT_ITEMS; r++) {
    const int i = base + (w * SORT_ITEMS + r) * 32 + lane;
    const bool ok = i < c.n;
    key[r] = ok ? keys[i] : 0xFFFFFFFFu;
    val[r] = ok ? vals[i] : 0u;
    const uint32_t dig = ok ? ((key[r] >> shift) & (R - 1)) : (uint32_t)R;  // R = "invalid"
    const uint32_t m = __match_any_sync(0xffffffffu, dig);
    const uint32_t old = ok ? cnt[w][dig] : 0u;
    __syncwarp();
    if (ok && (m & lt) == 0) cnt[w][dig] = (unsigned short)(old + __popc(m));
    __syncwarp();
    rk[r] = old + __popc(m & lt);
  }
  __syncthreads();
  // exclusive scan of the global histogram of this pass (every block redoes it: R values, a few dozen instructions)
  {
    uint32_t hv[DPT], run = 0;
#pragma unroll
    for (int k = 0; k < DPT; k++) {
      hv[k] = run;
      run += ws[pass * R + threadIdx.x * DPT + k];
    }
    uint32_t incl = run;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += t;
    }
    if (lane == 31) wtot[w] = incl;
    __syncthreads();
    uint32_t woff = 0;
    for (int ww = 0; ww < w; ww++) woff += wtot[ww];
    const uint32_t excl = woff + incl - run;
#pragma unroll
    for (int k = 0; k < DPT; k++) gbase[threadIdx.x * DPT + k] = excl + hv[k];
  }
  __syncthreads();
  // per digit: exclusive prefix over the warps of this tile, publish the tile's count, look back over earlier tiles.
  // A thread owns DPT digits (strided: consecutive threads publish consecutive words) and walks back for all of them
  // TOGETHER: the DPT loads of a step are independent, so a step costs one L2 round trip, not DPT.
  {
    uint32_t run[DPT], excl[DPT];
    bool open_[DPT];
#pragma unroll
    for (int k = 0; k < DPT; k++) {
      const int d = k * SORT_THREADS + threadIdx.x;
      uint32_t r = 0;
#pragma unroll
      for (int ww = 0; ww < NW; ww++) {
        const uint32_t t = cnt[ww][d];
        cnt[ww][d] = (unsigned short)r;
        r += t;
      }
      run[k] = r;
      excl[k] = 0;
      open_[k] = tile > 0;
      *(volatile uint32_t*)(look + (size_t)tile * R + d) = (tile == 0 ? LB_INC : LB_AGG) | r;
    }
    for (int t2 = tile - 1; t2 >= 0; t2--) {
      uint32_t v[DPT];
      bool any_open = false;
#pragma unroll
      for (int k = 0; k < DPT; k++) {
        v[k] = LB_INC;
        if (open_[k]) v[k] = *(volatile uint32_t*)(look + (size_t)t2 * R + k * SORT_THREADS + threadIdx.x);
      }
#pragma unroll
      for (int k = 0; k < DPT; k++) {
        if (!open_[k]) continue;
        while ((v[k] >> 30) == 0u) v[k] = *(volatile uint32_t*)(look + (size_t)t2 * R + k * SORT_THREADS + threadIdx.x);
        excl[k] += v[k] & LB_MASK;
        if ((v[k] >> 30) == 2u) open_[k] = false;
        any_open |= open_[k];
      }
      if (!any_open) break;
    }
#pragma unroll
    for (int k = 0; k < DPT; k++) {
      const int d = k * SORT_THREADS + threadIdx.x;
      if (tile > 0) *(volatile uint32_t*)(look + (size_t)tile * R + d) = LB_INC | (excl[k] + run[k]);
      gbase[d] += excl[k];
    }
  }
  __syncthreads();
#pragma unroll
  for (int r = 0; r < SORT_ITEMS; r++) {
    const int i = base + (w * SORT_ITEMS + r) * 32 + lane;
    if (i < c.n) {
      const uint32_t dig = (key[r] >> shift) & (R - 1);
      const uint32_t dst = gbase[dig] + cnt[w][dig] + rk[r];
      okeys[dst] = key[r];
      if (GATHER) {
        const float* p = c.raw + (size_t)val[r] * c.raw_stride;
        c.pts[dst] = make_float4(p[0], p[1], p[2], __int_as_float((int)val[r]));
        c.rank[val[r]] = (int)dst;
      } else {
        ovals[dst] = val[r];
      }
    }
  }
}

// Stable LSD radix sort of (keys[0], vals[0]) of every descriptor; result in keys/vals[radix_sort_result_buf()].
// Only the n / keys / vals / hist fields of the descriptors are used (also by the voxel grid, assemble.cu, and the
// descriptor ordering, quatro.cu, and the global map, map.cu); hist must point to radix_sort_ws_bytes() ZEROED bytes.
// key_bits <= 24: 3 x 8 bits, <= 30: 3 x 10 bits, otherwise 3 x 11 bits.
int launch_radix_sort(const CloudDev* d_clouds, int count, int max_n, int key_bits, cudaStream_t s) {
  const dim3 grid(sort_tiles(max_n), count);
  if (key_bits <= SORT8_MAX_BITS) {
    k_sort_ghist<8><<<grid, SORT_THREADS, SORT_PASSES * 256 * 4, s>>>(d_clouds);
    for (int p = 0; p < SORT_PASSES; p++) k_sort_pass<8, false><<<grid, SORT_THREADS, 0, s>>>(d_clouds, p);
  } else if (key_bits <= 30) {
    k_sort_ghist<10><<<grid, SORT_THREADS, SORT_PASSES * 1024 * 4, s>>>(d_clouds);
    for (int p = 0; p < SORT_PASSES; p++) k_sort_pass<10, false><<<grid, SORT_THREADS, 0, s>>>(d_clouds, p);
  } else {
    k_sort_ghist<11><<<grid, SORT_THREADS, SORT_PASSES * 2048 * 4, s>>>(d_clouds);
    for (int p = 0; p < SORT_PASSES; p++) k_sort_pass<11, false><<<grid, SORT_THREADS, 0, s>>>(d_clouds, p);
  }
  return 1 + SORT_PASSES;
}

// ---- Karras radix tree over the sorted keys -----------------------------------------
__device__ __forceinline__ int delta(const uint32_t* __restrict__ keys, int n, int i, int j) {
  if (j < 0 || j >= n) return -1;
  uint32_t x = keys[i] ^ keys[j];
  return x ? __clz(x) : 32 + __clz((uint32_t)i ^ (uint32_t)j);  // equal keys: fall back to the index
}

__global__ void __launch_bounds__(256) k_lbvh_topology(const CloudDev* clouds, int kbuf) {
  const CloudDev& c = clouds[blockIdx.y];
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const int n = c.n;
  if (i >= n - 1) return;
  const uint32_t* __restrict__ keys = c.keys[kbuf];
  const int d = (delta(keys, n, i, i + 1) - delta(keys, n, i, i - 1)) >= 0 ? 1 : -1;
  const int dmin = delta(keys, n, i, i - d);
  int lmax = 2;
  while (delta(keys, n, i, i + lmax * d) > dmin) lmax <<= 1;
  int l = 0;
  for (int t = lmax >> 1; t >= 1; t >>= 1)
    if (delta(keys, n, i, i + (l + t) * d) > dmin) l += t;
  const int j = i + l * d;
  const int dnode = delta(keys, n, i, j);
  int s = 0;
  int t = l;
  do {
    t = (t + 1) >> 1;
    if (delta(keys, n, i, i + (s + t) * d) > dnode) s += t;
  } while (t > 1);
  const int gamma = i + s * d + min(d, 0);
  const int first = min(i, j), last = max(i, j);
  const int left_leaf = first == gamma, right_leaf = last == gamma + 1;
  c.info[i] = make_int4(first, last, left_leaf | (right_leaf << 1), gamma);
  if (left_leaf) c.parent_leaf[gamma] = i; else c.parent_node[gamma] = i;
  if (right_leaf) c.parent_leaf[gamma + 1] = i; else c.parent_node[gamma + 1] = i;
}

// Bottom-up AABBs.  Work items: every point whose parent spans > LEAF points (a 1-point leaf) and every internal
// node that is the root of a collapsed leaf (<= LEAF points, parent > LEAF): it reduces its <= 8 points directly.
// Only about one candidate in six is a work item, and a climb is a chain of dependent atomics: the items of a block are
// therefore compacted first (ballot + prefix), so the warps that stay resident for the climb are fully populated.
// An item writes its box and its own reference into ITS half of the parent's traversal record and arrives at the
// parent's flag; the second arrival owns the parent, reads the finished 64-byte record back, merges the two boxes and
// carries on upwards.  (nbox, the separate per-node box array of round 1, is gone.)
__global__ void __launch_bounds__(256) k_lbvh_aabb(const CloudDev* clouds) {
  const CloudDev& c = clouds[blockIdx.y];
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  const int n = c.n;
  if (n <= LEAF || (int)(blockIdx.x * blockDim.x) >= 2 * n - 1) return;
  __shared__ int s_items[256];
  __shared__ int s_wcnt[8];
  bool is_item = false;
  if (t < n) {  // point t
    const int4 pi = c.info[c.parent_leaf[t]];
    is_item = pi.y - pi.x + 1 > LEAF;  // otherwise it lives inside a collapsed leaf
  } else if (t < 2 * n - 1) {  // internal node t - n
    const int i = t - n;
    const int4 inf = c.info[i];
    if (i != 0 && inf.y - inf.x + 1 <= LEAF) {
      const int4 pi = c.info[c.parent_node[i]];
      is_item = pi.y - pi.x + 1 > LEAF;  // otherwise an ancestor is the collapsed-leaf root
    }
  }
  const unsigned bal = __ballot_sync(0xffffffffu, is_item);
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0) s_wcnt[w] = __popc(bal);
  __syncthreads();
  int off = 0, total = 0;
  for (int k = 0; k < 8; k++) {
    if (k < w) off += s_wcnt[k];
    total += s_wcnt[k];
  }
  if (is_item) s_items[off + __popc(bal & ((1u << lane) - 1u))] = t;
  __syncthreads();
  if ((int)threadIdx.x >= total) return;
  const int item = s_items[threadIdx.x];
  // the item's own box, reference and parent
  float4 lo, hi;
  int ref, node, first;
  if (item < n) {
    const float4 q = c.pts[item];
    lo = q;
    hi = q;
    ref = leaf_ref(item, 1);
    node = c.parent_leaf[item];
    first = item;
  } else {
    const int i = item - n;
    const int4 inf = c.info[i];
    float lo0 = INFINITY, lo1 = INFINITY, lo2 = INFINITY, hi0 = -INFINITY, hi1 = -INFINITY, hi2 = -INFINITY;
    for (int p = inf.x; p <= inf.y; p++) {
      const float4 q = c.pts[p];
      lo0 = fminf(lo0, q.x); hi0 = fmaxf(hi0, q.x);
      lo1 = fminf(lo1, q.y); hi1 = fmaxf(hi1, q.y);
      lo2 = fminf(lo2, q.z); hi2 = fmaxf(hi2, q.z);
    }
    lo = make_float4(lo0, lo1, lo2, 0.f);
    hi = make_float4(hi0, hi1, hi2, 0.f);
    ref = leaf_ref(inf.x, inf.y - inf.x + 1);
    node = c.parent_node[i];
    first = inf.x;
  }
  for (;;) {
    // which child of `node` am I?  child 0 covers [info.x, split], child 1 (split, info.y]: compare first points
    const int4 pinf = c.info[node];
    const int k = first > pinf.w ? 1 : 0;
    float4* rec = c.tnodes + 4 * (size_t)node + 2 * k;
    __stcg(&rec[0], make_float4(lo.x, lo.y, lo.z, __int_as_float(ref)));
    __stcg(&rec[1], make_float4(hi.x, hi.y, hi.z, 0.f));
    __threadfence();
    if (atomicAdd(&c.flags[node], 1u) == 0u) return;  // the sibling is still on its way: it will take the parent
    __threadfence();
    const float4 olo = __ldcg(&c.tnodes[4 * (size_t)node + 2 * (1 - k)]);
    const float4 ohi = __ldcg(&c.tnodes[4 * (size_t)node + 2 * (1 - k) + 1]);
    if (node == 0) return;
    lo = make_float4(fminf(lo.x, olo.x), fminf(lo.y, olo.y), fminf(lo.z, olo.z), 0.f);
    hi = make_float4(fmaxf(hi.x, ohi.x), fmaxf(hi.y, ohi.y), fmaxf(hi.z, ohi.z), 0.f);
    ref = node;
    first = pinf.x;
    node = c.parent_node[node];
  }
}

// ------------------------------------------------------------------------------------
// host launcher: builds `count` clouds whose descriptors are already in device memory.
// c.hist = zeroed sort work memory (radix_sort_ws_bytes(n, 30)), c.flags zeroed, c.bbox = 6 * BBOX_BLOCKS floats.
// Returns the number of kernel launches issued.
int launch_index_build(const CloudDev* d_clouds, int count, int max_n, cudaStream_t s) {
  int launches = 0;
  const int gx = max(1, min((max_n + 255) / 256, BBOX_BLOCKS));
  k_bbox<<<dim3(gx, count), 256, 0, s>>>(d_clouds); launches++;
  const dim3 tiles(sort_tiles(max_n), count);
  k_morton_ghist<<<tiles, SORT_THREADS, 0, s>>>(d_clouds, gx); launches++;
  k_sort_pass<10, false><<<tiles, SORT_THREADS, 0, s>>>(d_clouds, 0); launches++;
  k_sort_pass<10, false><<<tiles, SORT_THREADS, 0, s>>>(d_clouds, 1); launches++;
  k_sort_pass<10, true><<<tiles, SORT_THREADS, 0, s>>>(d_clouds, 2); launches++;
  if (max_n > 1) {
    k_lbvh_topology<<<dim3((max_n + 254) / 256, count), 256, 0, s>>>(d_clouds, SORT_PASSES & 1); launches++;
    k_lbvh_aabb<<<dim3((2 * max_n + 254) / 256, count), 256, 0, s>>>(d_clouds); launches++;
  }
  return launches;
}

}  // namespace b200
