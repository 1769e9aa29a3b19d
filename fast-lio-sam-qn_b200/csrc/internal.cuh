// internal.cuh -- device-side data layout shared by the kernels of libb200reg.so.
//
// HBM layout of one cloud (all arrays in MORTON-SORTED order, position p):
//   pts    float4[P]      (x, y, z, __int_as_float(original index))
//   tnodes float4[4*(P-1)] linear BVH (Karras radix tree over the 30-bit Morton keys, index
//                         tie-break for equal keys).  Node i holds BOTH children:
//                           [4i+0] = (lo0.xyz, ref0)  [4i+1] = (hi0.xyz, -)
//                           [4i+2] = (lo1.xyz, ref1)  [4i+3] = (hi1.xyz, -)
//                         ref >= 0: internal node index; ref < 0: leaf, -1-ref = (start<<4)|count
//                         with count <= LEAF consecutive points.  Subtrees of <= LEAF points are
//                         collapsed into leaves, so only ~P/4 of the P-1 slots are ever read.
//   cov   double[6*P]     regularised covariance, symmetric 3x3 (xx,xy,xz,yy,yz,zz), 48 B/point
//   rank  int[P]          original index -> sorted position
// See DESIGN.md "Data layout in HBM".
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace b200 {

constexpr int LEAF = 8;            // max points per leaf (8 x 16 B = one 128-B line); must be <= 15
constexpr int SORT_THREADS = 256;  // radix sort tile = SORT_THREADS * SORT_ITEMS keys
constexpr int SORT_ITEMS = 8;
constexpr int SORT_TILE = SORT_THREADS * SORT_ITEMS;
constexpr int BBOX_BLOCKS = 296;   // per-block bounding-box partials of one cloud (k_bbox grid.x <= this)
constexpr int STEP_THREADS = 128;  // threads per block of the per-point kernels
constexpr int NRED = 28;           // 21 (H upper) + 6 (b) + 1 (err)
constexpr int FDIM = 33;           // FPFHSignature33
constexpr int FPAD = 36;           // descriptor record padded to 144 B (9 x float4, TMA-bulk friendly)
constexpr int MAX_STACK = 64;      // >= LBVH depth: 30 key bits + index tie-break bits

struct CloudDev {
  const float* raw;    // device copy of the caller's records (xyz at stride)
  int raw_stride;      // in floats
  int n;               // points
  int root_ref;        // 0 (internal root) or a leaf ref when n <= LEAF
  float4* pts;         // [n]
  float4* tnodes;      // [4 * (n - 1)]
  double* cov;         // [6 * n] (valid once has_cov)
  int* rank;           // [n]
  // Quatro features (allocated by b200reg_clouds_fpfh; sorted order)
  float4* nrm;         // [n] unit normal, w = 1 valid / 0 invalid (< 3 neighbours)
  float* spfh;         // [FPAD * n]
  float* fpfh;         // [FPAD * n]; slot 33 = original index (int bits), slot 34 = 1.0 if the descriptor is usable, slot 35 = hash of its bits
  float4* fproj;       // [n] filter coordinates (fpfh_basis.cuh): 3 projections + residual norm, ||a-b||^2 >= their squared distance
  // the matcher's view of the descriptors: records re-ordered by the Morton code of their filter coordinates, so that a
  // tile of 64 consecutive records is a small box in filter space and whole tiles can be skipped per query
  float* fpfh_s;       // [FPAD * n] (aliases spfh, which is dead once k_fpfh has run); unusable records last; slot 34 = 1 base
                       // record / 2 duplicate of its predecessor (query only), slot 35 = index a base record answers with
  float4* fproj_s;     // [n]
  float4* ftile;       // [2 * ceil(n / 64)] per tile: min and max filter coordinates of its base records (+inf / -inf if none)
  uint32_t* fcode_s;   // [n] sorted keys: 28-bit filter-space Morton code, 4 hash bits (0xFFFFFFFF for unusable records)
  // build-time temporaries (freed after the build)
  uint32_t* keys[2];   // sort ping-pong
  uint32_t* vals[2];
  uint32_t* hist;      // radix-sort work memory, ZEROED by the caller: radix_sort_ws_bytes(n, key_bits) (index_build.cu)
  uint32_t* flags;     // [n - 1] arrival flags of the bottom-up AABB pass, ZEROED by the caller
  int4* info;          // [n - 1] (first, last, leaf-child bits, split)
  int* parent_node;    // [n - 1]
  int* parent_leaf;    // [n]
  float* bbox;         // [6 * BBOX_BLOCKS] per-block min/max partials
};

// phase of the per-pair LM state machine
enum Phase : int { PH_LINEARIZE = 0, PH_TRIAL = 1, PH_FITNESS = 2, PH_DONE = 3 };

struct GicpParamsDev {
  int max_iterations;
  int lm_max_iterations;
  double max_corr_dist2;
  double transformation_eps;
  double rotation_eps;
  double lm_init_lambda_factor;
  double icp_score_thr;
};

struct PairState {
  // current estimate x0 and trial xi = delta * x0 (row-major R, t)
  double R[9], t[3];
  double Rt[9], tt[3];
  double dR[9], dt[3];  // delta of the current trial
  double d[6];
  double H[36], b[6];
  double y0;
  double y_trial;       // sum of errors of the last compute_error pass
  double lambda, nu;
  double fitness;
  float Tf[12];  // x0.cast<float>() rows (r0 r1 r2 t)
  int phase;
  int outer_it;  // index of the current outer iteration
  int inner_it;  // LM trials done in this outer iteration
  int converged;
  int lm_failed;
  int n_lin, n_err;
  int nr_iterations;
  unsigned int arrive;  // (unused since the controller became its own kernel; kept for layout stability)
  int pad;
};

// Device-side schedule of one batched LM solve: the step kernels run over WORK ITEMS (one 128-point block of one
// still-active pair).  Items are laid out with a uniform stride: item = slot * stride + block, slot indexing the list of
// active pairs, stride = the largest block count of any pair of the call (a few items of a shorter pair are empty).
// A block copies the slot list (pair id, block count, phase) into shared memory once, so locating an item costs no
// global load.  The last block of every step rebuilds the list from the pairs' phases: finished pairs cost nothing from
// the next step on, and the host (or the CUDA-graph while node) never looks at anything but the loop condition.
struct LmSlot {
  int pair;    // index into the call's pair array
  int nblk;    // ceil(src.n / STEP_THREADS)
  int phase;   // the pair's phase during this step
  int seeded;  // n_lin > 0: corr[] holds the previous linearization's correspondences
};
constexpr int LM_SMEM_SLOTS = 512;  // slot entries cached per block (8 KB); larger batches read the rest from global memory

struct LmSched {
  int n_pairs;
  int n_active;           // pairs whose phase != PH_DONE
  int stride;             // max over the call's pairs of their block count
  int total_items;        // n_active * stride
  int done;               // pairs that reached PH_DONE
  unsigned int arrive;    // blocks that finished the current step
  int steps;              // step iterations executed
  int pad;
  LmSlot* slots;          // [n_pairs]
};

// Per-call parameters of one batched LM solve, read by the kernels from device memory (not passed by value) so that the
// CUDA graph of the solve can be instantiated once per context and re-launched for every call.
struct LmCall {
  int count;            // pairs of this call
  int has_guess;        // guess16 holds count x 16 doubles (row-major); otherwise identity
  int max_steps;        // safety cap on the number of step iterations of the device-side loop
  int overrun;          // set by the device when max_steps was hit (a bug in the state machine, never expected)
  unsigned long long cond_handle;  // cudaGraphConditionalHandle of the while node, 0 when the step kernels are launched directly
  GicpParamsDev prm;
};

struct PairDev {
  CloudDev src, tgt;
  int* corr;       // [src.n] sorted target position or -1 (per sorted source position)
  float* sqd;      // [src.n]
  double* mahal;   // [6 * src.n]
  double* partial; // [ceil(src.n / 32) * NRED] one row per warp of the accumulate kernel
};

struct LmGraph {  // host side: the instantiated graph of one context's LM solve (gicp.cu: lm_graph_build)
  cudaGraph_t graph = nullptr;
  cudaGraphExec_t exec = nullptr;
  unsigned long long cond_handle = 0;
};

// ---- keyframe store / cloud assembly (SURVEY §8f) -------------------------------------------
constexpr int MAXSEG = 32;  // keyframes merged into one cloud: 2 * submap_range + 1 <= MAXSEG
struct KeyframeDev {
  const float4* pts;  // (x, y, z, intensity), LiDAR frame, original order
  int n;
  int pad;
};
struct SortBufs {  // what the radix sort needs (mirrors the CloudDev fields it reads)
  uint32_t* keys[2];
  uint32_t* vals[2];
  uint32_t* hist;   // zeroed work memory, radix_sort_ws_bytes(total, 32)
};
struct AssembleJob {  // one output cloud of setSrcAndDstCloud
  int nseg, total;
  int seg_kf[MAXSEG];
  int seg_off[MAXSEG + 1];
  float4* merged;   // [total] transformed, merged points
  float4* out;      // [total] voxel centroids (counters[0] of them)
  int* heads;       // [total]
  int* bbox;        // [6] ordered-int min/max
  int* counters;    // [0] voxels, [1] int32-overflow flag
  SortBufs sort;
};

// ---- global map: transformPcd over the whole store + one pcl::VoxelGrid (map.cu) ------------------
constexpr int MAP_THREADS = 256;
constexpr int MAP_TILE = 2048;  // points per block of the transform and of the run-head kernels
struct MapBlock {               // one tile of one keyframe (built on the host: no per-point keyframe search)
  const float4* src;            // first point of the tile in the keyframe's slab
  int kf;                       // keyframe (row of the pose table)
  int dst;                      // first merged index of the tile
  int n;                        // points, <= MAP_TILE
  int pad;
};
struct VoxelGridDev {
  int min_b[3];     // floor(min * (1/L))
  int div_b[3];     // floor(max * (1/L)) - min_b + 1
  long long cells;  // PCL's overflow test: prod((int64)((max - min) * (1/L)) + 1)
};
struct MapInfo {    // written by the device, read back by the host between the phases of a map build
  VoxelGridDev grid;
  int overflow;     // PCL's int32 guard tripped: the map is the merged cloud
  int key_bits;     // ceil(log2(div_b0 * div_b1 * div_b2)), at most 32
  int voxels;       // occupied voxels
  int pad;
};

// ---- Quatro matcher / solver workspace ---------------------------------------------------
// per-pair device workspace of the matcher / solver
struct MatchDev {
  CloudDev fi, fj;     // fi = larger cloud (base of the forward search), fj = smaller
  int swapped;         // 1 when fi is the DESTINATION cloud (matcher.cc:364-369)
  int* nn;             // [nj] original fi index of the 1-NN of fj point j (by ORIGINAL j), -1 if none
  float* dis;          // [nj]
  int* first_j;        // [ni] min original j that hit i (INT_MAX if none)
  int* rnn;            // [ni] original j returned by the reverse search (by ORIGINAL i)
  int* corres;         // [2 * nj] mutual (i, j) pairs, ascending j
  unsigned* tkey;      // [nj] first (trial*4 + slot) at which correspondence r would be added
  int* counters;       // [0] unused, [1] ncorr, [2] n_out, [3] valid, [4] clique size, [5] gnc iterations
  double* stats;       // [0..2] sum fi, [3..5] sum fj, then floats: mean fi(3) mean fj(3) scale (as float bits in doubles)
  int* out_corr;       // [2 * corr_cap] final (src, dst) pairs (corr_cap = MAXC, or BigSolveWs::cap for advancedMatching)
  double* T;           // [16] row-major result
  struct BigSolveWs* big;  // global-memory solver workspace (advancedMatching only; nullptr otherwise)
};

// Global-memory workspace of the multi-kernel TEASER++ solve used when the correspondence set is not capped at MAXC
// (Matcher::advancedMatching, matcher.cc:118-356).  cap is a multiple of 1024, words = cap / 32.
struct BigSolveWs {
  int cap, words;
  double* S;                 // [cap * 3] source points of the correspondences
  double* D;                 // [cap * 3]
  unsigned* adj;             // [cap * words] TIM consistency graph, bit j of row i
  unsigned* radj;            // [cap * words] same graph with vertices renamed by their rank in the clique order
  int *deg, *pdeg, *core, *alive, *rank, *order, *csize, *clique, *list;  // [cap] each
  unsigned long long* skey;  // [cap]
  double *w, *res;           // [cap]
  double* hval;              // [2 * cap]
  int* hidx;                 // [2 * cap]
};

struct QuatroParamsDev {
  float normal_r2, fpfh_r2;
  float thr2;          // distance_threshold^2 (feature space)
  float tuple_scale;
  int max_corres;
  double noise_bound, gnc_factor, cost_thr;
  int max_iter;
  unsigned long long seed;
  int advanced;        // 1: Matcher::advancedMatching (cross check, 3-edge tuple test, no cap); 0: optimizedMatching
};

constexpr int MAXC = 512;  // capacity of the final correspondence set (max_corres + 3 <= MAXC)
constexpr int BIGC = 8192; // capacity of the advancedMatching correspondence set (B200REG_ADV_CORR_CAPACITY)

// ---- ordered-int encoding of floats for atomicMin/atomicMax ------------------------
__device__ __forceinline__ int f2ord(float f) {
  int i = __float_as_int(f);
  return i >= 0 ? i : i ^ 0x7FFFFFFF;
}
__device__ __forceinline__ float ord2f(int i) { return __int_as_float(i >= 0 ? i : i ^ 0x7FFFFFFF); }

__host__ __device__ __forceinline__ int leaf_ref(int start, int count) { return -1 - ((start << 4) | count); }

}  // namespace b200
