// api.cu -- the C ABI declared in include/b200reg.h: contexts, cloud objects, batched drivers.
// Host orchestration only; every arithmetic step of the path runs in the kernels of
// index_build.cu / gicp.cu.  There is no CPU fallback anywhere in this library.
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <nccl.h>  // types only: the library is dlopen()ed in b200reg_comm_*

#include <algorithm>
#include <cstddef>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/b200reg.h"
#include "internal.cuh"

namespace b200 {
int launch_index_build(const CloudDev* d_clouds, int count, int max_n, cudaStream_t s);
size_t radix_sort_ws_bytes(int n, int key_bits);
int launch_covariances(const CloudDev* d_clouds, int count, int max_n, int k, int method, cudaStream_t s);
void launch_gicp_init(const PairDev* pairs, PairState* states, const double* d_guess, LmCall* call, LmSched* sched, cudaStream_t s);
int launch_gicp_step(const PairDev* pairs, PairState* states, int blocks_search, int blocks_accum, LmCall* call, LmSched* sched, cudaStream_t s);
void launch_gicp_search(const PairDev* pairs, const PairState* states, int blocks, const LmCall* call, const LmSched* sched, cudaStream_t s);
void launch_gicp_accum(const PairDev* pairs, const PairState* states, int blocks, const LmSched* sched, cudaStream_t s);
void launch_gicp_control(const PairDev* pairs, PairState* states, LmCall* call, LmSched* sched, cudaStream_t s);
cudaError_t lm_graph_build(LmGraph* g, const PairDev* pairs, PairState* states, const double* guess, LmCall* call, LmSched* sched,
                           int blocks_search, int blocks_accum);
void lm_graph_destroy(LmGraph* g);
int launch_knn_queries(const CloudDev& c, const float* d_q, int nq, int qstride, int k, int* idx, float* d2, cudaStream_t s, int brute);
void launch_transform_out(const CloudDev& c, const float* d_Tf, float* d_out3, cudaStream_t s);
void launch_set_covariances(const CloudDev& c, const double* d_cov9, cudaStream_t s);
int launch_fpfh(const CloudDev* d_clouds, int count, int max_n, float normal_r2, float fpfh_r2, cudaStream_t s);
int launch_quatro_match_solve(const MatchDev* d_pairs, int count, int max_ni, int max_nj, const QuatroParamsDev& prm, cudaStream_t s);
void launch_transform_raw(const CloudDev* d_clouds, const double* d_T16s, int count, int max_n, float4* const* d_outs, cudaStream_t s);
int launch_fetch_closest(const double* d_pos, const double* d_stamp, const int* d_queries, int count, double radius, double tdiff,
                         int* d_out, cudaStream_t s);
cudaError_t quatro_init_device();
void launch_ingest_world(const float* d_raw, int stride, int n, const double* d_Tinv, float4* d_out, cudaStream_t s);
void launch_pack_xyzi(const float* d_raw, int stride, int n, float4* d_out, cudaStream_t s);
int launch_assemble_voxelize(const AssembleJob* d_jobs, const CloudDev* d_sort, int count, int max_total, const KeyframeDev* d_kfs,
                             const double* d_poses, float inv_leaf, cudaStream_t s);
int launch_map_transform(const MapBlock* d_blocks, int nblocks, const double* d_poses, float inv_leaf, float4* d_merged,
                         float* d_partials, MapInfo* d_info, cudaStream_t s);
int launch_map_sort_heads(const float4* d_merged, int n, float inv_leaf, MapInfo* d_info, const CloudDev* d_sort, const CloudDev& sort,
                          int key_bits, int* d_tile_cnt, int* d_tile_off, int* d_heads, float4* d_sorted, cudaStream_t s);
int launch_map_centroids(const int* d_heads, const float4* d_sorted, int nv, float4* d_out, cudaStream_t s);
}  // namespace b200

using namespace b200;

static thread_local std::string g_err;
static int fail(int code, const std::string& msg) {
  g_err = msg;
  return code;
}
#define CU(call)                                                                                              \
  do {                                                                                                        \
    cudaError_t _e = (call);                                                                                  \
    if (_e != cudaSuccess)                                                                                    \
      return fail(B200REG_ECUDA, std::string(#call) + ": " + cudaGetErrorString(_e) + " @" + __FILE__ + ":" + \
                                     std::to_string(__LINE__));                                               \
  } while (0)

enum { CLS_BUILD = 0, CLS_COV = 1, CLS_STEP = 2, CLS_MISC = 3, CLS_FPFH = 4, CLS_MATCH = 5, CLS_SEARCH = 6, CLS_ACCUM = 7, CLS_CTRL = 8, NCLS = 9 };

struct b200reg_ctx {
  int device = 0;
  cudaStream_t own_stream = nullptr;
  cudaStream_t stream = nullptr;
  cudaStream_t copy_stream = nullptr;  // H2D uploads of later chunks overlap the compute of earlier ones
  cudaMemPool_t pool = nullptr;        // per-context pool: reuse never adds dependencies on another context's streams
  int pipeline_chunks = 4;
  int sm_count = 148;
  // persistent arena of the batched LM solve: every kernel argument of the solve's CUDA graph points in here, so the graph is
  // instantiated once and re-launched by every b200reg_gicp_align call until a larger batch makes the arena grow
  struct LmArena {
    int cap = 0;
    PairDev* d_pairs = nullptr;
    PairState* d_states = nullptr;
    LmSched* d_sched = nullptr;  // header + slots[cap]
    double* d_guess = nullptr;   // [16 * cap]
    LmCall* d_call = nullptr;
    LmCall* h_call = nullptr;    // pinned staging
    PairState* h_states = nullptr;  // pinned read-back
    LmGraph graph;
  } lm;
  // the path's one collective (b200reg_comm_*): NCCL communicator of this rank
  ncclComm_t comm = nullptr;
  int rank = -1, world = 1;
  int64_t launches = 0;
  // optional per-kernel-family timing with CUDA events on the launching stream
  bool profiling = false;
  struct Span { int cls; cudaEvent_t a, b; };
  std::vector<Span> pending;
  std::vector<cudaEvent_t> free_events;
  double prof_ms[NCLS] = {0};
  double prof_bytes[NCLS] = {0};
  int64_t prof_launches[NCLS] = {0};
};

// gicp_step = the whole LM loop of a solve when it runs as one graph launch; with profiling enabled the same kernels are
// launched one by one and timed per kernel: gicp_search / gicp_accum / gicp_control (and gicp_step stays empty)
static const char* kClassNames[NCLS] = {"index_build", "knn_covariance", "gicp_step", "misc", "fpfh", "quatro_match_solve",
                                        "gicp_search", "gicp_accum", "gicp_control"};

static cudaEvent_t prof_event(b200reg_ctx* c) {
  cudaEvent_t e;
  if (!c->free_events.empty()) {
    e = c->free_events.back();
    c->free_events.pop_back();
  } else {
    cudaEventCreate(&e);
  }
  return e;
}
struct ProfScope {  // brackets the kernels launched while it is alive
  b200reg_ctx* c;
  int cls;
  cudaEvent_t a = nullptr;
  int64_t l0;
  ProfScope(b200reg_ctx* c_, int cls_) : c(c_), cls(cls_), l0(c_->launches) {
    if (c->profiling) {
      a = prof_event(c);
      cudaEventRecord(a, c->stream);
    }
  }
  ~ProfScope() {
    if (c->profiling) {
      cudaEvent_t b = prof_event(c);
      cudaEventRecord(b, c->stream);
      c->pending.push_back({cls, a, b});
      c->prof_launches[cls] += c->launches - l0;
    }
  }
};
static void prof_resolve(b200reg_ctx* c) {
  for (auto& sp : c->pending) {
    float ms = 0.f;
    cudaEventSynchronize(sp.b);
    cudaEventElapsedTime(&ms, sp.a, sp.b);
    c->prof_ms[sp.cls] += ms;
    c->free_events.push_back(sp.a);
    c->free_events.push_back(sp.b);
  }
  c->pending.clear();
}

// Stream-ordered scratch memory with scope lifetime: everything allocated through it is returned to the context's
// pool when the scope ends -- on every path, including the early error returns of the CU() macro.
struct Scratch {
  b200reg_ctx* c;
  std::vector<void*> ptrs;
  explicit Scratch(b200reg_ctx* c_) : c(c_) {}
  Scratch(const Scratch&) = delete;
  Scratch& operator=(const Scratch&) = delete;
  cudaError_t alloc(void** p, size_t bytes) {
    cudaError_t e = cudaMallocFromPoolAsync(p, bytes ? bytes : 16, c->pool, c->stream);
    if (e == cudaSuccess) ptrs.push_back(*p);
    return e;
  }
  ~Scratch() {
    for (void* p : ptrs) cudaFreeAsync(p, c->stream);
  }
};

// scope guards: events and cloud handles created inside a call are released on EVERY exit path (the CU() macro returns early)
struct EventBag {
  std::vector<cudaEvent_t> ev;
  cudaError_t make(cudaEvent_t* e) {
    const cudaError_t r = cudaEventCreateWithFlags(e, cudaEventDisableTiming);
    if (r == cudaSuccess) ev.push_back(*e);
    return r;
  }
  ~EventBag() {
    for (cudaEvent_t e : ev) cudaEventDestroy(e);
  }
};
struct CloudBag {
  b200reg_ctx* c;
  std::vector<b200reg_cloud*> cl;
  explicit CloudBag(b200reg_ctx* c_) : c(c_) {}
  ~CloudBag();
};

struct b200reg_cloud {
  CloudDev dev;            // device pointers + sizes
  void* slab = nullptr;    // persistent allocation (pts, tnodes, cov, rank)
  void* fslab = nullptr;   // Quatro features (nrm, spfh, fpfh), allocated on demand
  bool has_cov = false;
  bool cov_user = false;   // set by b200reg_set_covariances: never recomputed on demand (nano_gicp_impl.hpp:162-167)
  int cov_k = 0;
  int cov_method = 3;
  bool has_fpfh = false;
  double normal_r = 0, fpfh_r = 0;
};

static size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

CloudBag::~CloudBag() {
  for (b200reg_cloud* p : cl) b200reg_cloud_destroy(c, p);
}

static void lm_arena_free(b200reg_ctx* c) {
  auto& a = c->lm;
  lm_graph_destroy(&a.graph);
  if (a.d_pairs) cudaFree(a.d_pairs);
  if (a.d_states) cudaFree(a.d_states);
  if (a.d_sched) cudaFree(a.d_sched);
  if (a.d_guess) cudaFree(a.d_guess);
  if (a.d_call) cudaFree(a.d_call);
  if (a.h_call) cudaFreeHost(a.h_call);
  if (a.h_states) cudaFreeHost(a.h_states);
  a = b200reg_ctx::LmArena();
}

// make the arena hold `count` pairs and make sure its graph exists
static int lm_arena_ensure(b200reg_ctx* c, int count) {
  auto& a = c->lm;
  if (count > a.cap) {
    CU(cudaStreamSynchronize(c->stream));  // nothing of an earlier solve may still read the old buffers
    lm_arena_free(c);
    const int cap = std::max(16, count + count / 2);
    CU(cudaMalloc(&a.d_pairs, sizeof(PairDev) * cap));
    CU(cudaMalloc(&a.d_states, sizeof(PairState) * cap));
    CU(cudaMemsetAsync(a.d_states, 0, sizeof(PairState) * cap, c->stream));  // the records travel to the host whole: no stale bytes
    CU(cudaMalloc((void**)&a.d_sched, 64 + sizeof(LmSlot) * (size_t)cap));
    CU(cudaMalloc(&a.d_guess, sizeof(double) * 16 * cap));
    CU(cudaMalloc(&a.d_call, sizeof(LmCall)));
    CU(cudaMallocHost(&a.h_call, sizeof(LmCall)));
    CU(cudaMallocHost(&a.h_states, sizeof(PairState) * cap));
    LmSched hs;
    memset(&hs, 0, sizeof(hs));
    static_assert(sizeof(LmSched) <= 64, "LmSched header");
    hs.slots = (LmSlot*)((char*)a.d_sched + 64);
    CU(cudaMemcpy(a.d_sched, &hs, sizeof(hs), cudaMemcpyHostToDevice));
    a.cap = cap;
  }
  if (!a.graph.exec) {
    // persistent grids: as many blocks as can be resident (search: 16 per SM at 32 registers, accumulate: 8 per SM);
    // blocks beyond the current number of work items exit at once
    const int bps = 32, bpa = 32;  // measured: 8 / 16 / 32 / 64 blocks per SM -> 1.83-1.92 ms per 16-pair solve, flat from 32 on
    const cudaError_t e = lm_graph_build(&a.graph, a.d_pairs, a.d_states, a.d_guess, a.d_call, a.d_sched, c->sm_count * bps, c->sm_count * bpa);
    if (e != cudaSuccess) return fail(B200REG_ECUDA, std::string("building the LM graph: ") + cudaGetErrorString(e));
  }
  return B200REG_OK;
}

extern "C" {

void b200reg_default_gicp_params(b200reg_gicp_params* p) {
  if (!p) return;
  p->k_correspondences = 15;
  p->max_iterations = 32;
  p->max_corr_dist = 52.5;
  p->transformation_eps = 0.01;
  p->rotation_eps = 2e-3;
  p->lm_max_iterations = 10;
  p->regularization = 3;  // PLANE
  p->lm_init_lambda_factor = 1e-9;
  p->icp_score_thr = 1.5;
}

const char* b200reg_last_error(void) { return g_err.c_str(); }
void b200reg_set_last_error(const char* message) { g_err = message ? message : ""; }
const char* b200reg_version(void) { return "b200reg 0.2 (sm_100a)"; }
size_t b200reg_struct_size(int which) {
  switch (which) {
    case 0: return sizeof(b200reg_gicp_params);
    case 1: return sizeof(b200reg_result);
    case 2: return sizeof(b200reg_quatro_params);
    case 3: return sizeof(b200reg_quatro_info);
    case 4: return sizeof(b200reg_loop_config);
    case 5: return sizeof(b200reg_loop_factor);
    default: return 0;
  }
}

int b200reg_ctx_create(int device, b200reg_ctx** out) {
  if (!out) return fail(B200REG_EINVAL, "out is NULL");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0 || device < 0 || device >= ndev)
    return fail(B200REG_ENODEV, "no usable CUDA device (this library has no CPU fallback)");
  CU(cudaSetDevice(device));
  CU(quatro_init_device());
  b200reg_ctx* c = new b200reg_ctx;
  c->device = device;
  struct Undo {  // a failure half way must not leak the context
    b200reg_ctx* c;
    bool ok = false;
    ~Undo() {
      if (!ok) b200reg_ctx_destroy(c);
    }
  } undo{c};
  CU(cudaStreamCreateWithFlags(&c->own_stream, cudaStreamNonBlocking));
  CU(cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking));
  c->stream = c->own_stream;
  cudaMemPoolProps props = {};
  props.allocType = cudaMemAllocationTypePinned;
  props.handleTypes = cudaMemHandleTypeNone;
  props.location.type = cudaMemLocationTypeDevice;
  props.location.id = device;
  CU(cudaMemPoolCreate(&c->pool, &props));
  uint64_t thr = UINT64_MAX;
  CU(cudaMemPoolSetAttribute(c->pool, cudaMemPoolAttrReleaseThreshold, &thr));
  CU(cudaDeviceGetAttribute(&c->sm_count, cudaDevAttrMultiProcessorCount, device));
  undo.ok = true;
  *out = c;
  return B200REG_OK;
}

int b200reg_ctx_destroy(b200reg_ctx* c) {
  if (!c) return B200REG_OK;
  cudaSetDevice(c->device);
  if (c->stream) cudaStreamSynchronize(c->stream);
  if (c->comm) b200reg_comm_destroy(c);
  lm_arena_free(c);
  if (c->own_stream) cudaStreamDestroy(c->own_stream);
  if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
  if (c->pool) cudaMemPoolDestroy(c->pool);
  delete c;
  return B200REG_OK;
}

int b200reg_ctx_set_stream(b200reg_ctx* c, void* s) {
  if (!c) return fail(B200REG_EINVAL, "ctx is NULL");
  c->stream = s ? (cudaStream_t)s : c->own_stream;
  return B200REG_OK;
}

int b200reg_ctx_synchronize(b200reg_ctx* c) {
  if (!c) return fail(B200REG_EINVAL, "ctx is NULL");
  CU(cudaSetDevice(c->device));
  CU(cudaStreamSynchronize(c->stream));
  return B200REG_OK;
}

int64_t b200reg_ctx_launch_count(const b200reg_ctx* c) { return c ? c->launches : 0; }

int b200reg_ctx_set_profiling(b200reg_ctx* c, int enable) {
  if (!c) return fail(B200REG_EINVAL, "ctx is NULL");
  CU(cudaSetDevice(c->device));
  prof_resolve(c);
  c->profiling = enable != 0;
  return B200REG_OK;
}

int b200reg_ctx_reset_profile(b200reg_ctx* c) {
  if (!c) return fail(B200REG_EINVAL, "ctx is NULL");
  prof_resolve(c);
  for (int i = 0; i < NCLS; i++) {
    c->prof_ms[i] = 0;
    c->prof_bytes[i] = 0;
    c->prof_launches[i] = 0;
  }
  return B200REG_OK;
}

int b200reg_ctx_get_profile(b200reg_ctx* c, int cls, const char** name, double* ms, double* algo_bytes, int64_t* launches) {
  if (!c || cls < 0 || cls >= NCLS) return fail(B200REG_EINVAL, "bad class");
  CU(cudaSetDevice(c->device));
  prof_resolve(c);
  if (name) *name = kClassNames[cls];
  if (ms) *ms = c->prof_ms[cls];
  if (algo_bytes) *algo_bytes = c->prof_bytes[cls];
  if (launches) *launches = c->prof_launches[cls];
  return B200REG_OK;
}

size_t b200reg_cloud_size(const b200reg_cloud* cl) { return cl ? (size_t)cl->dev.n : 0; }

// ------------------------------------------------------------------------------------------
int b200reg_clouds_create(b200reg_ctx* c, int count, const float* const* xyz, const size_t* n, size_t stride_bytes,
                          int on_device, b200reg_cloud** out) {
  if (!c || count <= 0 || !xyz || !n || !out) return fail(B200REG_EINVAL, "bad argument");
  if (stride_bytes < 12 || stride_bytes % 4) return fail(B200REG_EINVAL, "stride_bytes must be a multiple of 4, >= 12");
  for (int i = 0; i < count; i++)
    if (!xyz[i] || n[i] == 0 || n[i] > (size_t)(1u << 26)) return fail(B200REG_EINVAL, "empty or oversized cloud");
  CU(cudaSetDevice(c->device));
  cudaStream_t s = c->stream;
  Scratch scratch(c);
  std::vector<CloudDev> descs(count);
  int max_n = 0;
  for (int i = 0; i < count; i++) out[i] = nullptr;
  struct Guard {  // a failure half way must not leak the clouds already created
    b200reg_ctx* c;
    b200reg_cloud** out;
    int count;
    bool ok = false;
    ~Guard() {
      if (ok) return;
      for (int i = 0; i < count; i++) {
        if (out[i]) {
          if (out[i]->slab) cudaFreeAsync(out[i]->slab, c->stream);
          delete out[i];
          out[i] = nullptr;
        }
      }
    }
  } guard{c, out, count};
  // sort work memory and AABB arrival flags of the whole batch: ONE allocation, ONE memset
  std::vector<size_t> z_ws(count), z_fl(count);
  size_t z_total = 0;
  for (int i = 0; i < count; i++) {
    z_ws[i] = z_total;
    z_total = align_up(z_total + radix_sort_ws_bytes((int)n[i], 30), 256);
    z_fl[i] = z_total;
    z_total = align_up(z_total + (size_t)std::max((int)n[i] - 1, 1) * 4, 256);
  }
  char* zeroed = nullptr;
  CU(scratch.alloc((void**)&zeroed, z_total));
  CU(cudaMemsetAsync(zeroed, 0, z_total, s));
  for (int i = 0; i < count; i++) {
    b200reg_cloud* cl = new b200reg_cloud;
    out[i] = cl;
    CloudDev& d = cl->dev;
    d.n = (int)n[i];
    d.root_ref = d.n <= LEAF ? leaf_ref(0, d.n) : 0;
    d.raw_stride = (int)(stride_bytes / 4);
    const size_t nn = (size_t)std::max(d.n - 1, 1);
    // persistent slab
    size_t o_pts = 0;
    size_t o_tn = align_up(o_pts + (size_t)d.n * sizeof(float4), 256);
    size_t o_cov = align_up(o_tn + 4 * nn * sizeof(float4), 256);
    size_t o_rank = align_up(o_cov + (size_t)6 * d.n * sizeof(double), 256);
    size_t total = align_up(o_rank + (size_t)d.n * sizeof(int), 256);
    char* slab = nullptr;
    CU(cudaMallocFromPoolAsync((void**)&slab, total, c->pool, s));
    cl->slab = slab;
    d.pts = (float4*)(slab + o_pts);
    d.tnodes = (float4*)(slab + o_tn);
    d.cov = (double*)(slab + o_cov);
    d.rank = (int*)(slab + o_rank);
    d.nrm = nullptr;
    d.spfh = nullptr;
    d.fpfh = nullptr;
    d.fproj = nullptr;
    d.fpfh_s = nullptr;
    d.fproj_s = nullptr;
    d.ftile = nullptr;
    d.fcode_s = nullptr;
    // temporary slab (sort buffers, tree scratch, bbox partials, and the raw records when uploading)
    size_t t_k0 = 0;
    size_t t_k1 = align_up(t_k0 + (size_t)d.n * 4, 256);
    size_t t_v0 = align_up(t_k1 + (size_t)d.n * 4, 256);
    size_t t_v1 = align_up(t_v0 + (size_t)d.n * 4, 256);
    size_t t_i = align_up(t_v1 + (size_t)d.n * 4, 256);
    size_t t_pn = align_up(t_i + nn * sizeof(int4), 256);
    size_t t_pl = align_up(t_pn + nn * 4, 256);
    size_t t_b = align_up(t_pl + (size_t)d.n * 4, 256);
    size_t t_raw = align_up(t_b + 6 * BBOX_BLOCKS * sizeof(float), 256);
    size_t t_total = t_raw + (on_device ? 0 : align_up((size_t)d.n * stride_bytes, 256));
    char* tmp = nullptr;
    CU(scratch.alloc((void**)&tmp, t_total));
    d.keys[0] = (uint32_t*)(tmp + t_k0);
    d.keys[1] = (uint32_t*)(tmp + t_k1);
    d.vals[0] = (uint32_t*)(tmp + t_v0);
    d.vals[1] = (uint32_t*)(tmp + t_v1);
    d.hist = (uint32_t*)(zeroed + z_ws[i]);
    d.flags = (uint32_t*)(zeroed + z_fl[i]);
    d.info = (int4*)(tmp + t_i);
    d.parent_node = (int*)(tmp + t_pn);
    d.parent_leaf = (int*)(tmp + t_pl);
    d.bbox = (float*)(tmp + t_b);
    if (on_device) {
      d.raw = xyz[i];
    } else {
      CU(cudaMemcpyAsync(tmp + t_raw, xyz[i], (size_t)d.n * stride_bytes, cudaMemcpyHostToDevice, s));
      d.raw = (const float*)(tmp + t_raw);
    }
    descs[i] = d;
    out[i] = cl;
    max_n = std::max(max_n, d.n);
  }
  CloudDev* d_descs = nullptr;
  CU(scratch.alloc((void**)&d_descs, sizeof(CloudDev) * count));
  CU(cudaMemcpyAsync(d_descs, descs.data(), sizeof(CloudDev) * count, cudaMemcpyHostToDevice, s));
  {
    ProfScope ps(c, CLS_BUILD);
    c->launches += launch_index_build(d_descs, count, max_n, s);
    for (int i = 0; i < count; i++) c->prof_bytes[CLS_BUILD] += 36.0 * descs[i].n;  // SURVEY §8(d) K1
  }
  CU(cudaGetLastError());
  for (int i = 0; i < count; i++) {  // the temporaries are gone once the build has run
    CloudDev& d = out[i]->dev;
    d.raw = nullptr;
    d.keys[0] = d.keys[1] = d.vals[0] = d.vals[1] = d.hist = d.flags = nullptr;
    d.info = nullptr;
    d.parent_node = d.parent_leaf = nullptr;
    d.bbox = nullptr;
  }
  if (!on_device) CU(cudaStreamSynchronize(s));  // host buffers have been consumed when the call returns (pinned or not)
  guard.ok = true;
  return B200REG_OK;
}

int b200reg_cloud_destroy(b200reg_ctx* c, b200reg_cloud* cl) {
  if (!cl) return B200REG_OK;
  if (!c) return fail(B200REG_EINVAL, "ctx is NULL");
  CU(cudaSetDevice(c->device));
  if (cl->slab) CU(cudaFreeAsync(cl->slab, c->stream));
  if (cl->fslab) CU(cudaFreeAsync(cl->fslab, c->stream));
  delete cl;
  return B200REG_OK;
}

int b200reg_clouds_covariances(b200reg_ctx* c, int count, b200reg_cloud* const* clouds, int k) {
  return b200reg_clouds_covariances_ex(c, count, clouds, k, 3);
}

int b200reg_clouds_covariances_ex(b200reg_ctx* c, int count, b200reg_cloud* const* clouds, int k, int method) {
  if (!c || count <= 0 || !clouds) return fail(B200REG_EINVAL, "bad argument");
  if (method < 0 || method > 4) return fail(B200REG_EINVAL, "regularization must be 0..4 (NONE, MIN_EIG, NORMALIZED_MIN_EIG, PLANE, FROBENIUS)");
  if (k < 1 || k > 32) return fail(B200REG_EINVAL, "k_correspondences must be in 1..32");
  CU(cudaSetDevice(c->device));
  cudaStream_t s = c->stream;
  Scratch scratch(c);
  std::vector<CloudDev> descs;
  int max_n = 0;
  for (int i = 0; i < count; i++) {
    if (!clouds[i]) return fail(B200REG_EINVAL, "NULL cloud");
    if (clouds[i]->has_cov && !clouds[i]->cov_user && clouds[i]->cov_k == k && clouds[i]->cov_method == method) continue;
    bool dup = false;
    for (int j = 0; j < i; j++) dup |= clouds[j] == clouds[i];
    if (dup) continue;
    descs.push_back(clouds[i]->dev);
    max_n = std::max(max_n, clouds[i]->dev.n);
  }
  if (descs.empty()) return B200REG_OK;
  CloudDev* d_descs = nullptr;
  CU(scratch.alloc((void**)&d_descs, sizeof(CloudDev) * descs.size()));
  CU(cudaMemcpyAsync(d_descs, descs.data(), sizeof(CloudDev) * descs.size(), cudaMemcpyHostToDevice, s));
  {
    ProfScope ps(c, CLS_COV);
    int l = launch_covariances(d_descs, (int)descs.size(), max_n, k, method, s);
    if (l < 0) return fail(B200REG_EINVAL, "unsupported k");
    c->launches += l;
    for (auto& d : descs) c->prof_bytes[CLS_COV] += 64.0 * d.n;  // SURVEY §8(d) K2
  }
  CU(cudaGetLastError());
  for (int i = 0; i < count; i++) {
    clouds[i]->has_cov = true;
    clouds[i]->cov_user = false;
    clouds[i]->cov_k = k;
    clouds[i]->cov_method = method;
  }
  return B200REG_OK;
}

int b200reg_set_covariances(b200reg_ctx* c, b200reg_cloud* cl, const double* cov9, size_t n) {
  if (!c || !cl || !cov9) return fail(B200REG_EINVAL, "bad argument");
  if (n != (size_t)cl->dev.n) return fail(B200REG_EINVAL, "covariance count differs from the cloud size");
  CU(cudaSetDevice(c->device));
  cudaStream_t s = c->stream;
  Scratch scratch(c);
  double* d_cov9 = nullptr;
  CU(scratch.alloc((void**)&d_cov9, n * 72));
  CU(cudaMemcpyAsync(d_cov9, cov9, n * 72, cudaMemcpyHostToDevice, s));
  launch_set_covariances(cl->dev, d_cov9, s);
  c->launches++;
  CU(cudaGetLastError());
  CU(cudaStreamSynchronize(s));  // the caller's buffer may go away
  cl->has_cov = true;
  cl->cov_user = true;
  return B200REG_OK;
}

// ------------------------------------------------------------------------------------------
static GicpParamsDev to_dev(const b200reg_gicp_params& p) {
  GicpParamsDev d;
  d.max_iterations = p.max_iterations;
  d.lm_max_iterations = p.lm_max_iterations;
  d.max_corr_dist2 = p.max_corr_dist * p.max_corr_dist;
  d.transformation_eps = p.transformation_eps;
  d.rotation_eps = p.rotation_eps;
  d.lm_init_lambda_factor = p.lm_init_lambda_factor;
  d.icp_score_thr = p.icp_score_thr;
  return d;
}

struct PairWork {  // device memory comes from the caller's Scratch and goes back with it
  std::vector<PairDev> pairs;
  PairDev* d_pairs = nullptr;     // only with own_arrays (the debug taps): scratch copies of the solve's argument arrays
  PairState* d_states = nullptr;
  LmSched* d_sched = nullptr;
  LmCall* d_call = nullptr;
  LmSched sched_host;  // staging for the header upload (lives as long as the PairWork)
  LmCall call_host;
  int max_n = 0;
  long total_blocks = 0;  // work items of one step with every pair active
};

static int make_pair_work(b200reg_ctx* c, int count, b200reg_cloud* const* src, b200reg_cloud* const* tgt, PairWork& w, Scratch& scratch,
                          bool own_arrays, const GicpParamsDev* prm) {
  cudaStream_t s = c->stream;
  w.pairs.resize(count);
  for (int i = 0; i < count; i++) {
    PairDev& p = w.pairs[i];
    p.src = src[i]->dev;
    p.tgt = tgt[i]->dev;
    const int N = p.src.n;
    const int nblk = (N + STEP_THREADS - 1) / STEP_THREADS;
    size_t o_corr = 0;
    size_t o_sqd = align_up(o_corr + (size_t)N * 4, 256);
    size_t o_mah = align_up(o_sqd + (size_t)N * 4, 256);
    size_t o_par = align_up(o_mah + (size_t)N * 6 * 8, 256);
    size_t total = align_up(o_par + (size_t)((N + 31) / 32) * NRED * 8, 256);
    char* slab = nullptr;
    CU(scratch.alloc((void**)&slab, total));
    p.corr = (int*)(slab + o_corr);
    p.sqd = (float*)(slab + o_sqd);
    p.mahal = (double*)(slab + o_mah);
    p.partial = (double*)(slab + o_par);
    w.max_n = std::max(w.max_n, N);
    w.total_blocks += nblk;
  }
  if (!own_arrays) return B200REG_OK;  // b200reg_gicp_align: the argument arrays live in the context's LM arena
  CU(scratch.alloc((void**)&w.d_pairs, sizeof(PairDev) * count));
  CU(scratch.alloc((void**)&w.d_states, sizeof(PairState) * count));
  CU(cudaMemsetAsync(w.d_states, 0, sizeof(PairState) * count, c->stream));
  CU(scratch.alloc((void**)&w.d_call, sizeof(LmCall)));
  memset(&w.call_host, 0, sizeof(LmCall));
  w.call_host.count = count;
  w.call_host.has_guess = 1;
  w.call_host.max_steps = 1 << 30;
  w.call_host.prm = *prm;
  CU(cudaMemcpyAsync(w.d_call, &w.call_host, sizeof(LmCall), cudaMemcpyHostToDevice, s));
  {  // schedule header + slots[count]
    char* sm = nullptr;
    CU(scratch.alloc((void**)&sm, 64 + sizeof(LmSlot) * (size_t)count));
    LmSched hs;
    memset(&hs, 0, sizeof(hs));
    hs.slots = (LmSlot*)(sm + 64);
    w.d_sched = (LmSched*)sm;
    static_assert(sizeof(LmSched) <= 64, "LmSched header");
    w.sched_host = hs;
    CU(cudaMemcpyAsync(w.d_sched, &w.sched_host, sizeof(LmSched), cudaMemcpyHostToDevice, s));
  }
  CU(cudaMemcpyAsync(w.d_pairs, w.pairs.data(), sizeof(PairDev) * count, cudaMemcpyHostToDevice, s));
  return B200REG_OK;
}

int b200reg_gicp_align(b200reg_ctx* c, int count, b200reg_cloud* const* src, b200reg_cloud* const* tgt,
                       const double* guess16, const b200reg_gicp_params* params, b200reg_result* out) {
  if (!c || count <= 0 || !src || !tgt || !params || !out) return fail(B200REG_EINVAL, "bad argument");
  CU(cudaSetDevice(c->device));
  cudaStream_t s = c->stream;
  Scratch scratch(c);
  int rc;
  // covariances on demand (nano_gicp_impl.hpp:162-167)
  {
    std::vector<b200reg_cloud*> need;
    for (int i = 0; i < count; i++) {
      if (!src[i] || !tgt[i]) return fail(B200REG_EINVAL, "NULL cloud");
      const int m = params->regularization;
      auto stale = [&](const b200reg_cloud* cl) {
        return !cl->has_cov || (!cl->cov_user && (cl->cov_k != params->k_correspondences || cl->cov_method != m));
      };
      if (stale(src[i])) need.push_back(src[i]);
      if (stale(tgt[i])) need.push_back(tgt[i]);
    }
    if (!need.empty() &&
        (rc = b200reg_clouds_covariances_ex(c, (int)need.size(), need.data(), params->k_correspondences, params->regularization)))
      return rc;
  }
  const GicpParamsDev prm = to_dev(*params);
  PairWork w;
  if ((rc = make_pair_work(c, count, src, tgt, w, scratch, false, nullptr))) return rc;
  if ((rc = lm_arena_ensure(c, count))) return rc;
  auto& A = c->lm;
  // per-call inputs of the graph: pair descriptors, guesses, the call record
  CU(cudaMemcpyAsync(A.d_pairs, w.pairs.data(), sizeof(PairDev) * count, cudaMemcpyHostToDevice, s));
  if (guess16) CU(cudaMemcpyAsync(A.d_guess, guess16, sizeof(double) * 16 * count, cudaMemcpyHostToDevice, s));
  LmCall& hc = *A.h_call;
  memset(&hc, 0, sizeof(hc));
  hc.count = count;
  hc.has_guess = guess16 ? 1 : 0;
  // worst case: every outer iteration burns lm_max_iterations trials, plus the fitness pass
  hc.max_steps = std::max(params->max_iterations, 0) * (1 + std::max(params->lm_max_iterations, 1)) + 2;
  hc.cond_handle = A.graph.cond_handle;
  hc.prm = prm;
  CU(cudaMemcpyAsync(A.d_call, A.h_call, sizeof(LmCall), cudaMemcpyHostToDevice, s));
  static const bool env_no_graph = getenv("B200REG_LM_NO_GRAPH") != nullptr;  // Nsight Compute does not list kernels that run
  const bool no_graph = env_no_graph || c->profiling;                          // inside a conditional graph node
  if (no_graph) {
    // Profiling / ncu aid: the SAME kernels launched one by one, the host polling the schedule (what the while node does
    // on the device), each kernel bracketed by its own CUDA events
    A.h_call->cond_handle = 0;
    CU(cudaMemcpyAsync(A.d_call, A.h_call, sizeof(LmCall), cudaMemcpyHostToDevice, s));
    launch_gicp_init(A.d_pairs, A.d_states, A.d_guess, A.d_call, A.d_sched, s);
    for (;;) {
      LmSched hs;
      CU(cudaMemcpyAsync(&hs, A.d_sched, sizeof(LmSched), cudaMemcpyDeviceToHost, s));
      CU(cudaStreamSynchronize(s));
      if (hs.n_active == 0 || hs.steps > hc.max_steps) break;
      {
        ProfScope ps(c, CLS_SEARCH);
        launch_gicp_search(A.d_pairs, A.d_states, c->sm_count * 32, A.d_call, A.d_sched, s);
        c->launches++;
      }
      {
        ProfScope ps(c, CLS_ACCUM);
        launch_gicp_accum(A.d_pairs, A.d_states, c->sm_count * 32, A.d_sched, s);
        c->launches++;
      }
      {
        ProfScope ps(c, CLS_CTRL);
        launch_gicp_control(A.d_pairs, A.d_states, A.d_call, A.d_sched, s);
        c->launches++;
      }
    }
    c->launches++;
  } else {
    // init kernel + device-side while loop over {search, accumulate, control}: ONE launch, ONE synchronisation per solve
    ProfScope ps(c, CLS_STEP);
    CU(cudaGraphLaunch(A.graph.exec, s));
  }
  PairState* states = A.h_states;
  CU(cudaMemcpyAsync(states, A.d_states, sizeof(PairState) * count, cudaMemcpyDeviceToHost, s));
  CU(cudaMemcpyAsync(A.h_call, A.d_call, sizeof(LmCall), cudaMemcpyDeviceToHost, s));
  LmSched hsched;
  CU(cudaMemcpyAsync(&hsched, A.d_sched, sizeof(LmSched), cudaMemcpyDeviceToHost, s));
  CU(cudaStreamSynchronize(s));
  if (!no_graph) c->launches += 1 + 3 * (int64_t)hsched.steps;  // init + (search, accumulate, control) per executed step, counted by the device
  if (A.h_call->overrun) return fail(B200REG_ESTATE, "LM state machine did not terminate");
  for (int i = 0; i < count; i++) {
    const PairState& st = states[i];
    b200reg_result& r = out[i];
    memset(&r, 0, sizeof(r));
    for (int a = 0; a < 3; a++) {
      for (int b = 0; b < 3; b++) r.T[4 * a + b] = st.R[3 * a + b];
      r.T[4 * a + 3] = st.t[a];
    }
    r.T[15] = 1.0;
    for (int a = 0; a < 12; a++) r.Tf[a] = st.Tf[a];
    r.Tf[15] = 1.0f;
    if (st.n_lin > 0) memcpy(r.final_hessian, st.H, sizeof(r.final_hessian));
    else for (int a = 0; a < 6; a++) r.final_hessian[7 * a] = 1.0;  // final_hessian_.setIdentity() (lsq_registration_impl.hpp:62)
    r.fitness = st.fitness;
    r.converged = st.converged;
    r.valid = (st.converged && st.fitness < params->icp_score_thr) ? 1 : 0;
    for (int a = 0; a < 16; a++) r.pose_between[a] = (a % 5 == 0) ? 1.0 : 0.0;  // RegistrationOutput default (loop_closure.h:64-70)
    if (r.valid)  // getFinalTransformation().cast<double>() (loop_closure.cpp:133)
      for (int a = 0; a < 12; a++) r.pose_between[a] = (double)st.Tf[a];
    r.iterations = st.nr_iterations;
    r.n_linearize = st.n_lin;
    r.n_error = st.n_err;
    r.lm_failed = st.lm_failed;
    r.status = 0;
    // SURVEY §8(d): K3 136*N per linearize, K4 132*N per compute_error, K5 16*N fitness.  Per kernel: the search reads the
    // 16-byte points and writes the 8-byte correspondence record (24*N of K3; all 16*N of K5), the accumulate pass owns the rest
    const double N = w.pairs[i].src.n;
    if (no_graph) {
      c->prof_bytes[CLS_SEARCH] += (24.0 * st.n_lin + 16.0) * N;
      c->prof_bytes[CLS_ACCUM] += (112.0 * st.n_lin + 132.0 * st.n_err) * N;
    } else {
      c->prof_bytes[CLS_STEP] += (136.0 * st.n_lin + 132.0 * st.n_err + 16.0) * N;
    }
  }
  return B200REG_OK;
}

// one chunk of pairs, raw records already on the device
static int icp_alignment_device(b200reg_ctx* c, int count, const float* const* src_xyz, const size_t* src_n,
                                const float* const* tgt_xyz, const size_t* tgt_n, size_t stride_bytes,
                                const b200reg_gicp_params* params, b200reg_result* out) {
  std::vector<const float*> ptrs(2 * count);
  std::vector<size_t> ns(2 * count);
  for (int i = 0; i < count; i++) {
    ptrs[i] = src_xyz[i];
    ns[i] = src_n[i];
    ptrs[count + i] = tgt_xyz[i];
    ns[count + i] = tgt_n[i];
  }
  std::vector<b200reg_cloud*> clouds(2 * count, nullptr);
  int rc = b200reg_clouds_create(c, 2 * count, ptrs.data(), ns.data(), stride_bytes, 1, clouds.data());
  if (rc) return rc;
  rc = b200reg_clouds_covariances_ex(c, 2 * count, clouds.data(), params->k_correspondences, params->regularization);
  if (!rc) rc = b200reg_gicp_align(c, count, clouds.data(), clouds.data() + count, nullptr, params, out);
  for (b200reg_cloud* cl : clouds) b200reg_cloud_destroy(c, cl);
  return rc;
}

int b200reg_icp_alignment(b200reg_ctx* c, int count, const float* const* src_xyz, const size_t* src_n,
                          const float* const* tgt_xyz, const size_t* tgt_n, size_t stride_bytes, int on_device,
                          const b200reg_gicp_params* params, b200reg_result* out) {
  if (!c || count <= 0 || !src_xyz || !src_n || !tgt_xyz || !tgt_n || !params || !out)
    return fail(B200REG_EINVAL, "bad argument");
  if (stride_bytes < 12 || stride_bytes % 4) return fail(B200REG_EINVAL, "stride_bytes must be a multiple of 4, >= 12");
  for (int i = 0; i < count; i++)
    if (!src_xyz[i] || !tgt_xyz[i] || src_n[i] == 0 || tgt_n[i] == 0) return fail(B200REG_EINVAL, "empty cloud");
  CU(cudaSetDevice(c->device));
  if (on_device) return icp_alignment_device(c, count, src_xyz, src_n, tgt_xyz, tgt_n, stride_bytes, params, out);
  // Host buffers: all uploads are queued on the copy stream up front, chunk by chunk; the compute stream processes
  // chunk k as soon as its records have landed, so the PCIe time of chunk k+1 hides behind the kernels of chunk k.
  cudaStream_t s = c->stream;
  Scratch scratch(c);
  int want = c->pipeline_chunks;
  if (const char* e = getenv("B200REG_PIPELINE_CHUNKS")) want = atoi(e);
  const int nchunks = std::max(1, std::min(want, count));
  const int per = (count + nchunks - 1) / nchunks;
  size_t total = 0;
  std::vector<size_t> off_s(count), off_t(count);
  for (int i = 0; i < count; i++) {
    off_s[i] = total;
    total += align_up(src_n[i] * stride_bytes, 256);
    off_t[i] = total;
    total += align_up(tgt_n[i] * stride_bytes, 256);
  }
  char* stage = nullptr;
  CU(scratch.alloc((void**)&stage, total));
  EventBag events;
  struct CopyDrain {  // the uploads read the caller's buffers: they must have finished whenever this call returns
    cudaStream_t cs;
    ~CopyDrain() { cudaStreamSynchronize(cs); }
  } drain{c->copy_stream};
  cudaEvent_t ready;
  CU(events.make(&ready));
  CU(cudaEventRecord(ready, s));
  CU(cudaStreamWaitEvent(c->copy_stream, ready, 0));
  std::vector<cudaEvent_t> landed;
  for (int k0 = 0; k0 < count; k0 += per) {
    const int k1 = std::min(count, k0 + per);
    for (int i = k0; i < k1; i++) {
      CU(cudaMemcpyAsync(stage + off_s[i], src_xyz[i], src_n[i] * stride_bytes, cudaMemcpyHostToDevice, c->copy_stream));
      CU(cudaMemcpyAsync(stage + off_t[i], tgt_xyz[i], tgt_n[i] * stride_bytes, cudaMemcpyHostToDevice, c->copy_stream));
    }
    cudaEvent_t e;
    CU(events.make(&e));
    CU(cudaEventRecord(e, c->copy_stream));
    landed.push_back(e);
  }
  // index build + covariances chunk by chunk (they only need that chunk's records), then ONE batched LM solve over
  // all pairs: the host never blocks before the solve's first poll, so the GPU stays busy while later chunks land.
  int rc = B200REG_OK;
  int chunk = 0;
  std::vector<b200reg_cloud*> sc(count, nullptr), tc(count, nullptr);
  CloudBag bag(c);
  for (int k0 = 0; k0 < count && !rc; k0 += per, chunk++) {
    const int k1 = std::min(count, k0 + per), m = k1 - k0;
    CU(cudaStreamWaitEvent(s, landed[chunk], 0));
    std::vector<const float*> ptrs(2 * m);
    std::vector<size_t> ns(2 * m);
    std::vector<b200reg_cloud*> cl(2 * m, nullptr);
    for (int i = k0; i < k1; i++) {
      ptrs[i - k0] = (const float*)(stage + off_s[i]);
      ns[i - k0] = src_n[i];
      ptrs[m + i - k0] = (const float*)(stage + off_t[i]);
      ns[m + i - k0] = tgt_n[i];
    }
    rc = b200reg_clouds_create(c, 2 * m, ptrs.data(), ns.data(), stride_bytes, 1, cl.data());
    for (b200reg_cloud* p : cl)
      if (p) bag.cl.push_back(p);
    for (int i = k0; i < k1; i++) {
      sc[i] = cl[i - k0];
      tc[i] = cl[m + i - k0];
    }
    if (!rc) rc = b200reg_clouds_covariances_ex(c, 2 * m, cl.data(), params->k_correspondences, params->regularization);
  }
  if (!rc) rc = b200reg_gicp_align(c, count, sc.data(), tc.data(), nullptr, params, out);
  return rc;  // clouds, events and the copy stream are released / drained by the scope guards
}

int b200reg_transform_cloud(b200reg_ctx* c, const b200reg_cloud* cl, const float* Tf16, float* out_xyz) {
  if (!c || !cl || !Tf16 || !out_xyz) return fail(B200REG_EINVAL, "bad argument");
  CU(cudaSetDevice(c->device));
  cudaStream_t s = c->stream;
  Scratch scratch(c);
  float* d_T = nullptr;
  float* d_out = nullptr;
  CU(scratch.alloc((void**)&d_T, 64));
  CU(scratch.alloc((void**)&d_out, (size_t)cl->dev.n * 12));
  CU(cudaMemcpyAsync(d_T, Tf16, 64, cudaMemcpyHostToDevice, s));
  launch_transform_out(cl->dev, d_T, d_out, s);
  c->launches++;
  CU(cudaMemcpyAsync(out_xyz, d_out, (size_t)cl->dev.n * 12, cudaMemcpyDeviceToHost, s));
  CU(cudaStreamSynchronize(s));
  return B200REG_OK;
}

// ---- debug taps --------------------------------------------------------------------------
static int knn_impl(b200reg_ctx* c, const b200reg_cloud* cl, const float* queries, size_t nq, size_t qstride_bytes, int k,
                    int32_t* idx_out, float* d2_out, int brute);

int b200reg_knn(b200reg_ctx* c, const b200reg_cloud* cl, const float* queries, size_t nq, size_t qstride_bytes, int k,
                int32_t* idx_out, float* d2_out) {
  return knn_impl(c, cl, queries, nq, qstride_bytes, k, idx_out, d2_out, 0);
}

int b200reg_knn_bruteforce(b200reg_ctx* c, const b200reg_cloud* cl, const float* queries, size_t nq, size_t qstride_bytes, int k,
                           int32_t* idx_out, float* d2_out) {
  return knn_impl(c, cl, queries, nq, qstride_bytes, k, idx_out, d2_out, 1);
}

static int knn_impl(b200reg_ctx* c, const b200reg_cloud* cl, const float* queries, size_t nq, size_t qstride_bytes, int k,
                    int32_t* idx_out, float* d2_out, int brute) {
  if (!c || !cl || !queries || nq == 0 || k <= 0 || k > 32 || !idx_out || !d2_out || qstride_bytes < 12 || qstride_bytes % 4)
    return fail(B200REG_EINVAL, "bad argument (k must be 1..32)");
  CU(cudaSetDevice(c->device));
  cudaStream_t s = c->stream;
  Scratch scratch(c);
  float* d_q = nullptr;
  int* d_idx = nullptr;
  float* d_d2 = nullptr;
  CU(scratch.alloc((void**)&d_q, nq * qstride_bytes));
  CU(scratch.alloc((void**)&d_idx, nq * k * 4));
  CU(scratch.alloc((void**)&d_d2, nq * k * 4));
  CU(cudaMemcpyAsync(d_q, queries, nq * qstride_bytes, cudaMemcpyHostToDevice, s));
  if (launch_knn_queries(cl->dev, d_q, (int)nq, (int)(qstride_bytes / 4), k, d_idx, d_d2, s, brute) < 0)
    return fail(B200REG_EINVAL, "unsupported k");
  c->launches++;
  CU(cudaGetLastError());
  CU(cudaMemcpyAsync(idx_out, d_idx, nq * k * 4, cudaMemcpyDeviceToHost, s));
  CU(cudaMemcpyAsync(d2_out, d_d2, nq * k * 4, cudaMemcpyDeviceToHost, s));
  CU(cudaStreamSynchronize(s));
  return B200REG_OK;
}

int b200reg_get_covariances(b200reg_ctx* c, const b200reg_cloud* cl, double* cov9_out) {
  if (!c || !cl || !cov9_out) return fail(B200REG_EINVAL, "bad argument");
  if (!cl->has_cov) return fail(B200REG_ESTATE, "covariances not computed");
  CU(cudaSetDevice(c->device));
  cudaStream_t s = c->stream;
  const int n = cl->dev.n;
  std::vector<double> cov((size_t)n * 6);
  std::vector<float4> pts(n);
  CU(cudaMemcpyAsync(cov.data(), cl->dev.cov, (size_t)n * 48, cudaMemcpyDeviceToHost, s));
  CU(cudaMemcpyAsync(pts.data(), cl->dev.pts, (size_t)n * 16, cudaMemcpyDeviceToHost, s));
  CU(cudaStreamSynchronize(s));
  for (int p = 0; p < n; p++) {
    int o;
    memcpy(&o, &pts[p].w, 4);
    const double* a = &cov[(size_t)p * 6];
    double* m = &cov9_out[(size_t)o * 9];
    m[0] = a[0]; m[1] = a[1]; m[2] = a[2];
    m[3] = a[1]; m[4] = a[3]; m[5] = a[4];
    m[6] = a[2]; m[7] = a[4]; m[8] = a[5];
  }
  return B200REG_OK;
}

int b200reg_linearize(b200reg_ctx* c, const b200reg_cloud* src, const b200reg_cloud* tgt, const double* T16,
                      double max_corr_dist, double* H36, double* b6, double* err, int32_t* corr_out, float* sqd_out) {
  if (!c || !src || !tgt || !T16) return fail(B200REG_EINVAL, "bad argument");
  if (!src->has_cov || !tgt->has_cov) return fail(B200REG_ESTATE, "covariances not computed");
  CU(cudaSetDevice(c->device));
  cudaStream_t s = c->stream;
  Scratch scratch(c);
  PairWork w;
  b200reg_cloud* sp = const_cast<b200reg_cloud*>(src);
  b200reg_cloud* tp = const_cast<b200reg_cloud*>(tgt);
  int rc;
  b200reg_gicp_params p;
  b200reg_default_gicp_params(&p);
  p.max_corr_dist = max_corr_dist;
  const GicpParamsDev prm = to_dev(p);
  if ((rc = make_pair_work(c, 1, &sp, &tp, w, scratch, true, &prm))) return rc;
  double* d_guess = nullptr;
  CU(scratch.alloc((void**)&d_guess, sizeof(double) * 16));
  CU(cudaMemcpyAsync(d_guess, T16, sizeof(double) * 16, cudaMemcpyHostToDevice, s));
  launch_gicp_init(w.d_pairs, w.d_states, d_guess, w.d_call, w.d_sched, s);
  const int tap_blocks = (int)std::min(w.total_blocks, (long)c->sm_count * 8);
  c->launches += 1 + launch_gicp_step(w.d_pairs, w.d_states, tap_blocks, tap_blocks, w.d_call, w.d_sched, s);  // exactly one linearize pass
  PairState st;
  const int N = src->dev.n, M = tgt->dev.n;
  std::vector<int> corr(N);
  std::vector<float> sqd(N);
  std::vector<float4> sp_pts(N), tp_pts(M);
  CU(cudaMemcpyAsync(&st, w.d_states, sizeof(PairState), cudaMemcpyDeviceToHost, s));
  CU(cudaMemcpyAsync(corr.data(), w.pairs[0].corr, (size_t)N * 4, cudaMemcpyDeviceToHost, s));
  CU(cudaMemcpyAsync(sqd.data(), w.pairs[0].sqd, (size_t)N * 4, cudaMemcpyDeviceToHost, s));
  CU(cudaMemcpyAsync(sp_pts.data(), src->dev.pts, (size_t)N * 16, cudaMemcpyDeviceToHost, s));
  CU(cudaMemcpyAsync(tp_pts.data(), tgt->dev.pts, (size_t)M * 16, cudaMemcpyDeviceToHost, s));
  CU(cudaStreamSynchronize(s));
  if (H36) memcpy(H36, st.H, sizeof(double) * 36);
  if (b6) memcpy(b6, st.b, sizeof(double) * 6);
  if (err) *err = st.y0;
  for (int p_ = 0; p_ < N; p_++) {
    int o, to = -1;
    memcpy(&o, &sp_pts[p_].w, 4);
    if (corr[p_] >= 0) memcpy(&to, &tp_pts[corr[p_]].w, 4);
    if (corr_out) corr_out[o] = to;
    if (sqd_out) sqd_out[o] = sqd[p_];
  }
  return B200REG_OK;
}

int b200reg_compute_error(b200reg_ctx* c, const b200reg_cloud* src, const b200reg_cloud* tgt, const double* T_lin16,
                          const double* T_trial16, double max_corr_dist, double* err) {
  if (!c || !src || !tgt || !T_lin16 || !T_trial16 || !err) return fail(B200REG_EINVAL, "bad argument");
  if (!src->has_cov || !tgt->has_cov) return fail(B200REG_ESTATE, "covariances not computed");
  CU(cudaSetDevice(c->device));
  cudaStream_t s = c->stream;
  Scratch scratch(c);
  PairWork w;
  b200reg_cloud* sp = const_cast<b200reg_cloud*>(src);
  b200reg_cloud* tp = const_cast<b200reg_cloud*>(tgt);
  int rc;
  b200reg_gicp_params p;
  b200reg_default_gicp_params(&p);
  p.max_corr_dist = max_corr_dist;
  const GicpParamsDev prm = to_dev(p);
  if ((rc = make_pair_work(c, 1, &sp, &tp, w, scratch, true, &prm))) return rc;
  double* d_guess = nullptr;
  CU(scratch.alloc((void**)&d_guess, sizeof(double) * 16));
  CU(cudaMemcpyAsync(d_guess, T_lin16, sizeof(double) * 16, cudaMemcpyHostToDevice, s));
  const int blocks = (int)std::min(w.total_blocks, (long)c->sm_count * 8);
  launch_gicp_init(w.d_pairs, w.d_states, d_guess, w.d_call, w.d_sched, s);
  launch_gicp_step(w.d_pairs, w.d_states, blocks, blocks, w.d_call, w.d_sched, s);  // linearize: correspondences + Mahalanobis, phase -> TRIAL
  // overwrite the trial pose the LM controller prepared with the caller's
  double Rt[9], tt[3];
  for (int a = 0; a < 3; a++) {
    for (int b = 0; b < 3; b++) Rt[3 * a + b] = T_trial16[4 * a + b];
    tt[a] = T_trial16[4 * a + 3];
  }
  CU(cudaMemcpyAsync((char*)w.d_states + offsetof(PairState, Rt), Rt, sizeof(Rt), cudaMemcpyHostToDevice, s));
  CU(cudaMemcpyAsync((char*)w.d_states + offsetof(PairState, tt), tt, sizeof(tt), cudaMemcpyHostToDevice, s));
  launch_gicp_step(w.d_pairs, w.d_states, blocks, blocks, w.d_call, w.d_sched, s);  // compute_error at the trial pose
  c->launches += 7;
  PairState st;
  CU(cudaMemcpyAsync(&st, w.d_states, sizeof(PairState), cudaMemcpyDeviceToHost, s));
  CU(cudaStreamSynchronize(s));
  *err = st.y_trial;
  return B200REG_OK;
}


// ---- Quatro ------------------------------------------------------------------------------
void b200reg_default_quatro_params(b200reg_quatro_params* p) {
  if (!p) return;
  p->fpfh_normal_radius = 0.9;
  p->fpfh_radius = 1.5;
  p->noise_bound = 0.3;
  p->rot_gnc_factor = 1.4;
  p->rot_cost_thr = 1e-4;
  p->rot_max_iter = 50;
  p->max_corres = 200;
  p->distance_threshold = 35.0;
  p->tuple_scale = 0.95;
  p->seed = 1;
  p->estimate_scale = 0;
  p->use_optimized_matching = 1;
}

int b200reg_clouds_fpfh(b200reg_ctx* c, int count, b200reg_cloud* const* clouds, double normal_radius, double fpfh_radius) {
  if (!c || count <= 0 || !clouds || !(normal_radius > 0) || !(fpfh_radius > 0)) return fail(B200REG_EINVAL, "bad argument");
  CU(cudaSetDevice(c->device));
  cudaStream_t s = c->stream;
  Scratch scratch(c);
  std::vector<CloudDev> descs;
  std::vector<b200reg_cloud*> todo;
  int max_n = 0;
  for (int i = 0; i < count; i++) {
    b200reg_cloud* cl = clouds[i];
    if (!cl) return fail(B200REG_EINVAL, "NULL cloud");
    if (cl->has_fpfh && cl->normal_r == normal_radius && cl->fpfh_r == fpfh_radius) continue;
    if (std::find(todo.begin(), todo.end(), cl) != todo.end()) continue;
    if (!cl->fslab) {
      const size_t n = cl->dev.n;
      size_t o_n = 0;
      size_t o_s = align_up(o_n + n * sizeof(float4), 256);
      size_t o_f = align_up(o_s + n * FPAD * sizeof(float), 256);
      size_t o_fn = align_up(o_f + n * FPAD * sizeof(float), 256);
      size_t o_fns = align_up(o_fn + n * sizeof(float4), 256);
      size_t o_ft = align_up(o_fns + n * sizeof(float4), 256);
      size_t o_fc = align_up(o_ft + 2 * ((n + 63) / 64) * sizeof(float4), 256);
      size_t total = align_up(o_fc + n * sizeof(uint32_t), 256);
      char* fs = nullptr;
      CU(cudaMallocFromPoolAsync((void**)&fs, total, c->pool, s));
      cl->fslab = fs;
      cl->dev.nrm = (float4*)(fs + o_n);
      cl->dev.spfh = (float*)(fs + o_s);
      cl->dev.fpfh = (float*)(fs + o_f);
      cl->dev.fproj = (float4*)(fs + o_fn);
      cl->dev.fpfh_s = cl->dev.spfh;  // the SPFH table is dead once k_fpfh has consumed it
      cl->dev.fproj_s = (float4*)(fs + o_fns);
      cl->dev.ftile = (float4*)(fs + o_ft);
      cl->dev.fcode_s = (uint32_t*)(fs + o_fc);
    }
    todo.push_back(cl);
    descs.push_back(cl->dev);
    max_n = std::max(max_n, cl->dev.n);
  }
  if (todo.empty()) return B200REG_OK;
  {  // sort buffers of the filter-code ordering (scratch: only this call uses them); the work memory of all clouds is one
     // region, zeroed by one memset
    size_t ws_total = 0, k_total = 0;
    for (auto& d : descs) {
      ws_total += align_up(radix_sort_ws_bytes(d.n, 32), 256);
      k_total += 4 * align_up((size_t)d.n * 4, 256);
    }
    char* sb = nullptr;
    CU(scratch.alloc((void**)&sb, ws_total + k_total));
    CU(cudaMemsetAsync(sb, 0, ws_total, s));
    char* ws = sb;
    char* kb = sb + ws_total;
    for (auto& d : descs) {
      const size_t s_k = align_up((size_t)d.n * 4, 256);
      d.hist = (uint32_t*)ws;
      ws += align_up(radix_sort_ws_bytes(d.n, 32), 256);
      d.keys[0] = (uint32_t*)kb;
      d.keys[1] = (uint32_t*)(kb + s_k);
      d.vals[0] = (uint32_t*)(kb + 2 * s_k);
      d.vals[1] = (uint32_t*)(kb + 3 * s_k);
      kb += 4 * s_k;
    }
  }
  CloudDev* d_descs = nullptr;
  CU(scratch.alloc((void**)&d_descs, sizeof(CloudDev) * descs.size()));
  CU(cudaMemcpyAsync(d_descs, descs.data(), sizeof(CloudDev) * descs.size(), cudaMemcpyHostToDevice, s));
  {
    ProfScope ps(c, CLS_FPFH);
    const float nr2 = (float)(normal_radius * normal_radius), fr2 = (float)(fpfh_radius * fpfh_radius);
    c->launches += launch_fpfh(d_descs, (int)descs.size(), max_n, nr2, fr2, s);
    for (auto& d : descs) c->prof_bytes[CLS_FPFH] += (32.0 + 164.0 + 280.0) * d.n;  // SURVEY §8(d) Q1+Q2+Q3
  }
  CU(cudaGetLastError());
  for (b200reg_cloud* cl : todo) {
    cl->has_fpfh = true;
    cl->normal_r = normal_radius;
    cl->fpfh_r = fpfh_radius;
  }
  return B200REG_OK;
}

int b200reg_get_fpfh(b200reg_ctx* c, const b200reg_cloud* cl, float* normals_out, float* fpfh_out) {
  if (!c || !cl) return fail(B200REG_EINVAL, "bad argument");
  if (!cl->has_fpfh) return fail(B200REG_ESTATE, "FPFH not computed");
  CU(cudaSetDevice(c->device));
  cudaStream_t s = c->stream;
  const int n = cl->dev.n;
  std::vector<float4> pts(n), nrm(n);
  std::vector<float> f((size_t)n * FPAD);
  CU(cudaMemcpyAsync(pts.data(), cl->dev.pts, (size_t)n * 16, cudaMemcpyDeviceToHost, s));
  CU(cudaMemcpyAsync(nrm.data(), cl->dev.nrm, (size_t)n * 16, cudaMemcpyDeviceToHost, s));
  CU(cudaMemcpyAsync(f.data(), cl->dev.fpfh, (size_t)n * FPAD * 4, cudaMemcpyDeviceToHost, s));
  CU(cudaStreamSynchronize(s));
  for (int p = 0; p < n; p++) {
    int o;
    memcpy(&o, &pts[p].w, 4);
    if (normals_out) {
      const bool ok = nrm[p].w != 0.f;
      normals_out[3 * (size_t)o + 0] = ok ? nrm[p].x : NAN;
      normals_out[3 * (size_t)o + 1] = ok ? nrm[p].y : NAN;
      normals_out[3 * (size_t)o + 2] = ok ? nrm[p].z : NAN;
    }
    if (fpfh_out) memcpy(&fpfh_out[(size_t)o * FDIM], &f[(size_t)p * FPAD], FDIM * sizeof(float));
  }
  return B200REG_OK;
}

int b200reg_quatro_align(b200reg_ctx* c, int count, b200reg_cloud* const* src, b200reg_cloud* const* dst,
                         const b200reg_quatro_params* prm, b200reg_quatro_info* out, int32_t* corr_out) {
  if (!c || count <= 0 || !src || !dst || !prm || !out) return fail(B200REG_EINVAL, "bad argument");
  if (prm->estimate_scale) return fail(B200REG_EINVAL, "estimate_scale is not supported (the deployment sets it false)");
  const bool advanced = !prm->use_optimized_matching;  // Matcher::advancedMatching (matcher.cc:118-356)
  if (!advanced && (prm->max_corres < 1 || prm->max_corres > MAXC - 3)) return fail(B200REG_EINVAL, "max_corres must be in 1..509");
  const int corr_stride = advanced ? BIGC : MAXC;  // B200REG_ADV_CORR_CAPACITY / B200REG_CORR_CAPACITY
  CU(cudaSetDevice(c->device));
  cudaStream_t s = c->stream;
  Scratch scratch(c);
  int rc;
  {
    std::vector<b200reg_cloud*> all;
    for (int i = 0; i < count; i++) {
      if (!src[i] || !dst[i]) return fail(B200REG_EINVAL, "NULL cloud");
      all.push_back(src[i]);
      all.push_back(dst[i]);
    }
    if ((rc = b200reg_clouds_fpfh(c, (int)all.size(), all.data(), prm->fpfh_normal_radius, prm->fpfh_radius))) return rc;
  }
  std::vector<MatchDev> pairs(count);
  std::vector<BigSolveWs> big_host;
  big_host.reserve(count);  // addresses stay valid for the async copies below
  int max_ni = 0, max_nj = 0;
  for (int i = 0; i < count; i++) {
    MatchDev& m = pairs[i];
    const bool swapped = dst[i]->dev.n > src[i]->dev.n;  // fi = larger cloud (matcher.cc:364-369)
    m.fi = swapped ? dst[i]->dev : src[i]->dev;
    m.fj = swapped ? src[i]->dev : dst[i]->dev;
    m.swapped = swapped ? 1 : 0;
    const size_t ni = m.fi.n, nj = m.fj.n;
    size_t o = 0;
    auto take = [&](size_t bytes) {
      size_t r = o;
      o = align_up(o + bytes, 256);
      return r;
    };
    const size_t o_nn = take(nj * 4), o_dis = take(nj * 4), o_fj = take(ni * 4), o_rnn = take(ni * 4);
    // advancedMatching: the cross-checked set has at most nj members; the solver workspace is sized for the next
    // power of two (>= 1024, <= BIGC)
    int cap = 1024;
    while (advanced && cap < (int)nj && cap < BIGC) cap <<= 1;
    const size_t o_cor = take(2 * nj * 4), o_tk = take(nj * 4), o_cnt = take(8 * 4), o_st = take(8 * 8),
                 o_oc = take(2 * (size_t)(advanced ? cap : MAXC) * 4), o_T = take(16 * 8);
    const size_t words = cap / 32;
    size_t o_big = 0, o_S = 0, o_D = 0, o_adj = 0, o_radj = 0, o_int = 0, o_skey = 0, o_w = 0, o_res = 0, o_hval = 0, o_hidx = 0;
    if (advanced) {
      o_big = take(sizeof(BigSolveWs));
      o_S = take((size_t)cap * 24);
      o_D = take((size_t)cap * 24);
      o_adj = take((size_t)cap * words * 4);
      o_radj = take((size_t)cap * words * 4);
      o_int = take((size_t)cap * 4 * 9);
      o_skey = take((size_t)cap * 8);
      o_w = take((size_t)cap * 8);
      o_res = take((size_t)cap * 8);
      o_hval = take((size_t)cap * 16);
      o_hidx = take((size_t)cap * 8);
    }
    char* slab = nullptr;
    CU(scratch.alloc((void**)&slab, o));
    m.nn = (int*)(slab + o_nn);
    m.dis = (float*)(slab + o_dis);
    m.first_j = (int*)(slab + o_fj);
    m.rnn = (int*)(slab + o_rnn);
    m.corres = (int*)(slab + o_cor);
    m.tkey = (unsigned*)(slab + o_tk);
    m.counters = (int*)(slab + o_cnt);
    m.stats = (double*)(slab + o_st);
    m.out_corr = (int*)(slab + o_oc);
    m.T = (double*)(slab + o_T);
    m.big = nullptr;
    if (advanced) {
      BigSolveWs w;
      w.cap = cap;
      w.words = (int)words;
      w.S = (double*)(slab + o_S);
      w.D = (double*)(slab + o_D);
      w.adj = (unsigned*)(slab + o_adj);
      w.radj = (unsigned*)(slab + o_radj);
      int* ip = (int*)(slab + o_int);
      w.deg = ip; w.pdeg = ip + cap; w.core = ip + 2 * (size_t)cap; w.alive = ip + 3 * (size_t)cap; w.rank = ip + 4 * (size_t)cap;
      w.order = ip + 5 * (size_t)cap; w.csize = ip + 6 * (size_t)cap; w.clique = ip + 7 * (size_t)cap; w.list = ip + 8 * (size_t)cap;
      w.skey = (unsigned long long*)(slab + o_skey);
      w.w = (double*)(slab + o_w);
      w.res = (double*)(slab + o_res);
      w.hval = (double*)(slab + o_hval);
      w.hidx = (int*)(slab + o_hidx);
      m.big = (BigSolveWs*)(slab + o_big);
      big_host.push_back(w);
      CU(cudaMemcpyAsync(m.big, &big_host.back(), sizeof(BigSolveWs), cudaMemcpyHostToDevice, s));
    }
    max_ni = std::max(max_ni, (int)ni);
    max_nj = std::max(max_nj, (int)nj);
  }
  MatchDev* d_pairs = nullptr;
  CU(scratch.alloc((void**)&d_pairs, sizeof(MatchDev) * count));
  CU(cudaMemcpyAsync(d_pairs, pairs.data(), sizeof(MatchDev) * count, cudaMemcpyHostToDevice, s));
  QuatroParamsDev q;
  q.normal_r2 = (float)(prm->fpfh_normal_radius * prm->fpfh_normal_radius);
  q.fpfh_r2 = (float)(prm->fpfh_radius * prm->fpfh_radius);
  // advancedMatching searches without a distance gate: FLT_MAX makes every finite distance qualify
  q.thr2 = advanced ? 3.402823466e38f : (float)prm->distance_threshold * (float)prm->distance_threshold;
  q.advanced = advanced ? 1 : 0;
  q.tuple_scale = (float)prm->tuple_scale;
  q.max_corres = prm->max_corres;
  q.noise_bound = prm->noise_bound;
  q.gnc_factor = prm->rot_gnc_factor;
  q.cost_thr = prm->rot_cost_thr;
  q.max_iter = prm->rot_max_iter;
  q.seed = prm->seed;
  {
    ProfScope ps(c, CLS_MATCH);
    c->launches += launch_quatro_match_solve(d_pairs, count, max_ni, max_nj, q, s);
    for (int i = 0; i < count; i++) c->prof_bytes[CLS_MATCH] += 132.0 * (pairs[i].fi.n + pairs[i].fj.n) + 8.0 * pairs[i].fj.n;  // SURVEY §8(d) Q4
  }
  CU(cudaGetLastError());
  std::vector<int> counters(8 * (size_t)count);
  for (int i = 0; i < count; i++) {
    CU(cudaMemcpyAsync(&counters[8 * i], pairs[i].counters, 32, cudaMemcpyDeviceToHost, s));
    CU(cudaMemcpyAsync(out[i].T, pairs[i].T, 128, cudaMemcpyDeviceToHost, s));
    if (corr_out) {
      const size_t have = advanced ? (size_t)big_host[i].cap : (size_t)MAXC;  // what this pair's buffer holds
      CU(cudaMemcpyAsync(&corr_out[2 * (size_t)corr_stride * i], pairs[i].out_corr, 2 * have * 4, cudaMemcpyDeviceToHost, s));
    }
  }
  CU(cudaStreamSynchronize(s));
  for (int i = 0; i < count; i++)
    if (counters[8 * i + 6] > 0) {
      char msg[160];
      snprintf(msg, sizeof msg, "advancedMatching kept %d correspondences for pair %d; the solver workspace holds %d", counters[8 * i + 6], i,
               big_host[i].cap);
      return fail(B200REG_ESTATE, msg);
    }
  for (int i = 0; i < count; i++) {
    out[i].valid = counters[8 * i + 3];
    out[i].n_mutual = counters[8 * i + 1];
    out[i].n_corr = counters[8 * i + 2];
    out[i].clique_size = counters[8 * i + 4];
    out[i].gnc_iterations = counters[8 * i + 5];
    out[i].reserved = 0;
  }
  return B200REG_OK;
}

// LoopClosure::coarseToFineAlignment on cloud handles (loop_closure.cpp:138-159)
static int coarse_to_fine_on_clouds(b200reg_ctx* c, int count, b200reg_cloud* const* src, b200reg_cloud* const* dst,
                                    const b200reg_quatro_params* qp, const b200reg_gicp_params* gp, b200reg_result* out,
                                    b200reg_quatro_info* quatro_out) {
  cudaStream_t s = c->stream;
  Scratch scratch(c);
  std::vector<b200reg_quatro_info> qi(count);
  CloudBag coarse_bag(c);  // the transformed source clouds are released on every exit path
  std::vector<b200reg_cloud*>& coarse = coarse_bag.cl;
  int rc = b200reg_quatro_align(c, count, src, dst, qp, qi.data(), nullptr);
  if (rc) return rc;
  if (quatro_out) memcpy(quatro_out, qi.data(), sizeof(b200reg_quatro_info) * count);
  // pairs whose coarse stage is valid go on to icpAlignment(coarse_aligned_, dst) (loop_closure.cpp:145-156)
  std::vector<int> vidx;
  for (int i = 0; i < count; i++) {
    memset(&out[i], 0, sizeof(b200reg_result));
    for (int k = 0; k < 16; k++) {
      out[i].T[k] = qi[i].T[k];
      out[i].Tf[k] = (float)qi[i].T[k];
      out[i].pose_between[k] = qi[i].T[k];  // an invalid coarse stage returns what quatro::align returned (loop_closure.cpp:144-148)
    }
    out[i].fitness = 1.7976931348623157e308;  // RegistrationOutput::score_ default (loop_closure.h:68)
    if (qi[i].valid) vidx.push_back(i);
  }
  if (!vidx.empty()) {
    const int nv = (int)vidx.size();
    std::vector<CloudDev> sdesc(nv);
    std::vector<double> Ts(16 * (size_t)nv);
    std::vector<float4*> outs(nv);
    std::vector<const float*> cptr(nv);
    std::vector<size_t> cn(nv);
    int max_n = 0;
    for (int k = 0; k < nv; k++) {
      const int i = vidx[k];
      sdesc[k] = src[i]->dev;
      memcpy(&Ts[16 * (size_t)k], qi[i].T, 128);
      float4* raw = nullptr;
      CU(scratch.alloc((void**)&raw, (size_t)sdesc[k].n * 16));
      outs[k] = raw;
      cptr[k] = (const float*)raw;
      cn[k] = sdesc[k].n;
      max_n = std::max(max_n, sdesc[k].n);
    }
    CloudDev* d_desc = nullptr;
    double* d_T = nullptr;
    float4** d_outs = nullptr;
    CU(scratch.alloc((void**)&d_desc, sizeof(CloudDev) * nv));
    CU(scratch.alloc((void**)&d_T, 128 * (size_t)nv));
    CU(scratch.alloc((void**)&d_outs, sizeof(float4*) * nv));
    CU(cudaMemcpyAsync(d_desc, sdesc.data(), sizeof(CloudDev) * nv, cudaMemcpyHostToDevice, s));
    CU(cudaMemcpyAsync(d_T, Ts.data(), 128 * (size_t)nv, cudaMemcpyHostToDevice, s));
    CU(cudaMemcpyAsync(d_outs, outs.data(), sizeof(float4*) * nv, cudaMemcpyHostToDevice, s));
    launch_transform_raw(d_desc, d_T, nv, max_n, d_outs, s);
    c->launches++;
    coarse.assign(nv, nullptr);
    rc = b200reg_clouds_create(c, nv, cptr.data(), cn.data(), 16, 1, coarse.data());
    std::vector<b200reg_cloud*> tg(nv);
    for (int k = 0; k < nv; k++) tg[k] = dst[vidx[k]];
    std::vector<b200reg_result> gres(nv);
    if (!rc) rc = b200reg_gicp_align(c, nv, coarse.data(), tg.data(), nullptr, gp, gres.data());
    if (rc) return rc;
    for (int k = 0; k < nv; k++) {
      const int i = vidx[k];
      b200reg_result r = gres[k];
      // reg_output.pose_between_eig_ = fine (float -> double) * quatro_tf_  (loop_closure.cpp:156)
      double F[16], Q[16];
      for (int a = 0; a < 16; a++) {
        F[a] = (double)gres[k].Tf[a];
        Q[a] = qi[i].T[a];
      }
      for (int a = 0; a < 4; a++)
        for (int b = 0; b < 4; b++) {
          double v = 0, pb = 0;
          for (int m = 0; m < 4; m++) {
            v += F[4 * a + m] * Q[4 * m + b];
            pb += gres[k].pose_between[4 * a + m] * Q[4 * m + b];  // fine_output.pose_between_eig_ is Identity when the fine
          }                                                        // stage is not valid: the reference then keeps I * Q
          r.T[4 * a + b] = v;           // telemetry: the solver's own final transform composed with the coarse stage
          r.Tf[4 * a + b] = (float)v;
          r.pose_between[4 * a + b] = pb;
        }
      out[i] = r;
    }
  }
  return B200REG_OK;
}

int b200reg_loop_closure(b200reg_ctx* c, int count, const float* const* src_xyz, const size_t* src_n, const float* const* tgt_xyz,
                         const size_t* tgt_n, size_t stride_bytes, int on_device, const b200reg_quatro_params* qp,
                         const b200reg_gicp_params* gp, b200reg_result* out, b200reg_quatro_info* quatro_out) {
  if (!c || count <= 0 || !src_xyz || !src_n || !tgt_xyz || !tgt_n || !qp || !gp || !out) return fail(B200REG_EINVAL, "bad argument");
  CU(cudaSetDevice(c->device));
  std::vector<const float*> ptrs(2 * count);
  std::vector<size_t> ns(2 * count);
  for (int i = 0; i < count; i++) {
    ptrs[i] = src_xyz[i];
    ns[i] = src_n[i];
    ptrs[count + i] = tgt_xyz[i];
    ns[count + i] = tgt_n[i];
  }
  std::vector<b200reg_cloud*> clouds(2 * count, nullptr);
  int rc = b200reg_clouds_create(c, 2 * count, ptrs.data(), ns.data(), stride_bytes, on_device, clouds.data());
  if (!rc) rc = coarse_to_fine_on_clouds(c, count, clouds.data(), clouds.data() + count, qp, gp, out, quatro_out);
  for (b200reg_cloud* cl : clouds) b200reg_cloud_destroy(c, cl);
  return rc;
}

// ---- the one collective: all-gather of the result records over NCCL (SURVEY §8(e)) ------------------------
namespace {
struct NcclApi {
  void* h = nullptr;
  decltype(&ncclGetUniqueId) GetUniqueId = nullptr;
  decltype(&ncclCommInitRank) CommInitRank = nullptr;
  decltype(&ncclCommDestroy) CommDestroy = nullptr;
  decltype(&ncclAllGather) AllGather = nullptr;
  decltype(&ncclGetErrorString) GetErrorString = nullptr;
  std::string err;
};
NcclApi* nccl_api() {  // loaded once per process; a process that already holds libnccl.so.2 (torch) shares that copy
  static NcclApi api;
  static bool tried = false;
  static std::mutex mu;
  std::lock_guard<std::mutex> lk(mu);
  if (tried) return &api;
  tried = true;
  // 1. a copy this process already holds (e.g. the one a framework bundles and linked first): two NCCL builds under one
  //    soname would starve whichever library loads second of its symbols;  2. $B200REG_NCCL_LIB (the Python binding points
  //    it at the pip-bundled libnccl so that a LATER `import torch` finds the version it was built against);  3. the system's.
  api.h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD);
  const char* names[] = {getenv("B200REG_NCCL_LIB"), "libnccl.so.2", "libnccl.so"};
  for (const char* n : names) {
    if (api.h) break;
    if (!n || !*n) continue;
    api.h = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
  }
  if (!api.h) {
    api.err = std::string("cannot load libnccl.so.2: ") + dlerror();
    return &api;
  }
  api.GetUniqueId = (decltype(api.GetUniqueId))dlsym(api.h, "ncclGetUniqueId");
  api.CommInitRank = (decltype(api.CommInitRank))dlsym(api.h, "ncclCommInitRank");
  api.CommDestroy = (decltype(api.CommDestroy))dlsym(api.h, "ncclCommDestroy");
  api.AllGather = (decltype(api.AllGather))dlsym(api.h, "ncclAllGather");
  api.GetErrorString = (decltype(api.GetErrorString))dlsym(api.h, "ncclGetErrorString");
  if (!api.GetUniqueId || !api.CommInitRank || !api.CommDestroy || !api.AllGather || !api.GetErrorString) {
    api.err = "libnccl.so.2 lacks a required symbol";
    dlclose(api.h);
    api.h = nullptr;
  }
  return &api;
}
}  // namespace
#define NC(call)                                                                                               \
  do {                                                                                                         \
    ncclResult_t _r = (call);                                                                                  \
    if (_r != ncclSuccess) return fail(B200REG_ENCCL, std::string(#call) + ": " + api->GetErrorString(_r)); \
  } while (0)

static_assert(sizeof(ncclUniqueId) == B200REG_UNIQUE_ID_BYTES, "ncclUniqueId is 128 bytes");

int b200reg_comm_unique_id(void* id_out) {
  if (!id_out) return fail(B200REG_EINVAL, "id_out is NULL");
  NcclApi* api = nccl_api();
  if (!api->h) return fail(B200REG_ENCCL, api->err);
  ncclUniqueId id;
  NC(api->GetUniqueId(&id));
  memcpy(id_out, &id, sizeof(id));
  return B200REG_OK;
}

int b200reg_comm_init(b200reg_ctx* c, const void* id128, int rank, int world) {
  if (!c || !id128 || world < 1 || rank < 0 || rank >= world) return fail(B200REG_EINVAL, "bad argument");
  if (c->comm) return fail(B200REG_ESTATE, "the context already has a communicator");
  NcclApi* api = nccl_api();
  if (!api->h) return fail(B200REG_ENCCL, api->err);
  CU(cudaSetDevice(c->device));
  ncclUniqueId id;
  memcpy(&id, id128, sizeof(id));
  NC(api->CommInitRank(&c->comm, world, id, rank));
  c->rank = rank;
  c->world = world;
  return B200REG_OK;
}

int b200reg_comm_destroy(b200reg_ctx* c) {
  if (!c) return fail(B200REG_EINVAL, "ctx is NULL");
  if (!c->comm) return B200REG_OK;
  NcclApi* api = nccl_api();
  cudaSetDevice(c->device);
  cudaStreamSynchronize(c->stream);
  ncclComm_t comm = c->comm;
  c->comm = nullptr;
  c->rank = -1;
  c->world = 1;
  NC(api->CommDestroy(comm));
  return B200REG_OK;
}

int b200reg_comm_rank(const b200reg_ctx* c) { return c ? c->rank : -1; }
int b200reg_comm_world(const b200reg_ctx* c) { return c ? c->world : 1; }

int b200reg_allgather_results(b200reg_ctx* c, const b200reg_result* local, int n_local, b200reg_result* all_out) {
  if (!c || !local || n_local <= 0 || !all_out) return fail(B200REG_EINVAL, "bad argument");
  const size_t bytes = sizeof(b200reg_result) * (size_t)n_local;
  if (!c->comm || c->world == 1) {
    if (all_out != local) memcpy(all_out, local, bytes);
    return B200REG_OK;
  }
  NcclApi* api = nccl_api();
  CU(cudaSetDevice(c->device));
  cudaStream_t s = c->stream;
  Scratch scratch(c);
  char *d_local = nullptr, *d_all = nullptr;
  CU(scratch.alloc((void**)&d_local, bytes));
  CU(scratch.alloc((void**)&d_all, bytes * c->world));
  CU(cudaMemcpyAsync(d_local, local, bytes, cudaMemcpyHostToDevice, s));
  NC(api->AllGather(d_local, d_all, bytes, ncclChar, c->comm, s));
  CU(cudaMemcpyAsync(all_out, d_all, bytes * c->world, cudaMemcpyDeviceToHost, s));
  CU(cudaStreamSynchronize(s));
  return B200REG_OK;
}

// ---- "next" rows: keyframe store, candidate search, cloud assembly ----------------------------
// Keyframe clouds live in SLABS of their own (plain cudaMalloc, never the context's stream-ordered pool): a store only
// grows, while every registration call takes and returns hundreds of MB of scratch from the pool; 480 KB keyframes carved
// out of the pool's free scratch blocks between two calls fragmented it, and the pool then grew by a fresh block in almost
// every call (tens of ms each: profiles/diag_sequence_e2e.py measured 5.4 -> 11 ... 37 ms per 16-attempt step).
struct KfSlab {
  float4* base = nullptr;
  size_t cap = 0, used = 0;  // points
};
struct b200reg_keyframes {
  std::vector<float4*> pts;
  std::vector<int> n;
  std::vector<double> poses;   // 16 per keyframe, row-major
  std::vector<double> stamps;
  std::vector<KfSlab> slabs;
};
constexpr size_t KF_SLAB_POINTS = (size_t)8 << 20;  // 8 Mi points = 128 MB per slab unless reserved otherwise

// room for n more points: the tail of the last slab, else a new slab (cudaMalloc: a rare, synchronous event)
static int kf_alloc(b200reg_keyframes* kf, size_t n, size_t min_slab, float4** out) {
  if (kf->slabs.empty() || kf->slabs.back().cap - kf->slabs.back().used < n) {
    KfSlab sl;
    sl.cap = std::max(n, min_slab);
    CU(cudaMalloc((void**)&sl.base, sl.cap * sizeof(float4)));
    kf->slabs.push_back(sl);
  }
  KfSlab& sl = kf->slabs.back();
  *out = sl.base + sl.used;
  sl.used += n;
  return B200REG_OK;
}

void b200reg_default_loop_config(b200reg_loop_config* cfg) {
  if (!cfg) return;
  cfg->enable_quatro = 1;
  cfg->enable_submap_matching = 0;
  cfg->num_submap_keyframes = 5;
  cfg->reserved = 0;
  cfg->voxel_res = 0.3;
  cfg->loop_detection_radius = 35.0;
  cfg->loop_detection_timediff_threshold = 30.0;
  b200reg_default_gicp_params(&cfg->gicp);
  b200reg_default_quatro_params(&cfg->quatro);
}

int b200reg_keyframes_create(b200reg_ctx* c, b200reg_keyframes** out) {
  if (!c || !out) return fail(B200REG_EINVAL, "bad argument");
  *out = new b200reg_keyframes;
  return B200REG_OK;
}

int b200reg_keyframes_destroy(b200reg_ctx* c, b200reg_keyframes* kf) {
  if (!kf) return B200REG_OK;
  if (!c) return fail(B200REG_EINVAL, "ctx is NULL");
  CU(cudaSetDevice(c->device));
  CU(cudaStreamSynchronize(c->stream));  // nothing in flight may still read a keyframe
  for (KfSlab& sl : kf->slabs) CU(cudaFree(sl.base));
  delete kf;
  return B200REG_OK;
}

int b200reg_keyframes_reserve(b200reg_ctx* c, b200reg_keyframes* kf, size_t n_points) {
  if (!c || !kf) return fail(B200REG_EINVAL, "bad argument");
  CU(cudaSetDevice(c->device));
  if (!kf->slabs.empty() && kf->slabs.back().cap - kf->slabs.back().used >= n_points) return B200REG_OK;
  if (n_points == 0) return B200REG_OK;
  KfSlab sl;
  sl.cap = n_points;
  CU(cudaMalloc((void**)&sl.base, sl.cap * sizeof(float4)));
  kf->slabs.push_back(sl);
  return B200REG_OK;
}

int b200reg_keyframes_size(const b200reg_keyframes* kf) { return kf ? (int)kf->pts.size() : 0; }

int b200reg_keyframes_add(b200reg_ctx* c, b200reg_keyframes* kf, const float* xyzi, size_t n, size_t stride_bytes, const double* pose16,
                          double timestamp) {
  if (!c || !kf || !xyzi || n == 0 || !pose16 || stride_bytes < 16 || stride_bytes % 4) return fail(B200REG_EINVAL, "bad argument");
  CU(cudaSetDevice(c->device));
  float4* d = nullptr;
  {
    const int rc = kf_alloc(kf, n, KF_SLAB_POINTS, &d);
    if (rc) return rc;
  }
  if (stride_bytes == 16) {  // already packed (x, y, z, intensity): one linear copy (a 2-D copy of n 16-byte rows crawls)
    CU(cudaMemcpyAsync(d, xyzi, n * 16, cudaMemcpyHostToDevice, c->stream));
  } else {  // pcl::PointXYZI (32 B) and friends: upload the records as they are, repack on the device
    Scratch scratch(c);
    float* d_raw = nullptr;
    CU(scratch.alloc((void**)&d_raw, n * stride_bytes));
    CU(cudaMemcpyAsync(d_raw, xyzi, n * stride_bytes, cudaMemcpyHostToDevice, c->stream));
    launch_pack_xyzi(d_raw, (int)(stride_bytes / 4), (int)n, d, c->stream);
    c->launches++;
    CU(cudaGetLastError());
  }
  kf->pts.push_back(d);
  kf->n.push_back((int)n);
  kf->poses.insert(kf->poses.end(), pose16, pose16 + 16);
  kf->stamps.push_back(timestamp);
  return (int)kf->pts.size() - 1;
}

namespace {
// inverse of a 4x4 by cofactors (what pose_eig_.inverse() computes for a fixed-size 4x4; row-major in, row-major out)
bool inverse4(const double* m, double* inv) {
  double a[16];
  a[0] = m[5] * m[10] * m[15] - m[5] * m[11] * m[14] - m[9] * m[6] * m[15] + m[9] * m[7] * m[14] + m[13] * m[6] * m[11] - m[13] * m[7] * m[10];
  a[4] = -m[4] * m[10] * m[15] + m[4] * m[11] * m[14] + m[8] * m[6] * m[15] - m[8] * m[7] * m[14] - m[12] * m[6] * m[11] + m[12] * m[7] * m[10];
  a[8] = m[4] * m[9] * m[15] - m[4] * m[11] * m[13] - m[8] * m[5] * m[15] + m[8] * m[7] * m[13] + m[12] * m[5] * m[11] - m[12] * m[7] * m[9];
  a[12] = -m[4] * m[9] * m[14] + m[4] * m[10] * m[13] + m[8] * m[5] * m[14] - m[8] * m[6] * m[13] - m[12] * m[5] * m[10] + m[12] * m[6] * m[9];
  a[1] = -m[1] * m[10] * m[15] + m[1] * m[11] * m[14] + m[9] * m[2] * m[15] - m[9] * m[3] * m[14] - m[13] * m[2] * m[11] + m[13] * m[3] * m[10];
  a[5] = m[0] * m[10] * m[15] - m[0] * m[11] * m[14] - m[8] * m[2] * m[15] + m[8] * m[3] * m[14] + m[12] * m[2] * m[11] - m[12] * m[3] * m[10];
  a[9] = -m[0] * m[9] * m[15] + m[0] * m[11] * m[13] + m[8] * m[1] * m[15] - m[8] * m[3] * m[13] - m[12] * m[1] * m[11] + m[12] * m[3] * m[9];
  a[13] = m[0] * m[9] * m[14] - m[0] * m[10] * m[13] - m[8] * m[1] * m[14] + m[8] * m[2] * m[13] + m[12] * m[1] * m[10] - m[12] * m[2] * m[9];
  a[2] = m[1] * m[6] * m[15] - m[1] * m[7] * m[14] - m[5] * m[2] * m[15] + m[5] * m[3] * m[14] + m[13] * m[2] * m[7] - m[13] * m[3] * m[6];
  a[6] = -m[0] * m[6] * m[15] + m[0] * m[7] * m[14] + m[4] * m[2] * m[15] - m[4] * m[3] * m[14] - m[12] * m[2] * m[7] + m[12] * m[3] * m[6];
  a[10] = m[0] * m[5] * m[15] - m[0] * m[7] * m[13] - m[4] * m[1] * m[15] + m[4] * m[3] * m[13] + m[12] * m[1] * m[7] - m[12] * m[3] * m[5];
  a[14] = -m[0] * m[5] * m[14] + m[0] * m[6] * m[13] + m[4] * m[1] * m[14] - m[4] * m[2] * m[13] - m[12] * m[1] * m[6] + m[12] * m[2] * m[5];
  a[3] = -m[1] * m[6] * m[11] + m[1] * m[7] * m[10] + m[5] * m[2] * m[11] - m[5] * m[3] * m[10] - m[9] * m[2] * m[7] + m[9] * m[3] * m[6];
  a[7] = m[0] * m[6] * m[11] - m[0] * m[7] * m[10] - m[4] * m[2] * m[11] + m[4] * m[3] * m[10] + m[8] * m[2] * m[7] - m[8] * m[3] * m[6];
  a[11] = -m[0] * m[5] * m[11] + m[0] * m[7] * m[9] + m[4] * m[1] * m[11] - m[4] * m[3] * m[9] - m[8] * m[1] * m[7] + m[8] * m[3] * m[5];
  a[15] = m[0] * m[5] * m[10] - m[0] * m[6] * m[9] - m[4] * m[1] * m[10] + m[4] * m[2] * m[9] + m[8] * m[1] * m[6] - m[8] * m[2] * m[5];
  const double det = m[0] * a[0] + m[1] * a[4] + m[2] * a[8] + m[3] * a[12];
  if (det == 0.0) return false;
  for (int i = 0; i < 16; i++) inv[i] = a[i] / det;
  return true;
}
}  // namespace

int b200reg_keyframes_add_world(b200reg_ctx* c, b200reg_keyframes* kf, const float* xyzi_world, size_t n, size_t stride_bytes,
                                const double* pos, const double* q, double timestamp) {
  if (!c || !kf || !xyzi_world || n == 0 || !pos || !q || stride_bytes < 16 || stride_bytes % 4) return fail(B200REG_EINVAL, "bad argument");
  // tf::Matrix3x3(q) = setRotation(q) (tf/LinearMath/Matrix3x3.h; tf itself is not vendored): s = 2 / |q|^2
  const double x = q[0], y = q[1], z = q[2], w = q[3];
  const double d = x * x + y * y + z * z + w * w;
  if (!(d > 0.0)) return fail(B200REG_EINVAL, "zero quaternion");
  const double sc = 2.0 / d;
  const double xs = x * sc, ys = y * sc, zs = z * sc;
  const double wx = w * xs, wy = w * ys, wz = w * zs, xx = x * xs, xy = x * ys, xz = x * zs, yy = y * ys, yz = y * zs, zz = z * zs;
  const double P[16] = {1.0 - (yy + zz), xy - wz, xz + wy, pos[0], xy + wz, 1.0 - (xx + zz), yz - wx, pos[1],
                        xz - wy, yz + wx, 1.0 - (xx + yy), pos[2], 0.0, 0.0, 0.0, 1.0};
  double Tinv[16];
  if (!inverse4(P, Tinv)) return fail(B200REG_EINVAL, "singular pose");
  CU(cudaSetDevice(c->device));
  cudaStream_t s = c->stream;
  Scratch scratch(c);
  float* d_raw = nullptr;
  double* d_T = nullptr;
  float4* d_out = nullptr;
  CU(scratch.alloc((void**)&d_raw, n * stride_bytes));
  CU(scratch.alloc((void**)&d_T, 128));
  {
    const int rc = kf_alloc(kf, n, KF_SLAB_POINTS, &d_out);
    if (rc) return rc;
  }
  CU(cudaMemcpyAsync(d_raw, xyzi_world, n * stride_bytes, cudaMemcpyHostToDevice, s));
  CU(cudaMemcpyAsync(d_T, Tinv, 128, cudaMemcpyHostToDevice, s));
  launch_ingest_world(d_raw, (int)(stride_bytes / 4), (int)n, d_T, d_out, s);
  c->launches++;
  CU(cudaGetLastError());
  CU(cudaStreamSynchronize(s));  // Tinv lives on this stack frame; the caller's message buffer may go away
  kf->pts.push_back(d_out);
  kf->n.push_back((int)n);
  kf->poses.insert(kf->poses.end(), P, P + 16);
  kf->stamps.push_back(timestamp);
  return (int)kf->pts.size() - 1;
}

int b200reg_keyframes_get(b200reg_ctx* c, const b200reg_keyframes* kf, int idx, float* xyzi_out, double* pose16_out, double* ts_out) {
  if (!c || !kf || idx < 0 || idx >= (int)kf->pts.size()) return fail(B200REG_EINVAL, "bad argument");
  if (pose16_out) memcpy(pose16_out, &kf->poses[16 * (size_t)idx], 128);
  if (ts_out) *ts_out = kf->stamps[idx];
  if (xyzi_out) {
    CU(cudaSetDevice(c->device));
    CU(cudaMemcpyAsync(xyzi_out, kf->pts[idx], (size_t)kf->n[idx] * 16, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
  }
  return B200REG_OK;
}

size_t b200reg_keyframes_cloud_size(const b200reg_keyframes* kf, int idx) {
  return (kf && idx >= 0 && idx < (int)kf->n.size()) ? (size_t)kf->n[idx] : 0;
}

int b200reg_keyframes_set_pose(b200reg_ctx* c, b200reg_keyframes* kf, int idx, const double* pose16) {
  if (!c || !kf || !pose16 || idx < 0 || idx >= (int)kf->pts.size()) return fail(B200REG_EINVAL, "bad argument");
  memcpy(&kf->poses[16 * (size_t)idx], pose16, 128);
  return B200REG_OK;
}

// ---- result consumption (host arithmetic only) -------------------------------------------------------
namespace {
// poseEigToGtsamPose (utilities.hpp:67-75): tf::Matrix3x3::getRPY (getEulerYPR, solution 1), then gtsam::Rot3::RzRyRx
void pose_rpy_roundtrip(const double* P, double R[9], double t[3]) {
  const double m00 = P[0], m10 = P[4], m20 = P[8], m21 = P[9], m22 = P[10];
  double roll, pitch, yaw;
  if (fabs(m20) >= 1.0) {  // gimbal-lock branch of tf's getEulerYPR (tf is not vendored; restated from
                           // tf/LinearMath/Matrix3x3.h: yaw = 0, roll = atan2(m21, m22) in both sub-cases)
    yaw = 0.0;
    roll = atan2(m21, m22);
    pitch = m20 < 0 ? M_PI / 2.0 : -M_PI / 2.0;
  } else {
    pitch = -asin(m20);
    const double cp = cos(pitch);
    roll = atan2(m21 / cp, m22 / cp);
    yaw = atan2(m10 / cp, m00 / cp);
  }
  const double cx = cos(roll), sx = sin(roll), cy = cos(pitch), sy = sin(pitch), cz = cos(yaw), sz = sin(yaw);
  // Rz(yaw) * Ry(pitch) * Rx(roll)
  R[0] = cz * cy; R[1] = cz * sy * sx - sz * cx; R[2] = cz * sy * cx + sz * sx;
  R[3] = sz * cy; R[4] = sz * sy * sx + cz * cx; R[5] = sz * sy * cx - cz * sx;
  R[6] = -sy;     R[7] = cy * sx;                R[8] = cy * cx;
  t[0] = P[3]; t[1] = P[7]; t[2] = P[11];
}
}  // namespace

int b200reg_loop_factor_from_poses(const double* Tb, const double* Pl, const double* Pc, double score, int valid, int from_idx,
                                   int to_idx, b200reg_loop_factor* out) {
  if (!Tb || !Pl || !Pc || !out) return fail(B200REG_EINVAL, "bad argument");
  double F[16];  // pose_between_eig_ * latest.pose_corrected_eig_ (Matrix4d product)
  for (int r = 0; r < 4; r++)
    for (int cidx = 0; cidx < 4; cidx++) {
      double s = 0;
      for (int k = 0; k < 4; k++) s += Tb[4 * r + k] * Pl[4 * k + cidx];
      F[4 * r + cidx] = s;
    }
  double R1[9], t1[3], R2[9], t2[3];
  pose_rpy_roundtrip(F, R1, t1);
  pose_rpy_roundtrip(Pc, R2, t2);
  // Pose3::between: inverse(from) * to = (R1^T R2, R1^T (t2 - t1))
  double* M = out->measurement;
  for (int r = 0; r < 3; r++) {
    for (int cidx = 0; cidx < 3; cidx++) {
      double s = 0;
      for (int k = 0; k < 3; k++) s += R1[3 * k + r] * R2[3 * k + cidx];
      M[4 * r + cidx] = s;
    }
    double s = 0;
    for (int k = 0; k < 3; k++) s += R1[3 * k + r] * (t2[k] - t1[k]);
    M[4 * r + 3] = s;
  }
  M[12] = M[13] = M[14] = 0.0;
  M[15] = 1.0;
  for (int k = 0; k < 6; k++) out->variances[k] = score;
  out->from_idx = from_idx;
  out->to_idx = to_idx;
  out->valid = valid ? 1 : 0;
  out->reserved = 0;
  return B200REG_OK;
}

int b200reg_loop_factors(b200reg_ctx* c, const b200reg_keyframes* kf, int count, const int32_t* query_idx, const int32_t* closest_idx,
                         const b200reg_result* results, b200reg_loop_factor* out) {
  if (!c || !kf || count <= 0 || !query_idx || !closest_idx || !results || !out) return fail(B200REG_EINVAL, "bad argument");
  const int nk = (int)kf->pts.size();
  for (int i = 0; i < count; i++) {
    if (query_idx[i] < 0 || query_idx[i] >= nk || closest_idx[i] >= nk) return fail(B200REG_EINVAL, "keyframe index out of range");
    if (closest_idx[i] < 0) {  // no candidate: the reference returns before any registration (fast_lio_sam_qn.cpp:213-216)
      memset(&out[i], 0, sizeof(b200reg_loop_factor));
      out[i].from_idx = query_idx[i];
      out[i].to_idx = -1;
      continue;
    }
    const int rc = b200reg_loop_factor_from_poses(results[i].pose_between, &kf->poses[16 * (size_t)query_idx[i]], &kf->poses[16 * (size_t)closest_idx[i]],
                                                  results[i].fitness, results[i].valid, query_idx[i], closest_idx[i], &out[i]);
    if (rc) return rc;
  }
  return B200REG_OK;
}

int b200reg_fetch_closest_keyframes(b200reg_ctx* c, b200reg_keyframes* kf, int count, const int32_t* query_idx, double radius,
                                    double tdiff, int32_t* closest_out) {
  if (!c || !kf || count <= 0 || !query_idx || !closest_out) return fail(B200REG_EINVAL, "bad argument");
  const int nk = (int)kf->pts.size();
  for (int i = 0; i < count; i++)
    if (query_idx[i] < 0 || query_idx[i] >= nk) return fail(B200REG_EINVAL, "query index out of range");
  CU(cudaSetDevice(c->device));
  cudaStream_t s = c->stream;
  Scratch scratch(c);
  std::vector<double> pos(3 * (size_t)nk);
  for (int i = 0; i < nk; i++)
    for (int d = 0; d < 3; d++) pos[3 * (size_t)i + d] = kf->poses[16 * (size_t)i + 4 * d + 3];
  double *d_pos = nullptr, *d_st = nullptr;
  int *d_q = nullptr, *d_o = nullptr;
  CU(scratch.alloc((void**)&d_pos, pos.size() * 8));
  CU(scratch.alloc((void**)&d_st, (size_t)nk * 8));
  CU(scratch.alloc((void**)&d_q, (size_t)count * 4));
  CU(scratch.alloc((void**)&d_o, (size_t)count * 4));
  CU(cudaMemcpyAsync(d_pos, pos.data(), pos.size() * 8, cudaMemcpyHostToDevice, s));
  CU(cudaMemcpyAsync(d_st, kf->stamps.data(), (size_t)nk * 8, cudaMemcpyHostToDevice, s));
  CU(cudaMemcpyAsync(d_q, query_idx, (size_t)count * 4, cudaMemcpyHostToDevice, s));
  c->launches += launch_fetch_closest(d_pos, d_st, d_q, count, radius, tdiff, d_o, s);
  CU(cudaMemcpyAsync(closest_out, d_o, (size_t)count * 4, cudaMemcpyDeviceToHost, s));
  CU(cudaStreamSynchronize(s));
  return B200REG_OK;
}

int b200reg_assemble_clouds(b200reg_ctx* c, b200reg_keyframes* kf, int count, const int32_t* src_idx, const int32_t* dst_idx,
                            const b200reg_loop_config* cfg, int n_keyframes, b200reg_cloud** src_out, b200reg_cloud** dst_out) {
  if (!kf || count <= 0) return fail(B200REG_EINVAL, "bad argument");
  std::vector<int32_t> nks(count, n_keyframes > 0 ? n_keyframes : (int)kf->pts.size());
  return b200reg_assemble_clouds_at(c, kf, count, src_idx, dst_idx, cfg, nks.data(), src_out, dst_out);
}

int b200reg_assemble_clouds_at(b200reg_ctx* c, b200reg_keyframes* kf, int count, const int32_t* src_idx, const int32_t* dst_idx,
                               const b200reg_loop_config* cfg, const int32_t* n_keyframes, b200reg_cloud** src_out,
                               b200reg_cloud** dst_out) {
  if (!c || !kf || count <= 0 || !src_idx || !dst_idx || !cfg || !n_keyframes || !src_out || !dst_out)
    return fail(B200REG_EINVAL, "bad argument");
  for (int i = 0; i < count; i++)
    if (n_keyframes[i] <= 0 || n_keyframes[i] > (int)kf->pts.size()) return fail(B200REG_EINVAL, "n_keyframes out of range");
  const int range = cfg->num_submap_keyframes;
  if (2 * range + 1 > MAXSEG) return fail(B200REG_EINVAL, "num_submap_keyframes too large");
  if (!(cfg->voxel_res > 0)) return fail(B200REG_EINVAL, "voxel_res must be positive");
  CU(cudaSetDevice(c->device));
  cudaStream_t s = c->stream;
  Scratch scratch(c);
  const int njobs = 2 * count;  // jobs [0,count) = src clouds, [count, 2 count) = dst clouds
  std::vector<AssembleJob> jobs(njobs);
  std::vector<CloudDev> sorts(njobs);
  int max_total = 0;
  for (int j = 0; j < njobs; j++) {
    const bool is_src = j < count;
    const int centre = is_src ? src_idx[j] : dst_idx[j - count];
    const int nk = n_keyframes[is_src ? j : j - count];  // keyframes.size() at this pair's tick
    if (centre < 0 || centre >= nk) return fail(B200REG_EINVAL, "keyframe index out of range");
    AssembleJob& J = jobs[j];
    memset(&J, 0, sizeof(J));
    // loop_closure.cpp:68-105: which keyframes are merged
    const bool merged = cfg->enable_submap_matching || (!is_src && !cfg->enable_quatro);
    J.nseg = 0;
    J.seg_off[0] = 0;
    if (merged) {
      for (int i = centre - range; i < centre + range + 1; i++)
        if (i >= 0 && i < nk - 1) {  // the reference excludes the last keyframe (loop_closure.cpp:72,79,100)
          J.seg_kf[J.nseg] = i;
          J.seg_off[J.nseg + 1] = J.seg_off[J.nseg] + kf->n[i];
          J.nseg++;
        }
    } else {
      J.seg_kf[0] = centre;
      J.seg_off[1] = kf->n[centre];
      J.nseg = 1;
    }
    J.total = J.seg_off[J.nseg];
    if (J.total <= 0) return fail(B200REG_EINVAL, "empty merged cloud");
    const size_t n = J.total;
    size_t o = 0;
    auto take = [&](size_t bytes) {
      size_t r = o;
      o = align_up(o + bytes, 256);
      return r;
    };
    const size_t o_m = take(n * 16), o_o = take(n * 16), o_h = take(n * 4), o_b = take(32), o_c = take(16);
    const size_t o_k0 = take(n * 4), o_k1 = take(n * 4), o_v0 = take(n * 4), o_v1 = take(n * 4), o_hist = take(radix_sort_ws_bytes(J.total, 32));
    char* slab = nullptr;
    CU(scratch.alloc((void**)&slab, o));
    J.merged = (float4*)(slab + o_m);
    J.out = (float4*)(slab + o_o);
    J.heads = (int*)(slab + o_h);
    J.bbox = (int*)(slab + o_b);
    J.counters = (int*)(slab + o_c);
    J.sort.keys[0] = (uint32_t*)(slab + o_k0);
    J.sort.keys[1] = (uint32_t*)(slab + o_k1);
    J.sort.vals[0] = (uint32_t*)(slab + o_v0);
    J.sort.vals[1] = (uint32_t*)(slab + o_v1);
    J.sort.hist = (uint32_t*)(slab + o_hist);
    CU(cudaMemsetAsync(J.sort.hist, 0, radix_sort_ws_bytes(J.total, 32), s));
    CloudDev& sd = sorts[j];
    memset(&sd, 0, sizeof(sd));
    sd.n = J.total;
    sd.keys[0] = J.sort.keys[0];
    sd.keys[1] = J.sort.keys[1];
    sd.vals[0] = J.sort.vals[0];
    sd.vals[1] = J.sort.vals[1];
    sd.hist = J.sort.hist;
    max_total = std::max(max_total, J.total);
  }
  const int nkall = (int)kf->pts.size();
  std::vector<KeyframeDev> kd(nkall);
  for (int i = 0; i < nkall; i++) kd[i] = KeyframeDev{kf->pts[i], kf->n[i], 0};
  AssembleJob* d_jobs = nullptr;
  CloudDev* d_sorts = nullptr;
  KeyframeDev* d_kf = nullptr;
  double* d_poses = nullptr;
  CU(scratch.alloc((void**)&d_jobs, sizeof(AssembleJob) * njobs));
  CU(scratch.alloc((void**)&d_sorts, sizeof(CloudDev) * njobs));
  CU(scratch.alloc((void**)&d_kf, sizeof(KeyframeDev) * nkall));
  CU(scratch.alloc((void**)&d_poses, 128 * (size_t)nkall));
  CU(cudaMemcpyAsync(d_jobs, jobs.data(), sizeof(AssembleJob) * njobs, cudaMemcpyHostToDevice, s));
  CU(cudaMemcpyAsync(d_sorts, sorts.data(), sizeof(CloudDev) * njobs, cudaMemcpyHostToDevice, s));
  CU(cudaMemcpyAsync(d_kf, kd.data(), sizeof(KeyframeDev) * nkall, cudaMemcpyHostToDevice, s));
  CU(cudaMemcpyAsync(d_poses, kf->poses.data(), 128 * (size_t)nkall, cudaMemcpyHostToDevice, s));
  {
    ProfScope ps(c, CLS_MISC);
    const float inv_leaf = 1.0f / (float)cfg->voxel_res;
    c->launches += launch_assemble_voxelize(d_jobs, d_sorts, njobs, max_total, d_kf, d_poses, inv_leaf, s);
    for (int j = 0; j < njobs; j++) c->prof_bytes[CLS_MISC] += 68.0 * jobs[j].total;  // 16 in + 16 merged + 36 sort/centroid
  }
  CU(cudaGetLastError());
  std::vector<int> counters(4 * (size_t)njobs);
  for (int j = 0; j < njobs; j++) CU(cudaMemcpyAsync(&counters[4 * j], jobs[j].counters, 8, cudaMemcpyDeviceToHost, s));
  CU(cudaStreamSynchronize(s));
  // index the voxelised clouds (records are (x, y, z, intensity), 16-byte stride, already on the device)
  std::vector<const float*> ptrs(njobs);
  std::vector<size_t> ns(njobs);
  for (int j = 0; j < njobs; j++) {
    const bool overflow = counters[4 * j + 1] != 0;  // PCL returns the input unchanged in that case
    ptrs[j] = (const float*)(overflow ? jobs[j].merged : jobs[j].out);
    ns[j] = overflow ? (size_t)jobs[j].total : (size_t)counters[4 * j];
  }
  std::vector<b200reg_cloud*> clouds(njobs, nullptr);
  int rc = b200reg_clouds_create(c, njobs, ptrs.data(), ns.data(), 16, 1, clouds.data());
  for (int i = 0; i < count && !rc; i++) {
    src_out[i] = clouds[i];
    dst_out[i] = clouds[count + i];
  }
  return rc;
}

int b200reg_cloud_points(b200reg_ctx* c, const b200reg_cloud* cl, float* xyz_out) {
  if (!c || !cl || !xyz_out) return fail(B200REG_EINVAL, "bad argument");
  CU(cudaSetDevice(c->device));
  const int n = cl->dev.n;
  std::vector<float4> pts(n);
  CU(cudaMemcpyAsync(pts.data(), cl->dev.pts, (size_t)n * 16, cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  for (int p = 0; p < n; p++) {
    int o;
    memcpy(&o, &pts[p].w, 4);
    xyz_out[3 * (size_t)o] = pts[p].x;
    xyz_out[3 * (size_t)o + 1] = pts[p].y;
    xyz_out[3 * (size_t)o + 2] = pts[p].z;
  }
  return B200REG_OK;
}

int b200reg_perform_loop_closure(b200reg_ctx* c, b200reg_keyframes* kf, int count, const int32_t* query_idx, const int32_t* closest_idx,
                                 const b200reg_loop_config* cfg, b200reg_result* out, b200reg_quatro_info* quatro_out) {
  if (!c || !kf || count <= 0 || !query_idx || !closest_idx || !cfg || !out) return fail(B200REG_EINVAL, "bad argument");
  std::vector<int32_t> qs, cs;
  std::vector<int> where;
  for (int i = 0; i < count; i++) {
    memset(&out[i], 0, sizeof(b200reg_result));  // dummy output whose is_valid is false (loop_closure.cpp:201-204)
    out[i].T[0] = out[i].T[5] = out[i].T[10] = out[i].T[15] = 1.0;
    out[i].Tf[0] = out[i].Tf[5] = out[i].Tf[10] = out[i].Tf[15] = 1.f;
    out[i].pose_between[0] = out[i].pose_between[5] = out[i].pose_between[10] = out[i].pose_between[15] = 1.0;
    out[i].fitness = 1.7976931348623157e308;
    if (quatro_out) memset(&quatro_out[i], 0, sizeof(b200reg_quatro_info));
    if (closest_idx[i] >= 0) {
      qs.push_back(query_idx[i]);
      cs.push_back(closest_idx[i]);
      where.push_back(i);
    }
  }
  if (qs.empty()) return B200REG_OK;
  const int m = (int)qs.size();
  // at the time query q was the latest keyframe the vector held q + 1 keyframes (fast_lio_sam_qn.cpp:205-219); a batch
  // replays several ticks, so every pair carries the size its own tick saw (the sub-map bounds of loop_closure.cpp:72,79,100)
  std::vector<int32_t> nks(m);
  for (int k = 0; k < m; k++) nks[k] = qs[k] + 1;
  std::vector<b200reg_cloud*> sc(m, nullptr), dc(m, nullptr);
  int rc = b200reg_assemble_clouds_at(c, kf, m, qs.data(), cs.data(), cfg, nks.data(), sc.data(), dc.data());
  std::vector<b200reg_result> res(m);
  std::vector<b200reg_quatro_info> qi(m);
  if (!rc) {
    if (cfg->enable_quatro) rc = coarse_to_fine_on_clouds(c, m, sc.data(), dc.data(), &cfg->quatro, &cfg->gicp, res.data(), qi.data());
    else rc = b200reg_gicp_align(c, m, sc.data(), dc.data(), nullptr, &cfg->gicp, res.data());
  }
  for (int k = 0; k < m && !rc; k++) {
    out[where[k]] = res[k];
    if (quatro_out && cfg->enable_quatro) quatro_out[where[k]] = qi[k];
  }
  for (int k = 0; k < m; k++) {
    b200reg_cloud_destroy(c, sc[k]);
    b200reg_cloud_destroy(c, dc[k]);
  }
  return rc;
}

// ---- the corrected global map (map.cu) ----------------------------------------------------------------
// The records get a cudaMalloc of their own: they outlive the call (the reason keyframe slabs do, §6b); the workspace
// comes from the scratch pool.
struct b200reg_map {
  float4* d = nullptr;
  size_t n = 0;
  int voxelized = 0;
};
// the sort's look-back words carry 30-bit counts (index_build.cu: LB_MASK)
constexpr size_t MAP_MAX_POINTS = ((size_t)1 << 30) - 1;

int b200reg_map_build(b200reg_ctx* c, const b200reg_keyframes* kf, int n_keyframes, double voxel_res, b200reg_map** out) {
  if (!c || !kf || !out) return fail(B200REG_EINVAL, "bad argument");
  *out = nullptr;
  const int nkall = (int)kf->pts.size();
  if (nkall == 0) return fail(B200REG_EINVAL, "empty keyframe store");
  if (n_keyframes < 0 || n_keyframes > nkall) return fail(B200REG_EINVAL, "n_keyframes out of range");
  if (!(voxel_res > 0)) return fail(B200REG_EINVAL, "voxel_res must be positive");
  const int nk = n_keyframes > 0 ? n_keyframes : nkall;
  // block table: (keyframe, tile) -> source, first merged index, points
  std::vector<MapBlock> blocks;
  size_t total = 0;
  for (int i = 0; i < nk; i++) {
    for (int o = 0; o < kf->n[i]; o += MAP_TILE) blocks.push_back(MapBlock{kf->pts[i] + o, i, (int)(total + o), std::min(MAP_TILE, kf->n[i] - o), 0});
    total += kf->n[i];
    if (total > MAP_MAX_POINTS) return fail(B200REG_EINVAL, "more than 2^30 - 1 merged points");
  }
  const int n = (int)total, nb = (int)blocks.size();
  const float inv_leaf = 1.0f / (float)voxel_res;
  CU(cudaSetDevice(c->device));
  cudaStream_t s = c->stream;
  Scratch scratch(c);
  float4* d_merged = nullptr;
  float* d_partials = nullptr;
  MapBlock* d_blocks = nullptr;
  double* d_poses = nullptr;
  MapInfo* d_info = nullptr;
  CU(scratch.alloc((void**)&d_merged, (size_t)n * 16));
  CU(scratch.alloc((void**)&d_partials, (size_t)nb * 24));
  CU(scratch.alloc((void**)&d_blocks, sizeof(MapBlock) * (size_t)nb));
  CU(scratch.alloc((void**)&d_poses, 128 * (size_t)nk));
  CU(scratch.alloc((void**)&d_info, sizeof(MapInfo)));
  CU(cudaMemcpyAsync(d_blocks, blocks.data(), sizeof(MapBlock) * (size_t)nb, cudaMemcpyHostToDevice, s));
  CU(cudaMemcpyAsync(d_poses, kf->poses.data(), 128 * (size_t)nk, cudaMemcpyHostToDevice, s));
  MapInfo info;
  {
    ProfScope ps(c, CLS_MISC);
    c->launches += launch_map_transform(d_blocks, nb, d_poses, inv_leaf, d_merged, d_partials, d_info, s);
  }
  CU(cudaGetLastError());
  CU(cudaMemcpyAsync(&info, d_info, sizeof(MapInfo), cudaMemcpyDeviceToHost, s));
  CU(cudaStreamSynchronize(s));
  float4* rec = nullptr;
  if (info.overflow) {  // PCL returns the merged cloud as it is
    CU(cudaMalloc((void**)&rec, (size_t)n * 16));
    const cudaError_t e = cudaMemcpyAsync(rec, d_merged, (size_t)n * 16, cudaMemcpyDeviceToDevice, s);
    if (e != cudaSuccess) {
      cudaFree(rec);
      return fail(B200REG_ECUDA, std::string("map copy: ") + cudaGetErrorString(e));
    }
    c->prof_bytes[CLS_MISC] += 48.0 * n;  // 16 in + 16 merged + 16 copied
    *out = new b200reg_map{rec, (size_t)n, 0};
    return B200REG_OK;
  }
#ifndef B200REG_NO_SORT8
  const int key_bits = info.key_bits <= 24 ? info.key_bits : 32;  // 3 x 8-bit digits, or the 3 x 11 bits of the sub-map grid
#else  // development switch: every map on the 11-bit digits (profiles/map_build.py times the two against each other)
  const int key_bits = 32;
#endif
  const int ntiles = (n + MAP_TILE - 1) / MAP_TILE;
  const size_t ws = radix_sort_ws_bytes(n, key_bits);
  CloudDev sd;
  memset(&sd, 0, sizeof(sd));
  sd.n = n;
  int *d_tile_cnt = nullptr, *d_tile_off = nullptr, *d_heads = nullptr;
  float4* d_sorted = nullptr;
  CloudDev* d_sort = nullptr;
  for (int b = 0; b < 2; b++) {
    CU(scratch.alloc((void**)&sd.keys[b], (size_t)n * 4));
    CU(scratch.alloc((void**)&sd.vals[b], (size_t)n * 4));
  }
  CU(scratch.alloc((void**)&sd.hist, ws));
  CU(scratch.alloc((void**)&d_tile_cnt, (size_t)ntiles * 4));
  CU(scratch.alloc((void**)&d_tile_off, (size_t)ntiles * 4));
  CU(scratch.alloc((void**)&d_heads, ((size_t)n + 1) * 4));
  CU(scratch.alloc((void**)&d_sorted, (size_t)n * 16));
  CU(scratch.alloc((void**)&d_sort, sizeof(CloudDev)));
  CU(cudaMemsetAsync(sd.hist, 0, ws, s));
  CU(cudaMemcpyAsync(d_sort, &sd, sizeof(CloudDev), cudaMemcpyHostToDevice, s));
  {
    ProfScope ps(c, CLS_MISC);
    c->launches += launch_map_sort_heads(d_merged, n, inv_leaf, d_info, d_sort, sd, key_bits, d_tile_cnt, d_tile_off, d_heads, d_sorted, s);
  }
  CU(cudaGetLastError());
  int nv = 0;
  CU(cudaMemcpyAsync(&nv, &d_info->voxels, 4, cudaMemcpyDeviceToHost, s));
  CU(cudaStreamSynchronize(s));
  CU(cudaMalloc((void**)&rec, (size_t)nv * 16));
  {
    ProfScope ps(c, CLS_MISC);
    c->launches += launch_map_centroids(d_heads, d_sorted, nv, rec, s);
    c->prof_bytes[CLS_MISC] += 128.0 * n;  // 16 + 16 transform, 16 + 8 keys, 3 x 16 sort passes, 4 heads, 20 centroids
  }
  const cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    cudaFree(rec);
    return fail(B200REG_ECUDA, std::string("map centroids: ") + cudaGetErrorString(e));
  }
  *out = new b200reg_map{rec, (size_t)nv, 1};
  return B200REG_OK;
}

size_t b200reg_map_size(const b200reg_map* m) { return m ? m->n : 0; }

int b200reg_map_voxelized(const b200reg_map* m) { return m ? m->voxelized : 0; }

int b200reg_map_get(b200reg_ctx* c, const b200reg_map* m, float* xyzi_out) {
  if (!c || !m || (!xyzi_out && m->n)) return fail(B200REG_EINVAL, "bad argument");
  if (!m->n) return B200REG_OK;
  CU(cudaSetDevice(c->device));
  CU(cudaMemcpyAsync(xyzi_out, m->d, m->n * 16, cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  return B200REG_OK;
}

int b200reg_map_destroy(b200reg_ctx* c, b200reg_map* m) {
  if (!m) return B200REG_OK;
  if (!c) return fail(B200REG_EINVAL, "ctx is NULL");
  CU(cudaSetDevice(c->device));
  CU(cudaStreamSynchronize(c->stream));  // nothing in flight may still write the records
  CU(cudaFree(m->d));
  delete m;
  return B200REG_OK;
}

}  // extern "C"
