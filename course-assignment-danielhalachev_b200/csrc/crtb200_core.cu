// crtb200_core.cu -- C ABI (include/crtb200.h) of the B200-native renderer core: host flattener H1 (reference trees ->
// stack-free visiting-order layout), device memory management, and the per-frame launch sequence of the wavefront
// kernels in crt_kernels.cuh.  No CPU rendering path exists in this library.
#include <cuda_runtime.h>

#include <algorithm>
#include <chrono>
#include <condition_variable>
#include <functional>
#include <memory>
#include <mutex>
#include <thread>
#include <type_traits>
#include <utility>
#include <cstdio>
#include <cstdlib>
#include <cmath>
#include <cstring>
#include <limits>
#include <string>
#include <vector>

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include "../../include/crtb200.h"
#include "crt_build.cuh"
#include "crt_kernels.cuh"

using namespace crtd;

#ifndef CRT_REFILL
#define CRT_REFILL 16  // refill a warp when at least this many lanes are idle (8 until run r2aj: hw14 2.92 -> 2.77 ms)
#endif
#ifndef CRT_REFILL_CLOSEST
#define CRT_REFILL_CLOSEST CRT_REFILL
#endif
#ifndef CRT_REFILL_SHADOW
#define CRT_REFILL_SHADOW CRT_REFILL
#endif
#ifndef CRT_LOOP_MODE
#define CRT_LOOP_MODE 2  // 0 = while-while, 1 = merged loop, 2 = node phase + warp-cooperative triangle phase (crt_kernels.cuh)
#endif

struct crtb200_ctx;
static thread_local std::string g_error;
static thread_local crtb200_ctx *g_error_ctx = nullptr;  // context of the ABI call running on this thread (ErrScope)
static void note_ctx_error(crtb200_ctx *c, const std::string &msg);
static int fail(int code, const std::string &msg) {
  g_error = msg;
  if (g_error_ctx) note_ctx_error(g_error_ctx, msg);
  return code;
}
struct ErrScope {
  crtb200_ctx *prev;
  explicit ErrScope(crtb200_ctx *c) : prev(g_error_ctx) { g_error_ctx = c; }
  ~ErrScope() { g_error_ctx = prev; }
};

// One helper thread per GPU after the first of a multi-GPU context: launches are asynchronous, but issuing a frame's
// ~20 launches takes the host ~0.1 ms per GPU, which eight GPUs cannot afford serially when a shard renders in ~0.5 ms.
struct Worker {
  std::thread th;
  std::mutex m;
  std::condition_variable cv;
  std::function<void()> job;
  bool has = false, quit = false;
  Worker() {
    th = std::thread([this] {
      std::unique_lock<std::mutex> lk(m);
      for (;;) {
        cv.wait(lk, [this] { return has || quit; });
        if (quit) return;
        lk.unlock();
        job();
        lk.lock();
        has = false;
        cv.notify_all();
      }
    });
  }
  void post(std::function<void()> f) {
    std::unique_lock<std::mutex> lk(m);
    job = std::move(f);
    has = true;
    cv.notify_all();
  }
  void wait() {
    std::unique_lock<std::mutex> lk(m);
    cv.wait(lk, [this] { return !has; });
  }
  ~Worker() {
    {
      std::unique_lock<std::mutex> lk(m);
      quit = true;
      cv.notify_all();
    }
    th.join();
  }
};
#define CUDA_TRY(expr)                                                                                       \
  do {                                                                                                       \
    cudaError_t e_ = (expr);                                                                                 \
    if (e_ != cudaSuccess)                                                                                   \
      return fail(CRTB200_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorName(e_) + ": " + cudaGetErrorString(e_)); \
  } while (0)

// One device allocation, freed by its destructor; move-only.  Owners free on their own device: crtb200_destroy selects
// the context's device before deleting it.
template <typename T>
struct DevBuf {
  T *p = nullptr;
  size_t n = 0;
  DevBuf() = default;
  DevBuf(DevBuf &&o) noexcept : p(std::exchange(o.p, nullptr)), n(std::exchange(o.n, 0)) {}
  DevBuf &operator=(DevBuf o) noexcept {  // (o is moved in and frees what this held)
    std::swap(p, o.p);
    std::swap(n, o.n);
    return *this;
  }
  ~DevBuf() { release(); }
  cudaError_t ensure(size_t count) {
    if (count <= n && p) return cudaSuccess;
    release();
    if (count == 0) return cudaSuccess;
    cudaError_t e = cudaMalloc(&p, count * sizeof(T));
    if (e == cudaSuccess) n = count;
    return e;
  }
  cudaError_t upload(const std::vector<T> &v) {
    cudaError_t e = ensure(std::max<size_t>(v.size(), 1));
    if (e != cudaSuccess) return e;
    if (v.empty()) return cudaSuccess;
    return cudaMemcpy(p, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice);
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    n = 0;
  }
};

// One CUDA stream or event, destroyed by its destructor; move-only, null until create() makes it.
template <typename H>
struct CudaHandle {
  H h = nullptr;
  CudaHandle() = default;
  CudaHandle(CudaHandle &&o) noexcept : h(std::exchange(o.h, nullptr)) {}
  CudaHandle &operator=(CudaHandle o) noexcept {
    std::swap(h, o.h);
    return *this;
  }
  ~CudaHandle() {
    if (!h) return;
    if constexpr (std::is_same_v<H, cudaStream_t>) cudaStreamDestroy(h);
    else cudaEventDestroy(h);
  }
  operator H() const { return h; }
  // Creates the handle unless it exists.  Streams: flags cudaStreamNonBlocking and `priority` (0 is the default
  // priority); events: flags cudaEventDefault or cudaEventDisableTiming.
  cudaError_t create(unsigned flags, int priority = 0) {
    if (h) return cudaSuccess;
    H x = nullptr;
    cudaError_t e;
    if constexpr (std::is_same_v<H, cudaStream_t>) e = cudaStreamCreateWithPriority(&x, flags, priority);
    else e = cudaEventCreateWithFlags(&x, flags);
    if (e == cudaSuccess) h = x;
    return e;
  }
};
using Stream = CudaHandle<cudaStream_t>;
using Event = CudaHandle<cudaEvent_t>;

// counters of a render kept beside crtb200_stats: diffuse rays, and an adaptive step's pixel-samples and stopped pixels
struct SideCounts { uint64_t diffuse = 0, px_samples = 0, stopped = 0; };

// What a render or query counted: crtb200_stats and the side counts.  Read from one GPU's CRT_STAT_* slots it holds
// the counters only; totals add launches and times too.
struct Counts {
  crtb200_stats s{};
  SideCounts side;
};

// queues: `concurrency` independent buffer sets, each with its own stream.  Consecutive chunks of a frame go to the
// sets round-robin, so the latency-bound tails of one chunk's persistent kernels (and the small secondary-level
// launches of reflective / refractive scenes) are filled by the other chunks' kernels.
struct QueueSet {
  Levels lv{};
  DevBuf<float4> ray_o, ray_d, color, dq;
  DevBuf<uint32_t> hit_tri, ctl;  // ctl = counts | work cursors | hand-off counters, zeroed by one memset per chunk
  DevBuf<float> hit_t;
  DevBuf<uint4> comb;
  DevBuf<uint8_t> vis;
  DevBuf<uint4> ovf;          // walks handed off to k_coop (3 x uint4 per record)
  DevBuf<float4> acc;         // GI frames: per level-0 item of the chunk, the running sample sum (k_sample_acc)
  DevBuf<uint2> hit0;         //            ... and sample 0's primary hit
  DevBuf<uint32_t> alist, acount;  // adaptive passes: the chunk's active shard items and their count (k_adapt_compact)
  uint32_t *work = nullptr;   // into ctl
  Stream stream;              // (frames only: a query runs on the caller's stream)
  Event done;
  // early k_coop pass: low-priority side stream, forked before and joined behind every traversal launch
  Stream coop_stream;
  Event coop_fork, coop_join;
};

// One GPU of a context: what each GPU of a multi-GPU context holds for itself -- its stream, scene replica, queues,
// query scratch, progressive accumulator shard and tuning.
struct Gpu {
  int device = 0;
  int sm_count = 0;
  Stream stream;
  bool have_scene = false;

  // scene
  DScene sc{};
  // nodes / leaf_refs / tri_geom (everything the traversal kernels chase) live in ONE allocation so that a single L2
  // access-policy window can mark them persisting: the ~1 GB of ray / hit / colour queues a 4K frame streams through
  // the 126 MB L2 then stops evicting the scene between and during the traversal kernels
  DevBuf<uint8_t> arena;
  float4 *nodes_p = nullptr, *tri_geom_p = nullptr;
  uint32_t *leaf_refs_p = nullptr;
  size_t arena_used = 0;
  size_t l2_persist_max = 0, l2_window_max = 0;
  int l2_persist = 0;  // CRT_L2_PERSIST: 0 off (default, measured best), 1 arena persisting / rest of it streaming, 2 arena persisting / normal, 3 nodes only
  size_t nodes_bytes = 0;
  DevBuf<float4> vtx_normal;
  bool nested_ok = false;    // every child box of the uploaded mesh trees lies inside its parent's and no tree is deeper
                             // than the k_coop LIFO allows: the order-free walk of k_coop and the subtree culling are exact
  int tail_iters = 16;       // tail hand-off (crt_kernels.cuh): once a traversal kernel's queue is dry, walks longer than a
                             // falling threshold (512 node-phase iterations, halved every 4 rounds, never below this
                             // floor) go to k_coop.  CRT_TAIL_ITERS overrides (tools / tests): 0 = every walk still
                             // running (the threshold still falls from 512), -1 = off
  int tail_start = 512;      // CRT_TAIL_START (tests): the threshold's starting value, shadow pass
  int tail_start_closest = 256;  // CRT_TAIL_START_CLOSEST: ... closest-hit launches (runs r2aq, r2at: 10M 2.02 -> 1.95 ms against 512, hw07 0.96 -> 1.00; 128: 1.93 / 1.08)
  int tail_small = 32768;    // CRT_TAIL_SMALL: launches of at most this many rays hand off at the floor from the start
  int tail_cap = 8;          // hand-off capacity per launch, in walks per resident k_coop warp (CRT_TAIL_CAP; tests use
                             // a huge value so that every walk goes through k_coop)
  DevBuf<uint32_t> top_refs;
  DevBuf<uint4> tri_shade;
  DevBuf<float2> vtx_uv;
  DevBuf<DMesh> meshes;
  DevBuf<DMaterial> materials;
  DevBuf<DTexture> textures;
  DevBuf<float> texels;
  DevBuf<DLight> lights;
  bool has_reflective = false, has_refractive = false;
  uint32_t n_nodes = 0, n_leaf_refs = 0, n_top_refs = 0;  // of the uploaded scene (crtb200_debug_scene_layout)
  uint32_t n_triangles = 0;   // of the uploaded scene (crtb200_accum_load checks the hit records it is given)

  DevBuf<uint8_t> mask;
  std::vector<crtb200_rect> mask_rects;
  bool mask_valid = false, mask_needed = false;

  // frame queues and their plan
  std::vector<QueueSet> sets;
  Event fork_ev;
  DevBuf<unsigned long long> stats_dev;
  uint32_t cap_items = 0;
  uint32_t cap_depth = 0xFFFFFFFFu;
  uint32_t cap_sets = 0;
  uint32_t cap_branch = 0;    // worst-case children per ray-tree node the queues were planned for
  uint32_t n_chunks = 0;  // chunks of the current plan (chunk k runs on set k % cap_sets)
  uint32_t launches = 0;  // kernel launches of this GPU's part of the last frame
  // blocks per SM of k_coop's early pass (0 = final pass only); env CRT_COOP_EARLY.  Used for the primary level and the
  // shadow pass of frames that run on ONE stream (device frames, tile shards): with several chunk streams the tails
  // already overlap other chunks' work and waiting blocks would only take SM resources from them (run r2ad: 4.1 -> 8 ms);
  // the small secondary levels pay more for the extra launches and joins than they gain (hw11_room +2 %)
  int coop_early = CRT_COOP_MIN_BLOCKS;
  int blocks_closest = 0, blocks_closest_sec = 0, blocks_shadow = 0, blocks_coop = 0;

  // caller-supplied ray batches (crtb200_trace_rays_device, DESIGN.md 3.12): the query's own scratch on this GPU, a
  // QueueSet without ray queues or stream (work cursors and hand-off counters in ctl, hand-off records in ovf, the
  // early k_coop pass's side stream), its device counters and grid sizes
  QueueSet query;
  DevBuf<unsigned long long> query_stats_dev;
  int blocks_query_closest = 0, blocks_query_shadow = 0;
  bool query_ready = false;  // every part of the query scratch exists (set last by query_scratch)

  // progressive session: the accumulator of this GPU's tile shard, indexed by shard item
  DevBuf<float4> acc_sum, acc_sumsq;  // S and Q
  DevBuf<uint2> acc_hit;              // sample 0's primary hit {global triangle, bits(t)}

  Event multi_done;  // (GPUs after the first) its part of a multi-GPU pass is enqueued
};

// A context: one GPU, or several (crtb200_create_multi), and what exists once for all of them.  A multi-GPU frame's
// 8x4-pixel tiles are dealt round-robin over gpus (scene replicated); every GPU's k_store writes its pixels STRAIGHT
// into the first GPU's frame buffers through peer-mapped pointers (NVLink / NVSwitch), so no slab, gather or assemble
// pass exists.
struct crtb200_ctx {
  std::vector<std::unique_ptr<Gpu>> gpus;  // gpus[0]: the first GPU, which holds the frame and the caller's results
  std::vector<std::unique_ptr<Worker>> workers;  // workers[i - 1] enqueues for gpus[i]
  Event multi_fork;  // position of the caller's stream the other GPUs wait for before a multi-GPU pass

  // settings
  uint64_t queue_budget = 16ull << 30;
  uint32_t concurrency = 2;  // chunk streams of a host-bound frame (tools/e2e_time.py, run r2aq: 2 streams with one chunk each
                             // at 1080p, two each at 4K; 4 streams x 2 chunks cost 1080p frames 15-17 %)
  // sampling contract (crtb200_set_sampling); sampling.use_gi = 0: unsampled frames
  crtb200_sampling sampling{};

  // crtb200_upload_geometry: the trees it built, in the reference's numbering, kept on the first GPU of the context for
  // crtb200_scene_trees (40 bytes per node and 4 per mesh leaf reference; the top-level references are top_refs)
  bool trees_built = false;
  DevBuf<crtb200_kdnode> kd_nodes;
  DevBuf<uint32_t> kd_refs;
  std::vector<crtb200_mesh> kd_meshes;
  crtb200_trees kd_counts{};
  // the last upload's mesh records as given and its vertex count: crtb200_update_vertices_device rebuilds the trees
  // over the same meshes
  std::vector<crtb200_mesh> scene_meshes;
  uint32_t n_vertices = 0;

  // frame, on the first GPU
  DevBuf<float> frame;   // persistent colour buffer (RayTracer::colorBuffer, RayTracer.h:69)
  DevBuf<uint8_t> frame8;
  // crtb200_render_frames: frames alternate between (frame, frame8) and (frame_b, frame8_b); the device->host copy of
  // frame f runs on copy_stream while frame f + 1 is rendered into the other pair
  DevBuf<float> frame_b;
  DevBuf<uint8_t> frame8_b;
  Stream copy_stream;
  Event rendered[2], copied[2];
  DevBuf<HitRec> hits;
  Stream band_stream;  // device -> host band copies of a chunked host-bound frame
  Event band_done;
  std::vector<Event> chunk_done;
  std::vector<Event> dbg_ev;  // CRT_CHUNK_TIMES (tools): per chunk, end of k_store and end of its band copy
  uint32_t dbg_chunks = 0;

  // the last render: its span on the caller's stream, per-launch K2 / K3 timing events of the first GPU, statistics
  Event ev[2];
  std::vector<Event> kev;     // per-launch event pairs
  std::vector<int> kev_kind;  // 0 = closest, 1 = shadow, 2 / 3 their k_coop part (one entry per pair)
  size_t kev_used = 0;
  crtb200_stats last{};
  SideCounts last_side;
  uint32_t last_samples = 1;
  uint32_t frame_gpus = 1;     // GPUs whose device counters hold the last render's
  bool last_pending = false;   // crtb200_render_device: statistics not collected yet
  bool bands_copied = false;  // the last enqueue_frame copied its host destinations band by band

  // the last query (crtb200_trace_rays_device): span, GPU count and statistics
  Event query_ev[2];
  uint32_t query_gpus = 0;
  bool query_pending = false;
  crtb200_stats query_last{};

  // progressive session (crtb200_accum_*, DESIGN.md 3.10.1): the snapshots; each GPU keeps the accumulator of its own
  // tile shard
  bool acc_active = false;
  crtb200_camera acc_cam{};
  crtb200_options acc_opt{};
  std::vector<crtb200_rect> acc_rects;
  crtb200_sampling acc_smp{};
  uint32_t acc_done = 0;           // samples in the accumulator
  // adaptive session (crtb200_accum_begin_adaptive, DESIGN.md 3.10.2): the stop rule's parameters, and totals kept on
  // the host from each step's counters
  bool acc_adaptive = false;
  AdaptParams acc_ap{};
  uint64_t acc_covered = 0, acc_active_px = 0, acc_px_samples = 0;

  std::string error;                 // last error of a call on this context (crtb200_last_error_ctx)

  // joins the helper threads, then frees the GPUs after the first before it: their kernels store into its memory
  ~crtb200_ctx() {
    workers.clear();
    for (size_t i = gpus.size(); i-- > 0;) {
      cudaSetDevice(gpus[i]->device);  // the members free their buffers, streams and events on this device
      cudaStreamSynchronize(gpus[i]->stream);
      if (i) gpus[i].reset();
    }
  }
};
static void note_ctx_error(crtb200_ctx *c, const std::string &msg) { c->error = msg; }

extern "C" {

uint32_t crtb200_abi_version(void) { return CRTB200_ABI_VERSION; }
const char *crtb200_last_error(void) { return g_error.c_str(); }

int crtb200_device_count(int *count) {
  if (!count) return fail(CRTB200_ERR_ARG, "count is null");
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess) {
    *count = 0;
    return fail(CRTB200_ERR_CUDA, std::string("cudaGetDeviceCount: ") + cudaGetErrorString(e));
  }
  *count = n;
  return CRTB200_OK;
}

}  // extern "C"

// Adds GPU `device` to context c: device check, stream, occupancy grid sizes, tuning environment and, for a GPU after
// the first, access to the first GPU's memory (its kernels store into the first GPU's frame).
static int add_gpu(crtb200_ctx *c, int device) {
  int n = 0;
  CUDA_TRY(cudaGetDeviceCount(&n));
  if (device < 0 || device >= n) return fail(CRTB200_ERR_CUDA, "no such CUDA device (this library has no CPU fallback)");
  CUDA_TRY(cudaSetDevice(device));
  cudaDeviceProp prop;
  CUDA_TRY(cudaGetDeviceProperties(&prop, device));
  if (prop.major < 10)
    return fail(CRTB200_ERR_CUDA, std::string("device ") + prop.name + " is not sm_100-class; libcrtb200 is built for sm_100a only");
  c->gpus.emplace_back(new Gpu());
  Gpu &g = *c->gpus.back();
  g.device = device;
  g.sm_count = prop.multiProcessorCount;
  if (g.stream.create(cudaStreamNonBlocking) != cudaSuccess) return fail(CRTB200_ERR_CUDA, "cudaStreamCreate / cudaEventCreate failed");
  int occ = 0;
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_closest<CameraRays, true, false, CRT_REFILL_CLOSEST, CRT_LOOP_MODE, false, false>, CRT_TRAV_BLOCK, 0);
  g.blocks_closest = std::max(1, occ) * g.sm_count;
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_closest<QueueRays, false, false, CRT_REFILL_CLOSEST, CRT_LOOP_MODE, false, false>, CRT_TRAV_BLOCK, 0);
  g.blocks_closest_sec = std::max(1, occ) * g.sm_count;
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_shadow<ShadowPairs, 0, CRT_REFILL_SHADOW, CRT_LOOP_MODE, false, false>, CRT_TRAV_BLOCK, 0);
  g.blocks_shadow = std::max(1, occ) * g.sm_count;
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_coop<ShadowPairs, false, true, CRT_COOP_GROUP>, 32 * CRT_COOP_WARPS, 0);
  g.blocks_coop = std::max(1, occ) * g.sm_count;
  if (const char *env = getenv("CRT_BLOCKS_PER_SM")) {  // tuning only (tools/): resident persistent CTAs per SM
    const int b = atoi(env);
    if (b > 0) g.blocks_closest = g.blocks_closest_sec = g.blocks_shadow = b * g.sm_count;
  }
  if (const char *env = getenv("CRT_L2_PERSIST")) g.l2_persist = atoi(env);
  if (const char *env = getenv("CRT_TAIL_ITERS")) g.tail_iters = std::max(-1, atoi(env));
  if (const char *env = getenv("CRT_TAIL_CAP")) g.tail_cap = std::max(1, atoi(env));
  if (const char *env = getenv("CRT_TAIL_START")) g.tail_start = g.tail_start_closest = std::max(0, atoi(env));
  if (const char *env = getenv("CRT_TAIL_START_CLOSEST")) g.tail_start_closest = std::max(0, atoi(env));
  if (const char *env = getenv("CRT_TAIL_SMALL")) g.tail_small = std::max(0, atoi(env));
  if (const char *env = getenv("CRT_COOP_EARLY")) g.coop_early = std::max(0, std::min(CRT_COOP_MIN_BLOCKS, atoi(env)));
  g.l2_persist_max = (size_t)std::max(0, prop.persistingL2CacheMaxSize);
  g.l2_window_max = (size_t)std::max(0, prop.accessPolicyMaxWindowSize);
  if (g.l2_persist && g.l2_persist_max)
    cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, g.l2_persist_max);  // best effort: a refusal only loses the hint
  if (getenv("CRT_VERBOSE"))
    fprintf(stderr, "[crtb200] %s: %d SMs, L2 %d MiB, persisting L2 max %zu MiB, access-policy window max %zu MiB, persist %s\n", prop.name,
            prop.multiProcessorCount, prop.l2CacheSize >> 20, g.l2_persist_max >> 20, g.l2_window_max >> 20, g.l2_persist ? "on" : "off");
  if (c->gpus.size() == 1) return CRTB200_OK;
  const int first = c->gpus[0]->device;
  if (device != first) {
    int can = 0;
    cudaError_t e = cudaDeviceCanAccessPeer(&can, device, first);
    if (e == cudaSuccess && !can) e = cudaErrorPeerAccessUnsupported;
    if (e == cudaSuccess) e = cudaDeviceEnablePeerAccess(first, 0);
    if (e == cudaErrorPeerAccessAlreadyEnabled) {
      cudaGetLastError();
      e = cudaSuccess;
    }
    if (e != cudaSuccess)
      return fail(CRTB200_ERR_CUDA, std::string("peer access from device ") + std::to_string(device) + " to device " +
                                        std::to_string(first) + ": " + cudaGetErrorString(e));
  }
  if (g.multi_done.create(cudaEventDisableTiming) != cudaSuccess) return fail(CRTB200_ERR_CUDA, "cudaEventCreate failed");
  c->workers.emplace_back(new Worker());
  return CRTB200_OK;
}

// A context over the devices ids[0..n), the first device's current on return
static int create(const int *ids, int n, crtb200_ctx **out) {
  std::unique_ptr<crtb200_ctx> c(new crtb200_ctx());
  for (int i = 0; i < n; i++) {
    const int rc = add_gpu(c.get(), ids[i]);
    if (rc) return rc;
    if (i == 0 && (c->ev[0].create(cudaEventDefault) != cudaSuccess || c->ev[1].create(cudaEventDefault) != cudaSuccess))
      return fail(CRTB200_ERR_CUDA, "cudaStreamCreate / cudaEventCreate failed");
  }
  cudaSetDevice(ids[0]);
  if (n > 1 && c->multi_fork.create(cudaEventDisableTiming) != cudaSuccess) return fail(CRTB200_ERR_CUDA, "cudaEventCreate failed");
  *out = c.release();
  return CRTB200_OK;
}

extern "C" {

int crtb200_create(int device, crtb200_ctx **out) {
  if (!out) return fail(CRTB200_ERR_ARG, "out is null");
  *out = nullptr;
  return create(&device, 1, out);
}

const char *crtb200_last_error_ctx(const crtb200_ctx *c) { return c ? c->error.c_str() : g_error.c_str(); }

int crtb200_create_multi(const int *device_ids, int n, crtb200_ctx **out) {
  if (!out) return fail(CRTB200_ERR_ARG, "out is null");
  *out = nullptr;
  if (!device_ids || n < 1 || n > 64) return fail(CRTB200_ERR_ARG, "device list is null or its length is not in 1..64");
  return create(device_ids, n, out);
}

int crtb200_device_list(const crtb200_ctx *c, int *device_ids, int capacity, int *count) {
  if (!c || !count) return fail(CRTB200_ERR_ARG, "null argument");
  *count = (int)c->gpus.size();
  if (device_ids)
    for (int i = 0; i < capacity && i < *count; i++) device_ids[i] = c->gpus[i]->device;
  return CRTB200_OK;
}

int crtb200_destroy(crtb200_ctx *c) {
  delete c;
  return CRTB200_OK;
}

int crtb200_set_concurrency(crtb200_ctx *c, uint32_t chunks_in_flight) {
  ErrScope scope(c);
  if (!c) return fail(CRTB200_ERR_ARG, "ctx is null");
  if (chunks_in_flight < 1 || chunks_in_flight > 16) return fail(CRTB200_ERR_ARG, "concurrency must be 1..16");
  c->concurrency = chunks_in_flight;
  for (auto &g : c->gpus) g->cap_items = 0;
  return CRTB200_OK;
}

int crtb200_set_sampling(crtb200_ctx *c, const crtb200_sampling *s) {
  ErrScope scope(c);
  if (!c) return fail(CRTB200_ERR_ARG, "ctx is null");
  crtb200_sampling v{};
  if (s && s->use_gi) {
    if (s->rays_per_pixel == 0) return fail(CRTB200_ERR_ARG, "rays_per_pixel must be at least 1 with GI on");
    if (s->gi_samples > 1024) return fail(CRTB200_ERR_ARG, "gi_samples must be at most 1024");
    v = *s;
    v.use_gi = 1;
  }
  c->sampling = v;
  return CRTB200_OK;
}

int crtb200_last_sampling_stats(crtb200_ctx *c, crtb200_sampling_stats *stats) {
  ErrScope scope(c);
  if (!c || !stats) return fail(CRTB200_ERR_ARG, "null argument");
  crtb200_stats unused;
  const int rc = crtb200_last_stats(c, &unused);  // synchronises a pending render_device frame
  if (rc) return rc;
  stats->rays_diffuse = c->last_side.diffuse;
  stats->samples = c->last_samples;
  stats->reserved = 0;
  return CRTB200_OK;
}

int crtb200_set_queue_budget(crtb200_ctx *c, uint64_t bytes) {
  ErrScope scope(c);
  if (!c) return fail(CRTB200_ERR_ARG, "ctx is null");
  if (bytes < (64ull << 20)) return fail(CRTB200_ERR_ARG, "queue budget must be at least 64 MiB");
  c->queue_budget = bytes;
  for (auto &g : c->gpus) g->cap_items = 0;
  return CRTB200_OK;
}

// ---- host flattener H1: reference-numbered tree -> visiting-order, skip-linked nodes -------------------------
// The reference pops child[1] before child[0] (it pushes 0 then 1 on a std::stack, KDTree.cpp:65-72), visits every
// node whose box passes, and never reorders.  So the visiting order is a fixed total order of the nodes and a failed
// slab test simply jumps over the node's subtree.
static bool relayout_tree(const crtb200_kdnode *nodes, uint32_t n, uint32_t out_base, uint32_t ref_base,
                          uint32_t ref_count, std::vector<float4> &out, std::string &err, uint32_t *max_depth = nullptr) {
  if (max_depth) *max_depth = 0;
  if (n == 0) return true;
  std::vector<uint32_t> order;
  order.reserve(n);
  std::vector<uint32_t> stack;
  std::vector<uint8_t> seen(n, 0);
  stack.push_back(0);
  while (!stack.empty()) {
    uint32_t i = stack.back();
    stack.pop_back();
    if (i >= n) {
      err = "kd node child index out of range";
      return false;
    }
    if (seen[i]) {
      err = "kd tree is not a tree (node reachable twice)";
      return false;
    }
    seen[i] = 1;
    order.push_back(i);
    const crtb200_kdnode &nd = nodes[i];
    if (nd.leaf_count == 0) {
      if (nd.child[0] != CRTB200_INVALID) stack.push_back(nd.child[0]);
      if (nd.child[1] != CRTB200_INVALID) stack.push_back(nd.child[1]);
    } else if ((uint64_t)nd.leaf_start + nd.leaf_count > ref_count) {
      err = "kd leaf reference range out of bounds";
      return false;
    }
  }
  const uint32_t m = (uint32_t)order.size();
  if (max_depth) {  // order is a pre-order: a parent precedes its children
    std::vector<uint32_t> depth(n, 1);
    for (uint32_t k = 0; k < m; k++) {
      const crtb200_kdnode &nd = nodes[order[k]];
      *max_depth = std::max(*max_depth, depth[order[k]]);
      if (nd.leaf_count == 0)
        for (int side = 0; side < 2; side++)
          if (nd.child[side] != CRTB200_INVALID) depth[nd.child[side]] = depth[order[k]] + 1;
    }
  }
  std::vector<uint32_t> newidx(n, 0), size(n, 1);
  for (uint32_t k = 0; k < m; k++) newidx[order[k]] = k;
  for (uint32_t k = m; k-- > 0;) {
    const crtb200_kdnode &nd = nodes[order[k]];
    uint32_t s = 1;
    if (nd.leaf_count == 0) {
      if (nd.child[0] != CRTB200_INVALID) s += size[nd.child[0]];
      if (nd.child[1] != CRTB200_INVALID) s += size[nd.child[1]];
    }
    size[order[k]] = s;
  }
  out.resize(2 * (size_t)(out_base + m));
  for (uint32_t k = 0; k < m; k++) {
    const crtb200_kdnode &nd = nodes[order[k]];
    uint32_t a, b;
    if (nd.leaf_count) {
      a = CRT_LEAF_FLAG | nd.leaf_count;
      b = ref_base + nd.leaf_start;
    } else {
      a = out_base + k + size[order[k]];
      // b = the child visited second (child[0] when both exist): k_coop pushes both children of a passing node at once
      b = (nd.child[0] != CRTB200_INVALID && nd.child[1] != CRTB200_INVALID) ? out_base + newidx[nd.child[0]] : CRT_INVALID;
    }
    float4 lo = make_float4(nd.box_min[0], nd.box_min[1], nd.box_min[2], 0.f);
    float4 hi = make_float4(nd.box_max[0], nd.box_max[1], nd.box_max[2], 0.f);
    std::memcpy(&lo.w, &a, 4);
    std::memcpy(&hi.w, &b, 4);
    out[2 * (size_t)(out_base + k)] = lo;
    out[2 * (size_t)(out_base + k) + 1] = hi;
  }
  return true;
}

static bool box_nested(const crtb200_kdnode &parent, const crtb200_kdnode &child) {
  for (int k = 0; k < 3; k++)
    if (!(child.box_min[k] >= parent.box_min[k]) || !(child.box_max[k] <= parent.box_max[k]) || !(child.box_min[k] <= child.box_max[k]))
      return false;
  return true;
}

// ---- culling margin of one mesh (crt_device.cuh "Conservative culling", DESIGN.md section 3.6) -----------------------
// mu = overhang + 4 * slop + 64 ulp * |coordinates|, in double:
//   overhang  how far the bounding box of a triangle sticks out of a leaf that lists it (max over all leaf references):
//             then bbox(T) lies inside L inflated by overhang for EVERY leaf L through which the reference can meet T
//   slop      how far outside T a point can lie and still pass Triangle::pointIsInTriangle's -FLT_EPSILON tests
//             (Triangle.cpp:37-57): eps * (1 + 8 e^2) * perimeter / (2 * area), e = longest edge (rounding of the edge
//             functions included); x4 for safety
//   the ulp term covers the rounding of the hit point and of the slab parameters for this mesh's extent (the ray
//   origin's share is added per ray, cull_margin_for)
// +inf (never cull) when the tree does not nest or a triangle's uploaded normal is not its geometric unit normal (then
// the slop bound does not describe what the triangle test accepts).  Zero-area triangles with a zero / non-finite
// normal are harmless: they never yield a finite t (Ray.cpp:11-18).
static float mesh_cull_margin(const crtb200_scene *s, const crtb200_mesh &me, bool nested) {
  const float inf = std::numeric_limits<float>::infinity();
  if (!nested) return inf;
  double overhang = 0.0, slop = 0.0, absmax = 0.0;
  const crtb200_kdnode *nodes = s->mesh_nodes + me.first_node;
  for (uint32_t k = 0; k < me.n_nodes; k++) {
    const crtb200_kdnode &nd = nodes[k];
    for (int i = 0; i < 3; i++) absmax = std::max(absmax, std::max(std::fabs((double)nd.box_min[i]), std::fabs((double)nd.box_max[i])));
    for (uint32_t q = 0; q < nd.leaf_count; q++) {
      const uint32_t *iv = s->triangle_vertex + 3 * (size_t)(me.first_triangle + s->mesh_leaf_refs[me.first_leaf_ref + nd.leaf_start + q]);
      for (int i = 0; i < 3; i++) {
        const double x0 = s->vertex_position[3 * (size_t)iv[0] + i], x1 = s->vertex_position[3 * (size_t)iv[1] + i],
                     x2 = s->vertex_position[3 * (size_t)iv[2] + i];
        const double lo = std::min(x0, std::min(x1, x2)), hi = std::max(x0, std::max(x1, x2));
        overhang = std::max(overhang, std::max((double)nd.box_min[i] - lo, hi - (double)nd.box_max[i]));
      }
    }
  }
  for (uint32_t t = 0; t < me.n_triangles; t++) {
    const uint32_t *iv = s->triangle_vertex + 3 * (size_t)(me.first_triangle + t);
    double p[3][3];
    for (int v = 0; v < 3; v++)
      for (int i = 0; i < 3; i++) {
        p[v][i] = s->vertex_position[3 * (size_t)iv[v] + i];
        absmax = std::max(absmax, std::fabs(p[v][i]));
      }
    double len[3];
    for (int k = 0; k < 3; k++) {
      const double *a = p[k], *b = p[(k + 1) % 3];
      len[k] = std::sqrt((b[0] - a[0]) * (b[0] - a[0]) + (b[1] - a[1]) * (b[1] - a[1]) + (b[2] - a[2]) * (b[2] - a[2]));
    }
    const double u[3] = {p[1][0] - p[0][0], p[1][1] - p[0][1], p[1][2] - p[0][2]};
    const double w[3] = {p[2][0] - p[0][0], p[2][1] - p[0][1], p[2][2] - p[0][2]};
    const double cr[3] = {u[1] * w[2] - u[2] * w[1], u[2] * w[0] - u[0] * w[2], u[0] * w[1] - u[1] * w[0]};
    const double a2 = std::sqrt(cr[0] * cr[0] + cr[1] * cr[1] + cr[2] * cr[2]);
    const float *nn = s->triangle_normal + 3 * (size_t)(me.first_triangle + t);
    if (!(a2 > 0.0) || !std::isfinite(a2)) {
      for (int i = 0; i < 3; i++)
        if (std::isfinite(nn[i]) && nn[i] != 0.0f) return inf;
      continue;
    }
    for (int i = 0; i < 3; i++)
      if (!(std::fabs((double)nn[i] - cr[i] / a2) <= 1e-3)) return inf;
    const double emax = std::max(len[0], std::max(len[1], len[2]));
    slop = std::max(slop, (double)CRT_FLT_EPSILON * (1.0 + 8.0 * emax * emax) * (len[0] + len[1] + len[2]) / a2);
  }
  const double mu = overhang + 4.0 * slop + 64.0 * (double)CRT_FLT_EPSILON * absmax;
  return (std::isfinite(mu) && mu < 1e30) ? (float)(mu * (1.0 + 1e-6)) : inf;
}

}  // extern "C"

static int upload_one(crtb200_ctx *c, Gpu &g, const crtb200_scene *s);
static int upload_geometry_one(crtb200_ctx *c, Gpu &g, const crtb200_scene *s, bool keep);

// ends the progressive session of a context and frees its accumulators on every GPU
static void accum_release(crtb200_ctx *c) {
  c->acc_active = false;
  c->acc_adaptive = false;
  c->acc_done = 0;
  c->acc_covered = c->acc_active_px = c->acc_px_samples = 0;
  c->acc_rects.clear();
  for (auto &g : c->gpus) {
    cudaSetDevice(g->device);
    g->acc_sum.release();
    g->acc_sumsq.release();
    g->acc_hit.release();
  }
  cudaSetDevice(c->gpus[0]->device);
}

// runs fn(i, gpus[i]) for every GPU of the context, i > 0 on GPU i's helper thread and i = 0 on the calling thread;
// first error wins, a later GPU's prefixed with its device
template <typename F>
static int on_all_devices(crtb200_ctx *c, F fn) {
  const size_t n = c->gpus.size();
  std::vector<int> rcs(n, 0);
  std::vector<std::string> msgs(n);
  for (size_t i = 1; i < n; i++) {
    c->workers[i - 1]->post([&, i] {
      rcs[i] = fn(i, *c->gpus[i]);
      if (rcs[i]) msgs[i] = g_error;
    });
  }
  int rc = fn(0, *c->gpus[0]);
  for (size_t i = 1; i < n; i++) {
    c->workers[i - 1]->wait();
    if (rc == CRTB200_OK && rcs[i]) rc = fail(rcs[i], "device " + std::to_string(c->gpus[i]->device) + ": " + msgs[i]);
  }
  return rc;
}

// One multi-GPU pass over gpus[0..n): fn(i, gpu, stream) enqueues GPU i's part, GPU 0's on the caller's stream st and
// every other GPU's on its own stream, which first waits for st's position.  on_workers: the other GPUs enqueue on
// their helper threads (on_all_devices); otherwise they enqueue on the calling thread in order, up to the first that
// fails.  st then waits for every GPU that started, also when a later one failed: what it enqueued writes into the
// first GPU's memory.
template <typename F>
static int fan_out(crtb200_ctx *c, uint32_t n, cudaStream_t st, bool on_workers, F fn) {
  CUDA_TRY(cudaSetDevice(c->gpus[0]->device));
  if (n > 1) CUDA_TRY(cudaEventRecord(c->multi_fork, st));
  std::vector<uint8_t> started(n, 0);
  auto part = [&](size_t i, Gpu &g) -> int {
    if (i == 0) return fn(0u, g, st);
    CUDA_TRY(cudaSetDevice(g.device));
    CUDA_TRY(cudaStreamWaitEvent(g.stream, c->multi_fork, 0));
    started[i] = 1;
    int rc = fn((uint32_t)i, g, (cudaStream_t)g.stream);
    if (cudaEventRecord(g.multi_done, g.stream) != cudaSuccess && rc == CRTB200_OK) rc = fail(CRTB200_ERR_CUDA, "cudaEventRecord failed");
    return rc;
  };
  int rc = CRTB200_OK;
  if (on_workers)
    rc = on_all_devices(c, part);
  else
    for (uint32_t i = 0; i < n && rc == CRTB200_OK; i++) rc = part(i, *c->gpus[i]);
  CUDA_TRY(cudaSetDevice(c->gpus[0]->device));
  for (uint32_t i = 1; i < n; i++)
    if (started[i]) CUDA_TRY(cudaStreamWaitEvent(st, c->gpus[i]->multi_done, 0));
  return rc;
}

extern "C" {

int crtb200_upload_scene(crtb200_ctx *c, const crtb200_scene *s) {
  if (!c || !s) return fail(CRTB200_ERR_ARG, "null argument");
  ErrScope scope(c);
  if (c->acc_active) accum_release(c);  // a new scene ends the progressive session
  c->trees_built = false;
  c->kd_nodes.release();
  c->kd_refs.release();
  // scene replicated on every GPU (SURVEY 8(e)); the host relayout runs once per GPU, in parallel
  const int rc = on_all_devices(c, [&](size_t, Gpu &g) { return upload_one(c, g, s); });
  if (rc == CRTB200_OK) {
    c->scene_meshes.assign(s->meshes, s->meshes + s->n_meshes);
    c->n_vertices = s->n_vertices;
  }
  return rc;
}

int crtb200_upload_geometry(crtb200_ctx *c, const crtb200_scene *s) {
  if (!c || !s) return fail(CRTB200_ERR_ARG, "null argument");
  ErrScope scope(c);
  if (s->n_mesh_nodes || s->n_mesh_leaf_refs || s->n_top_nodes || s->n_top_leaf_refs || s->mesh_nodes || s->mesh_leaf_refs ||
      s->top_nodes || s->top_leaf_refs)
    return fail(CRTB200_ERR_ARG, "crtb200_upload_geometry builds the trees: the scene's tree counts must be 0 and their arrays NULL");
  if (c->acc_active) accum_release(c);
  c->trees_built = false;
  c->kd_nodes.release();
  c->kd_refs.release();
  // one build per GPU, in parallel; only the first GPU keeps the reference-numbered trees for crtb200_scene_trees
  const int rc = on_all_devices(c, [&](size_t i, Gpu &g) { return upload_geometry_one(c, g, s, i == 0); });
  if (rc) {
    c->trees_built = false;
    c->kd_nodes.release();
    c->kd_refs.release();
  } else {
    c->scene_meshes.assign(s->meshes, s->meshes + s->n_meshes);
    c->n_vertices = s->n_vertices;
  }
  return rc;
}

}  // extern "C"

// What both upload paths build on the host from the scene's arrays (everything but the trees), after validating them.
struct SceneRecords {
  std::vector<float4> geom;
  std::vector<uint4> shade;
  std::vector<float4> vn;
  std::vector<float2> uv;
  std::vector<DMaterial> mats;
  std::vector<DTexture> texs;
  std::vector<float> texels;
  std::vector<DLight> lights;
};

// Validation and host records of the triangles, vertices, materials, textures and lights; `trees`: also check the
// meshes' node and leaf-reference ranges (crtb200_upload_scene).  Selects g's device and drops its scene.
static int pack_records(Gpu &g, const crtb200_scene *s, bool trees, SceneRecords &r) {
  if (s->abi_version != CRTB200_ABI_VERSION) return fail(CRTB200_ERR_ARG, "crtb200_scene.abi_version mismatch");
  if (s->width == 0 || s->height == 0) return fail(CRTB200_ERR_SCENE, "image size is zero");
  if ((uint64_t)s->width * s->height > 0x7FFFFFFFull / 4) return fail(CRTB200_ERR_SCENE, "image too large");
  if ((s->n_vertices && (!s->vertex_position || !s->vertex_normal)) || (s->n_triangles && (!s->triangle_vertex || !s->triangle_normal)) ||
      (s->n_meshes && !s->meshes) || (s->n_materials && !s->materials) || (s->n_lights && !s->lights) ||
      (s->n_textures && !s->textures) || (s->n_mesh_nodes && !s->mesh_nodes) || (s->n_top_nodes && !s->top_nodes) ||
      (s->n_mesh_leaf_refs && !s->mesh_leaf_refs) || (s->n_top_leaf_refs && !s->top_leaf_refs))
    return fail(CRTB200_ERR_SCENE, "a non-empty scene array is null");
  if (s->n_triangles >= 0x7FFFFFFFu || s->n_mesh_nodes >= 0x7FFFFFF0u) return fail(CRTB200_ERR_SCENE, "scene too large for 31-bit indices");
  CUDA_TRY(cudaSetDevice(g.device));
  g.have_scene = false;

  // triangles
  r.geom.resize(3 * (size_t)s->n_triangles);
  r.shade.resize(s->n_triangles);
  std::vector<uint32_t> tri_mesh(s->n_triangles, CRTB200_INVALID);
  for (uint32_t m = 0; m < s->n_meshes; m++) {
    const crtb200_mesh &me = s->meshes[m];
    if ((uint64_t)me.first_triangle + me.n_triangles > s->n_triangles) return fail(CRTB200_ERR_SCENE, "mesh triangle range out of bounds");
    if (me.material >= s->n_materials) return fail(CRTB200_ERR_SCENE, "mesh material index out of range");
    if (trees && (uint64_t)me.first_node + me.n_nodes > s->n_mesh_nodes) return fail(CRTB200_ERR_SCENE, "mesh node range out of bounds");
    if (trees && (uint64_t)me.first_leaf_ref + me.n_leaf_refs > s->n_mesh_leaf_refs) return fail(CRTB200_ERR_SCENE, "mesh leaf-ref range out of bounds");
    for (uint32_t t = 0; t < me.n_triangles; t++) tri_mesh[me.first_triangle + t] = m;
  }
  for (uint32_t t = 0; t < s->n_triangles; t++) {
    const uint32_t *iv = s->triangle_vertex + 3 * (size_t)t;
    if (iv[0] >= s->n_vertices || iv[1] >= s->n_vertices || iv[2] >= s->n_vertices) return fail(CRTB200_ERR_SCENE, "triangle vertex index out of range");
    if (tri_mesh[t] == CRTB200_INVALID) return fail(CRTB200_ERR_SCENE, "triangle not owned by any mesh");
    const float *n = s->triangle_normal + 3 * (size_t)t;
    for (int k = 0; k < 3; k++) {
      const float *p = s->vertex_position + 3 * (size_t)iv[k];
      r.geom[3 * (size_t)t + k] = make_float4(p[0], p[1], p[2], n[k]);
    }
    r.shade[t] = make_uint4(iv[0], iv[1], iv[2], tri_mesh[t]);
  }

  r.vn.resize(s->n_vertices);
  for (uint32_t v = 0; v < s->n_vertices; v++)
    r.vn[v] = make_float4(s->vertex_normal[3 * (size_t)v], s->vertex_normal[3 * (size_t)v + 1], s->vertex_normal[3 * (size_t)v + 2], 0.f);
  if (s->vertex_uv) {
    r.uv.resize(s->n_vertices);
    for (uint32_t v = 0; v < s->n_vertices; v++) r.uv[v] = make_float2(s->vertex_uv[3 * (size_t)v], s->vertex_uv[3 * (size_t)v + 1]);
  }
  r.mats.resize(s->n_materials);
  for (uint32_t m = 0; m < s->n_materials; m++) {
    const crtb200_material &mm = s->materials[m];
    if (mm.texture != CRTB200_INVALID && mm.texture >= s->n_textures) return fail(CRTB200_ERR_SCENE, "material texture index out of range");
    r.mats[m].type = mm.type;
    r.mats[m].smooth = mm.smooth_shading;
    r.mats[m].texture = mm.texture;
    r.mats[m].ior = mm.ior;
    for (int k = 0; k < 3; k++) r.mats[m].albedo[k] = mm.albedo[k];
    r.mats[m].pad = 0.f;
  }
  r.texs.resize(s->n_textures);
  for (uint32_t t = 0; t < s->n_textures; t++) {
    const crtb200_texture &tt = s->textures[t];
    DTexture &d = r.texs[t];
    d.kind = tt.kind;
    for (int k = 0; k < 3; k++) {
      d.color_a[k] = tt.color_a[k];
      d.color_b[k] = tt.color_b[k];
    }
    d.scalar = tt.scalar;
    d.width = tt.width;
    d.height = tt.height;
    d.texel_offset = tt.texel_offset;
    if (tt.kind == CRTB200_TEX_BITMAP) {
      if (tt.width == 0 || tt.height == 0 || tt.texel_offset + (uint64_t)tt.width * tt.height > s->n_texels || !s->texels)
        return fail(CRTB200_ERR_SCENE, "bitmap texture texel range out of bounds");
    }
  }
  r.texels.assign(s->texels ? s->texels : nullptr, s->texels ? s->texels + 3 * s->n_texels : nullptr);
  r.lights.resize(s->n_lights);
  for (uint32_t l = 0; l < s->n_lights; l++) {
    for (int k = 0; k < 3; k++) r.lights[l].pos[k] = s->lights[l].position[k];
    r.lights[l].intensity = static_cast<float>(s->lights[l].intensity);  // RayTracer.cpp:320
  }
  return CRTB200_OK;
}

// The scene arena (nodes | leaf references | triangle geometry, one allocation, see Gpu::arena) for n_nodes
// nodes, n_refs mesh leaf references and the scene's triangles.
static int place_arena(Gpu &g, size_t n_nodes, size_t n_refs, size_t n_geom) {
  auto al = [](size_t v) { return (v + 255) & ~(size_t)255; };
  const size_t b_nodes = al(n_nodes * 2 * sizeof(float4)), b_refs = al(n_refs * sizeof(uint32_t)), b_geom = al(n_geom * sizeof(float4));
  g.arena_used = b_nodes + b_refs + b_geom;
  g.nodes_bytes = b_nodes;
  CUDA_TRY(g.arena.ensure(std::max<size_t>(g.arena_used, 256)));
  g.nodes_p = reinterpret_cast<float4 *>(g.arena.p);
  g.leaf_refs_p = reinterpret_cast<uint32_t *>(g.arena.p + b_nodes);
  g.tri_geom_p = reinterpret_cast<float4 *>(g.arena.p + b_nodes + b_refs);
  return CRTB200_OK;
}

// The trees' part of GPU g's device scene, once the arena (nodes, references, triangle records), top_refs and meshes
// hold them: pointers, counts, the top-level tree's node range and the nesting flag.
static void commit_trees(Gpu &g, uint32_t n_meshes, uint32_t n_nodes, uint32_t n_refs, uint32_t n_top_refs, uint32_t top_begin,
                         uint32_t top_end, bool nested_ok) {
  g.n_nodes = n_nodes;
  g.n_leaf_refs = n_refs;
  g.n_top_refs = n_top_refs;
  g.nested_ok = nested_ok;
  DScene &d = g.sc;
  d.nodes = g.nodes_p;
  d.leaf_refs = g.leaf_refs_p;
  d.top_refs = g.top_refs.p;
  d.tri_geom = g.tri_geom_p;
  d.meshes = g.meshes.p;
  d.n_meshes = n_meshes;
  d.top_begin = top_begin;
  d.top_end = top_end;
  d.dedup_meshes = n_meshes <= 64 ? 1u : (n_meshes <= 512 ? 2u : 0u);
  d.dedup_words = d.dedup_meshes == 2u ? (n_meshes + 31u) / 32u : 0u;
}

// Uploads the records to GPU g and completes its device scene, and on the context's first GPU the frame buffers; the
// trees are committed (commit_trees).
static int commit_records(crtb200_ctx *c, Gpu &g, const crtb200_scene *s, const SceneRecords &r) {
  g.has_reflective = g.has_refractive = false;
  for (uint32_t m = 0; m < s->n_meshes; m++) {
    const uint32_t type = s->materials[s->meshes[m].material].type;
    if (type == CRTB200_MAT_REFLECTIVE) g.has_reflective = true;
    if (type == CRTB200_MAT_REFRACTIVE) g.has_refractive = true;
  }
  CUDA_TRY(g.tri_shade.upload(r.shade));
  CUDA_TRY(g.vtx_normal.upload(r.vn));
  if (!r.uv.empty()) CUDA_TRY(g.vtx_uv.upload(r.uv));
  CUDA_TRY(g.materials.upload(r.mats));
  CUDA_TRY(g.textures.upload(r.texs));
  CUDA_TRY(g.texels.upload(r.texels));
  CUDA_TRY(g.lights.upload(r.lights));
  g.n_triangles = s->n_triangles;

  DScene &d = g.sc;
  d.tri_shade = g.tri_shade.p;
  d.vtx_normal = g.vtx_normal.p;
  d.vtx_uv = r.uv.empty() ? nullptr : g.vtx_uv.p;
  d.materials = g.materials.p;
  d.textures = g.textures.p;
  d.texels = g.texels.p;
  d.lights = g.lights.p;
  d.n_lights = s->n_lights;
  d.width = s->width;
  d.height = s->height;
  for (int k = 0; k < 3; k++) d.bg[k] = s->background[k];

  const size_t px = (size_t)s->width * s->height;
  if (&g == c->gpus[0].get()) {
    CUDA_TRY(c->frame.ensure(px * 3));
    CUDA_TRY(cudaMemset(c->frame.p, 0, px * 3 * sizeof(float)));  // colorBuffer starts at (0,0,0), RayTracer.cpp:47-50
    CUDA_TRY(c->frame8.ensure(px * 3));
    CUDA_TRY(cudaMemset(c->frame8.p, 0, px * 3));
  }
  CUDA_TRY(g.stats_dev.ensure(CRT_STAT_SLOTS));
  g.mask_valid = false;
  g.cap_items = 0;
  g.have_scene = true;
  return CRTB200_OK;
}

static int upload_one(crtb200_ctx *c, Gpu &g, const crtb200_scene *s) {
  SceneRecords r;
  int rc = pack_records(g, s, true, r);
  if (rc) return rc;
  // trees: mesh trees first, top-level tree last, one node array
  std::vector<float4> nodes;
  bool nested_ok = true;
  std::vector<uint32_t> refs(s->n_mesh_leaf_refs);
  std::vector<DMesh> meshes(s->n_meshes);
  uint32_t node_cursor = 0;
  std::string err;
  for (uint32_t m = 0; m < s->n_meshes; m++) {
    const crtb200_mesh &me = s->meshes[m];
    for (uint32_t k = 0; k < me.n_leaf_refs; k++) {
      uint32_t local = s->mesh_leaf_refs[me.first_leaf_ref + k];
      if (local >= me.n_triangles) return fail(CRTB200_ERR_SCENE, "mesh leaf reference out of range");
      refs[me.first_leaf_ref + k] = me.first_triangle + local;
    }
    const size_t before = nodes.size() / 2;
    uint32_t depth = 0;
    if (!relayout_tree(s->mesh_nodes + me.first_node, me.n_nodes, node_cursor, me.first_leaf_ref, me.n_leaf_refs, nodes, err, &depth))
      return fail(CRTB200_ERR_SCENE, err);
    if (depth > 40) nested_ok = false;  // k_coop's LIFOs are sized for trees up to this deep (the reference's limit is 26 levels)
    const uint32_t placed = (uint32_t)(nodes.size() / 2 - before);
    meshes[m].node_begin = node_cursor;
    meshes[m].node_end = node_cursor + placed;
    meshes[m].material = me.material;
    meshes[m].first_triangle = me.first_triangle;
    meshes[m].cull_margin = std::numeric_limits<float>::infinity();
    node_cursor += placed;
    for (uint32_t k = 0; k < me.n_nodes && nested_ok; k++) {  // relayout_tree has validated the child indices
      const crtb200_kdnode &p = s->mesh_nodes[me.first_node + k];
      for (int k3 = 0; k3 < 3; k3++)
        if (!(p.box_min[k3] <= p.box_max[k3])) nested_ok = false;
      if (p.leaf_count) continue;
      for (int side = 0; side < 2; side++)
        if (p.child[side] != CRTB200_INVALID && !box_nested(p, s->mesh_nodes[me.first_node + p.child[side]])) nested_ok = false;
    }
  }
  for (uint32_t k = 0; k < s->n_top_leaf_refs; k++)
    if (s->top_leaf_refs[k] >= s->n_meshes) return fail(CRTB200_ERR_SCENE, "top-level leaf reference out of range");
  const uint32_t top_begin = node_cursor;
  {
    const size_t before = nodes.size() / 2;
    if (!relayout_tree(s->top_nodes, s->n_top_nodes, node_cursor, 0, s->n_top_leaf_refs, nodes, err)) return fail(CRTB200_ERR_SCENE, err);
    node_cursor += (uint32_t)(nodes.size() / 2 - before);
  }
  const uint32_t top_end = node_cursor;
  // culling margins (one pass over the leaf references and the triangles of each mesh; meshes in parallel would be easy,
  // but this is 0.1 s per million triangles)
  for (uint32_t m = 0; m < s->n_meshes; m++) meshes[m].cull_margin = mesh_cull_margin(s, s->meshes[m], nested_ok);
  std::vector<uint32_t> top_refs(s->top_leaf_refs, s->top_leaf_refs + s->n_top_leaf_refs);

  rc = place_arena(g, nodes.size() / 2, refs.size(), r.geom.size());
  if (rc) return rc;
  if (!nodes.empty()) CUDA_TRY(cudaMemcpy(g.nodes_p, nodes.data(), nodes.size() * sizeof(float4), cudaMemcpyHostToDevice));
  if (!refs.empty()) CUDA_TRY(cudaMemcpy(g.leaf_refs_p, refs.data(), refs.size() * sizeof(uint32_t), cudaMemcpyHostToDevice));
  if (!r.geom.empty()) CUDA_TRY(cudaMemcpy(g.tri_geom_p, r.geom.data(), r.geom.size() * sizeof(float4), cudaMemcpyHostToDevice));
  CUDA_TRY(g.top_refs.upload(top_refs));
  CUDA_TRY(g.meshes.upload(meshes));
  commit_trees(g, s->n_meshes, (uint32_t)(nodes.size() / 2), (uint32_t)refs.size(), (uint32_t)top_refs.size(), top_begin, top_end, nested_ok);
  return commit_records(c, g, s, r);
}

// ---- device KD build: crtb200_upload_geometry (csrc/crt_build.cuh, DESIGN.md 3.11) -------------------------------
// Scratch of one build, freed when the build returns (cudaFree synchronises the device); `peak` is what
// crtb200_scene_trees reports.
struct BuildScratch {
  std::vector<std::pair<void *, size_t>> live_ptrs;
  size_t live = 0, peak = 0;
  template <typename T>
  bool alloc(T *&p, size_t n) {
    p = nullptr;
    const size_t bytes = std::max<size_t>(n, 1) * sizeof(T);
    if (cudaMalloc(reinterpret_cast<void **>(&p), bytes) != cudaSuccess) {
      cudaGetLastError();  // an allocation failure is not sticky; clear it for the caller's later launches
      p = nullptr;
      return false;
    }
    live_ptrs.emplace_back(p, bytes);
    live += bytes;
    peak = std::max(peak, live);
    return true;
  }
  void free(void *p) {
    for (size_t i = 0; i < live_ptrs.size(); i++)
      if (live_ptrs[i].first == p) {
        cudaFree(p);
        live -= live_ptrs[i].second;
        live_ptrs.erase(live_ptrs.begin() + i);
        return;
      }
  }
  ~BuildScratch() {
    for (auto &q : live_ptrs) cudaFree(q.first);
  }
};

// One level of the build: its nodes and, per node, child indices (into the next level), leaf reference count and
// offset (into this level's leaf buffer), subtree node / reference counts, and the three numberings.
struct BuildLevel {
  uint32_t n = 0;
  BNode *nodes = nullptr;
  uint32_t *child = nullptr, *leaf_cnt = nullptr, *leaf_off = nullptr, *size = nullptr, *rsize = nullptr;
  uint32_t *pre = nullptr, *vis = nullptr, *ref = nullptr, *leafbuf = nullptr;
};

struct BuildAdd2 {
  __host__ __device__ uint2 operator()(const uint2 &a, const uint2 &b) const { return make_uint2(a.x + b.x, a.y + b.y); }
};
struct BuildAdd4 {
  __host__ __device__ uint4 operator()(const uint4 &a, const uint4 &b) const {
    return make_uint4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w);
  }
};

static unsigned build_blocks(uint64_t n) { return (unsigned)std::max<uint64_t>(1, (n + 255) / 256); }

static int build_nomem(const Gpu &g, const BuildScratch &sc) {
  return fail(CRTB200_ERR_MEMORY, "device KD build: scratch does not fit on device " + std::to_string(g.device) + " (" +
                                      std::to_string(sc.live) + " bytes allocated)");
}

// Builds the trees of M meshes (their first_triangle, n_triangles and material are read) over the n_tris triangle
// records `geom` (3 per triangle, in sc on g's device, written on g's stream) on GPU g of context c, places the arena
// (geom copied into it), top_refs and meshes with their culling margins, and commits them (commit_trees); keep: also
// keep the reference-numbered trees for crtb200_scene_trees.  Shared by crtb200_upload_geometry and
// crtb200_update_vertices_device.
static int build_trees(crtb200_ctx *c, Gpu &g, const crtb200_mesh *in_meshes, uint32_t M, uint32_t n_tris, float4 *geom,
                       BuildScratch &sc, bool keep) {
  const uint32_t T = M + 1;
  const size_t n_geom = 3 * (size_t)n_tris;
  std::vector<uint32_t> item_base(M + 1), mesh_tri(std::max(M, 1u), 0);
  uint64_t items = 0;
  for (uint32_t m = 0; m < M; m++) {
    item_base[m] = (uint32_t)std::min<uint64_t>(items, 0xFFFFFFFFu);
    mesh_tri[m] = in_meshes[m].first_triangle;
    items += in_meshes[m].n_triangles;
  }
  if (items + M >= 0x7FFFFFFFull) return fail(CRTB200_ERR_SCENE, "scene too large for 31-bit indices");
  item_base[M] = (uint32_t)items;
  const uint32_t NI = (uint32_t)items, NE = NI + M;
  cudaStream_t st = g.stream;

  bool ok = true;
  auto al = [&](auto *&p, size_t n) { ok = ok && sc.alloc(p, n); };
  auto nomem = [&]() { return build_nomem(g, sc); };
  uint32_t *d_item_base, *d_mesh_tri, *nested, *lelem, *lnode;
  BBox *ebox;
  unsigned long long *mslots, *slots;
  al(d_item_base, M + 1);
  al(d_mesh_tri, mesh_tri.size());
  al(ebox, NE);
  al(mslots, 6 * (size_t)T);
  al(slots, 4 * (size_t)T);
  al(nested, 1);
  al(lelem, NE);
  al(lnode, NE);
  std::vector<BuildLevel> lv(1);
  auto alloc_level = [&](BuildLevel &L, uint32_t n) {
    L.n = n;
    uint32_t *w = nullptr;
    al(L.nodes, n);
    al(w, 9 * (size_t)n);
    if (!ok) return;
    L.child = w;
    L.leaf_cnt = w + 2 * (size_t)n;
    L.leaf_off = w + 3 * (size_t)n;
    L.size = w + 4 * (size_t)n;
    L.rsize = w + 5 * (size_t)n;
    L.pre = w + 6 * (size_t)n;
    L.vis = w + 7 * (size_t)n;
    L.ref = w + 8 * (size_t)n;
  };
  alloc_level(lv[0], T);
  if (!ok) return nomem();

  Event ev0, ev1;
  CUDA_TRY(ev0.create(cudaEventDefault));
  CUDA_TRY(ev1.create(cudaEventDefault));

  CUDA_TRY(cudaMemcpyAsync(d_item_base, item_base.data(), item_base.size() * 4, cudaMemcpyHostToDevice, st));
  CUDA_TRY(cudaMemcpyAsync(d_mesh_tri, mesh_tri.data(), mesh_tri.size() * 4, cudaMemcpyHostToDevice, st));
  CUDA_TRY(cudaMemsetAsync(mslots, 0xFF, 6 * (size_t)T * sizeof(unsigned long long), st));
  CUDA_TRY(cudaMemsetAsync(slots, 0, 4 * (size_t)T * sizeof(unsigned long long), st));
  CUDA_TRY(cudaMemsetAsync(nested, 0xFF, sizeof(uint32_t), st));
  CUDA_TRY(cudaEventRecord(ev0, st));

  // boxes, roots and the level-0 listing
  if (NI) k_build_item_boxes<<<build_blocks(NI), 256, 0, st>>>(geom, d_item_base, d_mesh_tri, M, NI, ebox, mslots);
  if (M) k_build_roots<<<build_blocks(M), 256, 0, st>>>(d_item_base, M, NI, ebox, mslots, lv[0].nodes);
  k_build_scene_box<<<1, 1, 0, st>>>(M, NI, ebox, lv[0].nodes);
  if (NE) k_build_listing0<<<build_blocks(NE), 256, 0, st>>>(d_item_base, M, NI, lelem, lnode);
  CUDA_TRY(cudaGetLastError());

  // levels: classify, scan, count, scan, emit the children and scatter the listings
  void *cub_tmp = nullptr;
  size_t cub_bytes = 0;
  auto cub_room = [&](size_t need) {
    if (need <= cub_bytes) return;
    if (cub_tmp) sc.free(cub_tmp);
    cub_tmp = nullptr;
    cub_bytes = 0;
    uint8_t *p = nullptr;
    al(p, need);
    if (ok) {
      cub_tmp = p;
      cub_bytes = need;
    }
  };
  uint32_t nL = NE;
  for (uint32_t level = 0;; level++) {
    const uint32_t nF = lv[level].n;
    uint2 *S;
    uint4 *NS;
    al(S, (size_t)nL + 1);
    al(NS, (size_t)nF + 1);
    size_t b2 = 0, b4 = 0;
    CUDA_TRY(cub::DeviceScan::ExclusiveScan(nullptr, b2, S, S, BuildAdd2(), make_uint2(0u, 0u), (int)nL + 1, st));
    CUDA_TRY(cub::DeviceScan::ExclusiveScan(nullptr, b4, NS, NS, BuildAdd4(), make_uint4(0u, 0u, 0u, 0u), (int)nF + 1, st));
    cub_room(std::max(b2, b4));
    uint2 *flags;
    uint4 *nc;
    al(flags, (size_t)nL + 1);
    al(nc, (size_t)nF + 1);
    if (!ok) return nomem();
    k_build_flags<<<build_blocks((uint64_t)nL + 1), 256, 0, st>>>(lv[level].nodes, lelem, lnode, nL, level, M, ebox, flags);
    CUDA_TRY(cub::DeviceScan::ExclusiveScan(cub_tmp, b2, flags, S, BuildAdd2(), make_uint2(0u, 0u), (int)nL + 1, st));
    k_build_counts<<<build_blocks((uint64_t)nF + 1), 256, 0, st>>>(lv[level].nodes, nF, level, M, S, nc);
    CUDA_TRY(cub::DeviceScan::ExclusiveScan(cub_tmp, b4, nc, NS, BuildAdd4(), make_uint4(0u, 0u, 0u, 0u), (int)nF + 1, st));
    uint4 tot;
    CUDA_TRY(cudaMemcpyAsync(&tot, NS + nF, sizeof(uint4), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    sc.free(flags);
    sc.free(nc);
    if (tot.y >= 0x7FFFFFFFu) return fail(CRTB200_ERR_SCENE, "device KD build: a level lists more than 2^31 elements");
    al(lv[level].leafbuf, tot.z);
    uint32_t *next_elem = nullptr, *next_node = nullptr;
    if (tot.x) {
      lv.emplace_back();
      alloc_level(lv.back(), tot.x);
      al(next_elem, tot.y);
      al(next_node, tot.y);
    }
    if (!ok) return nomem();
    BuildLevel &L = lv[level];
    BNode *next = tot.x ? lv[level + 1].nodes : nullptr;
    k_build_emit<<<build_blocks(nF), 256, 0, st>>>(L.nodes, nF, level, M, S, NS, next, L.child, L.leaf_cnt, L.leaf_off);
    if (nL) k_build_scatter<<<build_blocks(nL), 256, 0, st>>>(L.nodes, lelem, lnode, nL, level, M, S, NS, next_elem, next_node, L.leafbuf);
    CUDA_TRY(cudaGetLastError());
    sc.free(S);
    sc.free(NS);
    sc.free(lelem);
    sc.free(lnode);
    lelem = next_elem;
    lnode = next_node;
    nL = tot.y;
    if (!tot.x) break;
  }
  const uint32_t D = (uint32_t)lv.size();

  // numbering: subtree sizes bottom-up, then the per-tree bases on the host from the roots' sizes, then top-down
  for (uint32_t l = D; l-- > 0;) {
    const BuildLevel &L = lv[l];
    const BuildLevel *N = l + 1 < D ? &lv[l + 1] : nullptr;
    k_build_up<<<build_blocks(L.n), 256, 0, st>>>(L.nodes, L.n, M, L.child, L.leaf_cnt, L.size, L.rsize, N ? N->nodes : nullptr,
                                                  N ? N->size : nullptr, N ? N->rsize : nullptr, nested);
  }
  CUDA_TRY(cudaGetLastError());
  std::vector<uint32_t> root_size(T), root_rsize(T);
  CUDA_TRY(cudaMemcpyAsync(root_size.data(), lv[0].size, T * 4, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaMemcpyAsync(root_rsize.data(), lv[0].rsize, T * 4, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaStreamSynchronize(st));
  std::vector<uint32_t> node_base(T), ref_base(T);
  uint64_t n_nodes = 0, n_refs = 0;
  for (uint32_t t = 0; t < T; t++) {
    node_base[t] = (uint32_t)std::min<uint64_t>(n_nodes, 0xFFFFFFFFu);
    n_nodes += root_size[t];
    ref_base[t] = t < M ? (uint32_t)std::min<uint64_t>(n_refs, 0xFFFFFFFFu) : 0u;
    if (t < M) n_refs += root_rsize[t];
  }
  if (n_nodes >= 0x7FFFFFF0u || n_refs >= 0x7FFFFFF0u) return fail(CRTB200_ERR_SCENE, "scene too large for 31-bit indices");
  const uint32_t n_top_refs = root_rsize[M], top_begin = node_base[M];
  uint32_t *d_node_base, *d_ref_base;
  al(d_node_base, T);
  al(d_ref_base, T);
  if (!ok) return nomem();
  CUDA_TRY(cudaMemcpyAsync(d_node_base, node_base.data(), T * 4, cudaMemcpyHostToDevice, st));
  CUDA_TRY(cudaMemcpyAsync(d_ref_base, ref_base.data(), T * 4, cudaMemcpyHostToDevice, st));
  CUDA_TRY(cudaMemsetAsync(lv[0].pre, 0, 3 * (size_t)T * sizeof(uint32_t), st));  // pre, vis, ref of the roots
  for (uint32_t l = 0; l + 1 < D; l++) {
    const BuildLevel &L = lv[l], &N = lv[l + 1];
    k_build_down<<<build_blocks(L.n), 256, 0, st>>>(L.n, L.child, L.pre, L.vis, L.ref, N.size, N.rsize, N.pre, N.vis, N.ref);
  }
  CUDA_TRY(cudaGetLastError());

  // the scene's device arrays: arena, top-level references, meshes (the margins follow), kept trees
  CUDA_TRY(cudaStreamSynchronize(st));
  const int rc = place_arena(g, n_nodes, n_refs, n_geom);
  if (rc) return rc;
  if (n_geom) CUDA_TRY(cudaMemcpyAsync(g.tri_geom_p, geom, n_geom * sizeof(float4), cudaMemcpyDeviceToDevice, st));
  CUDA_TRY(g.top_refs.ensure(std::max<uint32_t>(n_top_refs, 1)));
  std::vector<DMesh> meshes(M);
  for (uint32_t m = 0; m < M; m++) {
    meshes[m].node_begin = node_base[m];
    meshes[m].node_end = node_base[m] + root_size[m];
    meshes[m].material = in_meshes[m].material;
    meshes[m].first_triangle = in_meshes[m].first_triangle;
    meshes[m].cull_margin = std::numeric_limits<float>::infinity();
  }
  CUDA_TRY(g.meshes.upload(meshes));
  if (keep) {
    if (c->kd_nodes.ensure(std::max<uint64_t>(n_nodes, 1)) != cudaSuccess || c->kd_refs.ensure(std::max<uint64_t>(n_refs, 1)) != cudaSuccess) {
      cudaGetLastError();
      return fail(CRTB200_ERR_MEMORY, "device KD build: the built trees do not fit on device " + std::to_string(g.device));
    }
  }
  for (uint32_t l = 0; l < D; l++) {
    const BuildLevel &L = lv[l];
    const BuildLevel *N = l + 1 < D ? &lv[l + 1] : nullptr;
    k_build_write<<<build_blocks(L.n), 256, 0, st>>>(L.nodes, L.n, M, NI, L.child, L.leaf_cnt, L.leaf_off, L.leafbuf, L.size, L.pre, L.vis,
                                                     L.ref, N ? N->pre : nullptr, N ? N->vis : nullptr, d_node_base, d_ref_base,
                                                     d_item_base, d_mesh_tri, geom, g.nodes_p, g.leaf_refs_p, g.top_refs.p,
                                                     keep ? c->kd_nodes.p : nullptr, keep ? c->kd_refs.p : nullptr, slots);
  }
  if (NI) k_build_tri_margin<<<build_blocks(NI), 256, 0, st>>>(geom, d_item_base, d_mesh_tri, M, NI, slots);
  if (M) k_build_margins<<<build_blocks(M), 256, 0, st>>>(M, slots, nested, g.meshes.p);
  CUDA_TRY(cudaGetLastError());
  CUDA_TRY(cudaEventRecord(ev1, st));
  uint32_t nested_h = 0;
  CUDA_TRY(cudaMemcpyAsync(&nested_h, nested, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaStreamSynchronize(st));
  float build_ms = 0.f;
  cudaEventElapsedTime(&build_ms, ev0, ev1);

  if (keep) {
    c->kd_meshes.assign(in_meshes, in_meshes + M);
    for (uint32_t m = 0; m < M; m++) {
      c->kd_meshes[m].first_node = node_base[m];
      c->kd_meshes[m].n_nodes = root_size[m];
      c->kd_meshes[m].first_leaf_ref = ref_base[m];
      c->kd_meshes[m].n_leaf_refs = root_rsize[m];
    }
    crtb200_trees &k = c->kd_counts;
    k = crtb200_trees{};
    k.n_meshes = M;
    k.n_mesh_nodes = top_begin;
    k.n_mesh_leaf_refs = (uint32_t)n_refs;
    k.n_top_nodes = root_size[M];
    k.n_top_leaf_refs = n_top_refs;
    k.peak_scratch_bytes = sc.peak;
    k.build_ms = build_ms;
  }
  // every tree is at most 26 levels deep: k_coop's limit of 40 always holds
  commit_trees(g, M, (uint32_t)n_nodes, (uint32_t)n_refs, n_top_refs, top_begin, (uint32_t)n_nodes, nested_h != 0);
  return CRTB200_OK;
}

// Builds the trees of `s` on GPU g of context c and uploads the scene; keep: also keep the reference-numbered trees for
// crtb200_scene_trees.
static int upload_geometry_one(crtb200_ctx *c, Gpu &g, const crtb200_scene *s, bool keep) {
  SceneRecords r;
  int rc = pack_records(g, s, false, r);
  if (rc) return rc;
  BuildScratch sc;
  float4 *geom;
  if (!sc.alloc(geom, r.geom.size())) return build_nomem(g, sc);
  if (!r.geom.empty()) CUDA_TRY(cudaMemcpyAsync(geom, r.geom.data(), r.geom.size() * sizeof(float4), cudaMemcpyHostToDevice, g.stream));
  rc = build_trees(c, g, s->meshes, s->n_meshes, s->n_triangles, geom, sc, keep);
  if (rc) return rc;
  rc = commit_records(c, g, s, r);
  if (rc == CRTB200_OK && keep) c->trees_built = true;
  return rc;
}

// GPU g's part of crtb200_update_vertices_device, once the caller's stream reached `fork`: the positions (GPUs after
// the first copy them from the first GPU), the triangle records and face normals, the incidence list (corners sorted
// stably by vertex id) and the vertex normals, then the build.  The old scene is gone from the first write on.
static int update_one(crtb200_ctx *c, Gpu &g, const float *d_positions, uint32_t n_vertices, cudaEvent_t fork, bool keep) {
  CUDA_TRY(cudaSetDevice(g.device));
  g.have_scene = false;
  cudaStream_t st = g.stream;
  CUDA_TRY(cudaStreamWaitEvent(st, fork, 0));
  const uint32_t T = g.n_triangles, V = n_vertices;
  const uint64_t NC = 3 * (uint64_t)T;
  BuildScratch sc;
  const float *pos = d_positions;
  float *pos_copy = nullptr;
  if (&g != c->gpus[0].get() && V) {
    if (!sc.alloc(pos_copy, 3 * (size_t)V)) return build_nomem(g, sc);
    CUDA_TRY(cudaMemcpyPeerAsync(pos_copy, g.device, d_positions, c->gpus[0]->device, 3 * (size_t)V * sizeof(float), st));
    pos = pos_copy;
  }
  float4 *geom, *face_n;
  uint32_t *corner_vtx, *corner_tri, *sorted_vtx, *sorted_tri;
  if (!sc.alloc(geom, NC) || !sc.alloc(face_n, T) || !sc.alloc(corner_vtx, NC) || !sc.alloc(corner_tri, NC) ||
      !sc.alloc(sorted_vtx, NC) || !sc.alloc(sorted_tri, NC))
    return build_nomem(g, sc);
  int end_bit = 1;  // the sort's key bits: enough for the largest vertex id
  while (end_bit < 32 && ((V - 1u) >> end_bit)) end_bit++;
  size_t cub_bytes = 0;
  CUDA_TRY(cub::DeviceRadixSort::SortPairs(nullptr, cub_bytes, corner_vtx, sorted_vtx, corner_tri, sorted_tri, NC, 0, end_bit, st));
  uint8_t *cub_tmp;
  if (!sc.alloc(cub_tmp, cub_bytes)) return build_nomem(g, sc);
  if (T) {
    k_update_tri_records<<<build_blocks(T), 256, 0, st>>>(pos, g.tri_shade.p, T, geom, face_n, corner_vtx, corner_tri);
    CUDA_TRY(cub::DeviceRadixSort::SortPairs(cub_tmp, cub_bytes, corner_vtx, sorted_vtx, corner_tri, sorted_tri, NC, 0, end_bit, st));
  }
  if (V) k_update_vertex_normals<<<build_blocks(V), 256, 0, st>>>(sorted_vtx, sorted_tri, NC, V, face_n, g.vtx_normal.p);
  CUDA_TRY(cudaGetLastError());
  for (void *p : {(void *)cub_tmp, (void *)sorted_tri, (void *)sorted_vtx, (void *)corner_tri, (void *)corner_vtx, (void *)face_n, (void *)pos_copy})
    if (p) sc.free(p);
  const int rc = build_trees(c, g, c->scene_meshes.data(), (uint32_t)c->scene_meshes.size(), T, geom, sc, keep);
  if (rc) return rc;
  g.have_scene = true;
  if (keep) c->trees_built = true;
  return CRTB200_OK;
}

static int check_device_ptr(const Gpu &g, const void *p, size_t align, const char *what);

extern "C" {

int crtb200_update_vertices_device(crtb200_ctx *c, const float *d_positions, uint32_t n_vertices, void *stream) {
  if (!c) return fail(CRTB200_ERR_ARG, "null argument");
  ErrScope scope(c);
  for (auto &g : c->gpus)
    if (!g->have_scene) return fail(CRTB200_ERR_STATE, "no scene uploaded");
  if (n_vertices != c->n_vertices)
    return fail(CRTB200_ERR_ARG, "n_vertices is " + std::to_string(n_vertices) + ", the uploaded scene has " + std::to_string(c->n_vertices));
  Gpu &g0 = *c->gpus[0];
  CUDA_TRY(cudaSetDevice(g0.device));
  if (n_vertices) {
    const int rc = check_device_ptr(g0, d_positions, 4, "positions");
    if (rc) return rc;
  }
  if (c->acc_active) accum_release(c);
  c->trees_built = false;
  c->kd_nodes.release();
  c->kd_refs.release();
  // every GPU starts once the work enqueued on the caller's stream so far (renders, queries, the positions' writes) is done
  Event fork;
  CUDA_TRY(fork.create(cudaEventDisableTiming));
  CUDA_TRY(cudaEventRecord(fork, (cudaStream_t)stream));
  const int rc = on_all_devices(c, [&](size_t i, Gpu &g) { return update_one(c, g, d_positions, n_vertices, fork, i == 0); });
  if (rc) {
    c->trees_built = false;
    c->kd_nodes.release();
    c->kd_refs.release();
  }
  cudaSetDevice(g0.device);
  return rc;
}

}  // extern "C"

// ---- frame planning ------------------------------------------------------------------------------------------
// worst-case children of one ray-tree node: refractive hits spawn two (RayTracer.cpp:398-412), reflective ones one, and
// in GI frames diffuse hits G (crtb200_sampling.gi_samples)
static uint32_t node_branching(const Gpu &g, const crtb200_sampling &smp) {
  uint32_t b = g.has_refractive ? 2u : (g.has_reflective ? 1u : 0u);
  if (smp.use_gi) b = std::max(b, smp.gi_samples);
  return b;
}

static uint32_t branching_sum(const Gpu &g, const crtb200_sampling &smp, uint32_t max_depth, uint64_t *per_level) {
  // worst-case rays per level-0 item at each level: branching^level, saturated at 2^40 (far beyond any queue budget)
  const uint64_t branch = node_branching(g, smp), cap = 1ull << 40;
  uint64_t sum = 0, b = 1;
  for (uint32_t l = 0; l <= max_depth; l++) {
    per_level[l] = b;
    sum += b;
    b = std::min<uint64_t>(b * branch, cap);
  }
  return (uint32_t)std::min<uint64_t>(sum, 0xFFFFFFFFull);
}

// Marks the scene arena as L2-persisting for the kernels of `st` (one access-policy window per stream).  When the arena
// is larger than the persisting carve-out, hitRatio makes a matching fraction of its lines persist instead of thrashing.
static void apply_l2_window(const Gpu &g, cudaStream_t st) {
  if (!g.l2_persist || !g.l2_persist_max || !g.l2_window_max || !g.arena_used) return;
  cudaStreamAttrValue v{};
  const size_t bytes = std::min(g.l2_persist == 3 ? g.nodes_bytes : g.arena_used, g.l2_window_max);
  v.accessPolicyWindow.base_ptr = g.arena.p;
  v.accessPolicyWindow.num_bytes = bytes;
  v.accessPolicyWindow.hitRatio = (float)std::min(1.0, (double)g.l2_persist_max / (double)bytes);
  v.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
  v.accessPolicyWindow.missProp = g.l2_persist == 1 ? cudaAccessPropertyStreaming : cudaAccessPropertyNormal;
  cudaStreamSetAttribute(st, cudaStreamAttributeAccessPolicyWindow, &v);
  cudaGetLastError();  // a hint: never an error of the render
}

// Queues of GPU g for a frame with sampling smp, under the context's queue budget and concurrency
static int plan_queues(const crtb200_ctx *c, Gpu &g, const crtb200_sampling &smp, uint32_t shard_items, uint32_t max_depth,
                       uint32_t row_items, bool pipelined) {
  uint64_t per_level[CRT_MAX_LEVELS] = {0};
  branching_sum(g, smp, max_depth, per_level);
  uint64_t sum = 0;
  for (uint32_t l = 0; l <= max_depth; l++) sum += per_level[l];
  const uint32_t n_lights = std::max<uint32_t>(1, g.sc.n_lights);
  const uint64_t bytes_per_node = 32 + 8 + 16 + 16 + 48 + n_lights;  // ray + hit + colour + comb + diffuse item + visibility bytes
  // sets used: up to `concurrency`, but never chunks smaller than 64 Ki items (launch overhead would dominate)
  uint32_t n_sets = std::max<uint32_t>(1, std::min<uint32_t>(c->concurrency, (shard_items + 65535u) / 65536u));
  // host-bound frames: chunks of at least ~512 Ki items (smaller ones only add launches and tails)
  if (pipelined) n_sets = std::max<uint32_t>(1, std::min<uint32_t>(n_sets, (shard_items + (1u << 19) - 1u) >> 19));
  // measured (profiles/r1_tuning.md): overlapping chunks only pays when band copies to the host ride along; the
  // persistent kernels already fill the GPU, extra chunks just add launches and tails
  if (!pipelined) {
    n_sets = 1;
    if (const char *env = getenv("CRT_DEVICE_CHUNKS")) n_sets = std::max(1, std::min<int>(atoi(env), (int)std::min<uint32_t>(16u, (shard_items + 65535u) / 65536u)));
  }
  uint64_t items = c->queue_budget / (bytes_per_node * sum * n_sets);
  items &= ~31ull;
  if (items < 32 * 64)
    return fail(CRTB200_ERR_MEMORY, smp.use_gi ? "queue budget too small for one chunk of 2048 pixels: the GI ray tree has up to "
                                                             "gi_samples^max_depth nodes per pixel; lower gi_samples or max_depth"
                                                       : "queue budget too small for one chunk at this ray depth");
  // host-bound frames: one chunk per stream at 1080p, two at 4K (a band's copy overlaps the traversal of the next band;
  // every chunk pays its own kernel tails and, in reflective scenes, the latency of every level again)
  uint32_t per_set = (pipelined && n_sets > 1 && shard_items >= (1u << 22)) ? 2u : 1u;
  if (const char *env = getenv("CRT_HOST_CHUNKS_PER_SET")) per_set = (uint32_t)std::max(1, std::min(8, atoi(env)));  // tools: e2e tuning
  const uint32_t parts = n_sets * per_set;
  uint64_t even = ((uint64_t)shard_items + parts - 1) / parts;
  even = ((even + row_items - 1) / row_items) * row_items;
  items = std::min<uint64_t>(items, even);
  // node ids and (diffuse item, light) slots are 32-bit on the device
  if (items * sum * n_lights >= 0x7FFFFFFFull) items = ((0x7FFFFFFFull / (sum * n_lights)) - 32) & ~31ull;
  if (items < 32) return fail(CRTB200_ERR_MEMORY, "too many lights x ray-tree nodes for 32-bit queue slots");
  if (items >= row_items) items = (items / row_items) * row_items;  // whole tile rows (band copies need it)
  g.n_chunks = (uint32_t)((shard_items + items - 1) / items);
  if (g.cap_items == items && g.cap_depth == max_depth && g.cap_sets == n_sets && g.cap_branch == node_branching(g, smp)) return CRTB200_OK;
  if (g.sets.size() < n_sets) g.sets.resize(n_sets);
  CUDA_TRY(g.fork_ev.create(cudaEventDisableTiming));
  for (uint32_t k = 0; k < n_sets; k++) {
    QueueSet &q = g.sets[k];
    CUDA_TRY(q.stream.create(cudaStreamNonBlocking));
    apply_l2_window(g, q.stream);
    CUDA_TRY(q.done.create(cudaEventDisableTiming));
    uint64_t total = 0;
    for (uint32_t l = 0; l <= max_depth; l++) {
      q.lv.offset[l] = (uint32_t)total;
      total += per_level[l] * items;
    }
    for (uint32_t l = max_depth + 1; l <= CRT_MAX_LEVELS; l++) q.lv.offset[l] = (uint32_t)total;
    const uint64_t secondary = total - items;
    CUDA_TRY(q.ray_o.ensure(std::max<uint64_t>(secondary, 1)));
    CUDA_TRY(q.ray_d.ensure(std::max<uint64_t>(secondary, 1)));
    CUDA_TRY(q.hit_tri.ensure(total));
    CUDA_TRY(q.hit_t.ensure(total));
    CUDA_TRY(q.color.ensure(total));
    CUDA_TRY(q.comb.ensure(total));
    CUDA_TRY(q.dq.ensure(3 * total));
    CUDA_TRY(q.vis.ensure(std::max<uint64_t>(1, total * std::max<uint32_t>(1, g.sc.n_lights))));
    // hand-off records: every lane of a traversal grid hands off at most once per launch
    const uint64_t ovf_cap = (uint64_t)std::max(g.blocks_closest, g.blocks_shadow) * CRT_TRAV_BLOCK;
    CUDA_TRY(q.ovf.ensure(3 * ovf_cap));
    // every record starts out "not published" (r0.x = CRT_INVALID); k_coop leaves a taken record in that state again
    CUDA_TRY(cudaMemsetAsync(q.ovf.p, 0xFF, 3 * ovf_cap * sizeof(uint4), q.stream));
    int lo = 0, hi = 0;
    CUDA_TRY(cudaDeviceGetStreamPriorityRange(&lo, &hi));  // lo = least priority: the traversal kernel's blocks go first
    CUDA_TRY(q.coop_stream.create(cudaStreamNonBlocking, lo));
    CUDA_TRY(q.coop_fork.create(cudaEventDisableTiming));
    CUDA_TRY(q.coop_join.create(cudaEventDisableTiming));
    // counts | work cursors | hand-off counters; every cursor / counter group on a 128-byte line of its own
    const size_t n_counts = 64, n_work = CRT_CTL_STRIDE * (CRT_MAX_LEVELS + 2), n_ovf = CRT_CTL_STRIDE * (CRT_MAX_LEVELS + 1);
    CUDA_TRY(q.ctl.ensure(n_counts + n_work + n_ovf));
    q.work = q.ctl.p + n_counts;
    q.lv.ovf = q.ovf.p;
    q.lv.ovf_ctl = q.ctl.p + n_counts + n_work;
    q.lv.ovf_cap = (uint32_t)std::min<uint64_t>(ovf_cap, (uint64_t)g.tail_cap * g.blocks_coop * CRT_COOP_WARPS);
    q.lv.tail_iters = 0;
    q.lv.tail_start = 512;
    q.lv.tail_start_closest = 256;
    q.lv.tail_small = 0;
    q.lv.skip_zero_terms = 0;
    q.lv.ray_o = q.ray_o.p;
    q.lv.ray_d = q.ray_d.p;
    q.lv.hit_tri = q.hit_tri.p;
    q.lv.hit_t = q.hit_t.p;
    q.lv.color = q.color.p;
    q.lv.comb = q.comb.p;
    q.lv.dq = q.dq.p;
    q.lv.vis = q.vis.p;
    q.lv.counts = q.ctl.p;
    q.lv.stats = g.stats_dev.p;
  }
  g.cap_items = (uint32_t)items;
  g.cap_depth = max_depth;
  g.cap_sets = n_sets;
  g.cap_branch = node_branching(g, smp);
  return CRTB200_OK;
}

// Pixel coverage of the rectangle list; the mask is only needed when the rectangles do not tile the image exactly
// (SURVEY App. B-1: the reference then leaves pixels unrendered).
// per-pixel coverage of a rect list (m: W*H bytes, 1 = covered) and the number of covered pixels
static size_t rect_coverage(uint32_t W, uint32_t H, const std::vector<crtb200_rect> &rects, std::vector<uint8_t> &m) {
  m.assign((size_t)W * H, 0);
  for (const auto &r : rects) {
    const uint32_t r1 = std::min<uint64_t>(H, (uint64_t)r.row + r.height), c1 = std::min<uint64_t>(W, (uint64_t)r.col + r.width);
    for (uint32_t y = r.row; y < r1; y++) std::memset(&m[(size_t)y * W + r.col], 1, r.col < c1 ? c1 - r.col : 0);
  }
  size_t covered = 0;
  for (uint8_t v : m) covered += v;
  return covered;
}

static int plan_mask(Gpu &g, const crtb200_options *o) {
  const uint32_t W = g.sc.width, H = g.sc.height;
  std::vector<crtb200_rect> rects(o->rects, o->rects + o->n_rects);
  if (g.mask_valid && rects.size() == g.mask_rects.size() &&
      (rects.empty() || !std::memcmp(rects.data(), g.mask_rects.data(), rects.size() * sizeof(crtb200_rect))))
    return CRTB200_OK;
  g.mask_rects = rects;
  g.mask_needed = false;
  if (!rects.empty()) {
    std::vector<uint8_t> m;
    if (rect_coverage(W, H, rects, m) != m.size()) {
      g.mask_needed = true;
      CUDA_TRY(g.mask.ensure(m.size()));
      CUDA_TRY(cudaMemcpy(g.mask.p, m.data(), m.size(), cudaMemcpyHostToDevice));
    }
  }
  g.mask_valid = true;
  return CRTB200_OK;
}

// records the frame's next per-launch timing event on st, creating it on first use
static cudaError_t record_next_event(crtb200_ctx *c, cudaStream_t st) {
  if (c->kev_used == c->kev.size()) c->kev.emplace_back();
  Event &e = c->kev[c->kev_used++];
  const cudaError_t err = e.create(cudaEventDefault);
  return err != cudaSuccess ? err : cudaEventRecord(e, st);
}

// dynamic shared memory of the kernels that walk one ray per lane: the visited-mesh bitset of scenes with > 64 meshes
static size_t dyn_smem(const Gpu &g, int block) { return (size_t)g.sc.dedup_words * (size_t)block * sizeof(uint32_t); }

// A caller's device pointer: device memory of the context's first GPU g, `align`-byte aligned
static int check_device_ptr(const Gpu &g, const void *p, size_t align, const char *what) {
  if (!p) return fail(CRTB200_ERR_ARG, std::string(what) + " is null");
  if (reinterpret_cast<uintptr_t>(p) % align) return fail(CRTB200_ERR_ARG, std::string(what) + " is not " + std::to_string(align) + "-byte aligned");
  cudaPointerAttributes a{};
  const cudaError_t e = cudaPointerGetAttributes(&a, p);
  if (e != cudaSuccess) cudaGetLastError();  // (not a CUDA pointer: not sticky)
  if (e != cudaSuccess || a.type != cudaMemoryTypeDevice || a.device != g.device)
    return fail(CRTB200_ERR_ARG, std::string(what) + " is not device memory of the context's first GPU");
  return CRTB200_OK;
}

// The kernel flavours of one frame.  traversal 0 (default): conservative culling + tail hand-off, both exact and both
// resting on the nesting property of the uploaded trees; traversal 1 and the visit-all counting mode walk the
// reference's literal itinerary.  The WIDE flavour (visited-mesh set in shared memory) only for scenes that need it, and
// never when counting the reference's visit-all work (no de-duplication there).
struct Flavour {
  uint32_t count_work;
  bool cull, handoff, gi, wide_closest, wide_shadow;
};

static Flavour frame_flavour(const Gpu &g, const crtb200_options *o, const crtb200_sampling &smp) {
  const bool wide = g.sc.dedup_meshes == 2u;
  return Flavour{o->count_work,
                 o->traversal == 0 && o->count_work != 1 && g.nested_ok,
                 o->traversal == 0 && o->count_work == 0 && g.nested_ok && g.tail_iters >= 0,
                 smp.use_gi != 0,
                 o->count_work == 0 && wide,
                 o->count_work != 1 && wide};
}

// The kernel flavours of a caller's ray batch (crtb200_trace_rays_device): a frame's with the batch's traversal and
// count_work -- literal walk without hand-off for traversal 1, count_work 1 and trees that do not nest -- never GI.
static Flavour query_flavour(const Gpu &g, const crtb200_ray_batch *b) {
  crtb200_options o{};
  o.traversal = b->traversal;
  o.count_work = b->count_work;
  return frame_flavour(g, &o, crtb200_sampling{});
}

// f(v) with v as a compile-time constant: how the launch functions below turn a Flavour into template arguments
template <typename F>
static void as_const(bool v, F &&f) { v ? f(std::true_type{}) : f(std::false_type{}); }
template <typename F>
static void as_const_count(uint32_t v, F &&f) {
  v == 1 ? f(std::integral_constant<int, 1>{}) : v == 2 ? f(std::integral_constant<int, 2>{}) : f(std::integral_constant<int, 0>{});
}

// The launches of one traversal over the rays of `src` at `level` (k_closest or k_shadow, and k_coop) on st; primary:
// the primary ray's back-face rule.  Sources run with the flags they can have: camera rays are primary and jittered in
// GI frames, a frame's queue is neither, a caller's rays are never jittered; queries skip refractive meshes and hand off
// only culled walks (hand-off implies culling).
template <class Src>
static void launch_closest(const Gpu &g, const Flavour &fl, const Frame &fr, QueueSet &q, uint32_t level, const Src &src,
                           bool primary, int blocks, cudaStream_t st) {
  constexpr bool camera = std::is_same<Src, CameraRays>::value, queue = std::is_same<Src, QueueRays>::value;
  as_const(fl.count_work != 0, [&](auto count) { as_const(fl.cull, [&](auto cull) { as_const(fl.wide_closest, [&](auto wide) {
    as_const(primary, [&](auto prim) { as_const(camera && fl.gi, [&](auto jitter) {
      if constexpr (!(count && wide) && (camera ? prim : !jitter && !(queue && prim)))
        k_closest<Src, prim, count, CRT_REFILL_CLOSEST, CRT_LOOP_MODE, cull, wide, jitter>
            <<<blocks, CRT_TRAV_BLOCK, dyn_smem(g, CRT_TRAV_BLOCK), st>>>(g.sc, fr, q.lv, level, q.work + CRT_CTL_STRIDE * level, src);
    }); }); }); }); });
}
// SKIPR = false in GI frames
template <class Src>
static void launch_shadow(const Gpu &g, const Flavour &fl, const Frame &fr, QueueSet &q, const Src &src, int blocks, cudaStream_t st) {
  constexpr bool query = std::is_same<Src, QueryShadow>::value;
  as_const_count(fl.count_work, [&](auto count) { as_const(fl.cull, [&](auto cull) { as_const(fl.wide_shadow, [&](auto wide) {
    as_const(!fl.gi, [&](auto skipr) {
      if constexpr ((count != 1 || !(cull || wide)) && (skipr || !query))
        k_shadow<Src, count, CRT_REFILL_SHADOW, CRT_LOOP_MODE, cull, wide, skipr>
            <<<blocks, CRT_TRAV_BLOCK, wide ? dyn_smem(g, CRT_TRAV_BLOCK) : 0, st>>>(
                g.sc, fr, q.lv, q.work + CRT_CTL_STRIDE * CRT_MAX_LEVELS, src);
    }); }); }); });
}
template <class Src>
static void launch_coop(const Gpu &g, const Flavour &fl, const Frame &fr, QueueSet &q, uint32_t level, const Src &src,
                        bool primary, int blocks, cudaStream_t st, uint32_t early) {
  constexpr bool shadow = Src::SHADOW, camera = std::is_same<Src, CameraRays>::value, queue = std::is_same<Src, QueueRays>::value;
  constexpr bool query = std::is_same<Src, QueryClosest>::value || std::is_same<Src, QueryShadow>::value;
  as_const(primary, [&](auto prim) { as_const(fl.cull, [&](auto cull) { as_const(!(shadow && fl.gi), [&](auto skipr) {
    if constexpr (!(shadow && prim) && ((shadow && !query) || skipr) && (cull || !query) && (camera ? prim : !(queue && prim)))
      k_coop<Src, prim, cull, CRT_COOP_GROUP, skipr><<<blocks, 32 * CRT_COOP_WARPS, 0, st>>>(g.sc, fr, q.lv, level, early, src);
  }); }); });
}

// One traversal launch over the rays of `src` on st -- k_closest of level `level`, or k_shadow -- and with hand-off
// k_coop around it (DESIGN.md 3.8).  blocks: the traversal kernel's grid.  With an early pass (`early_ok`: one queue
// set, and not a secondary level of a frame) the side stream is forked BEFORE the traversal kernel is launched; behind
// it k_mark marks the traversal kernel's end, the early pass starts on the side stream (its blocks get SM resources as
// the traversal kernel's blocks exit) and joins, and the final pass runs over what is left.
// timed: the context whose per-launch events time them (closest_ms, shadow_ms, coop_*_ms), null for none; a mark with a
// kind (0 closest, 1 shadow, 2 / 3 their k_coop part) opens a span and the next mark closes it, collect_stats reads
// them in pairs.
template <class Src>
static int traverse(Gpu &g, const Flavour &fl, bool early_ok, QueueSet &q, cudaStream_t st, const Frame &fr, uint32_t level,
                    const Src &src, bool primary, int blocks, crtb200_ctx *timed, uint32_t &launches) {
  constexpr bool shadow = Src::SHADOW;
  auto mark = [&](int kind) {
    if (timed && kind >= 0) timed->kev_kind.push_back(kind);
    return timed ? record_next_event(timed, st) : cudaSuccess;
  };
  const bool early = fl.handoff && g.coop_early > 0 && early_ok;
  CUDA_TRY(mark(shadow ? 1 : 0));
  if (early) {
    CUDA_TRY(cudaEventRecord(q.coop_fork, st));
    CUDA_TRY(cudaStreamWaitEvent(q.coop_stream, q.coop_fork, 0));
  }
  if constexpr (shadow)
    launch_shadow(g, fl, fr, q, src, blocks, st);
  else
    launch_closest(g, fl, fr, q, level, src, primary, blocks, st);
  if (fl.handoff) {
    CUDA_TRY(mark(-1));
    CUDA_TRY(mark(shadow ? 3 : 2));
    if (early) {
      k_mark<<<1, 32, 0, st>>>(q.lv.ovf_ctl + CRT_CTL_STRIDE * (shadow ? (uint32_t)CRT_MAX_LEVELS : level) + 24u);
      launch_coop(g, fl, fr, q, level, src, primary, g.sm_count * g.coop_early, q.coop_stream, 1u);
      CUDA_TRY(cudaEventRecord(q.coop_join, q.coop_stream));
      CUDA_TRY(cudaStreamWaitEvent(st, q.coop_join, 0));
      launches += 2;
    }
    launch_coop(g, fl, fr, q, level, src, primary, g.blocks_coop, st, 0u);
    launches++;
  }
  CUDA_TRY(mark(-1));
  return CRTB200_OK;
}

// traverse for k_closest of level `level` (QueueRays, or the request's level-0 source) or the shadow pass (ShadowPairs)
// of a frame's chunk
template <class Src>
static int traverse_frame(Gpu &g, const Flavour &fl, const Frame &fr, QueueSet &q, uint32_t level, const Src &src, bool primary,
                          crtb200_ctx *timed, uint32_t &launches) {
  const int blocks = Src::SHADOW ? g.blocks_shadow : level == 0 ? g.blocks_closest : g.blocks_closest_sec;
  return traverse(g, fl, g.cap_sets == 1 && (Src::SHADOW || level == 0), q, q.stream, fr, level, src, primary, blocks, timed,
                  launches);
}

// One query batch `qb` on GPU x (its range of a multi-GPU batch) on stream st: the query's counters zeroed, then
// traverse over the batch at level 0 (a zero Frame).  Closest hits use the work cursor and hand-off line of launch 0,
// shadow queries those of launch CRT_MAX_LEVELS.
static int enqueue_query(Gpu &x, const Flavour &fl, uint32_t ray_type, const QueryBatch &qb, cudaStream_t st,
                         uint32_t &launches) {
  QueueSet &q = x.query;
  q.lv.tail_iters = fl.handoff ? (uint32_t)(x.tail_iters + 1) : 0u;
  q.lv.tail_start = (uint32_t)x.tail_start;
  q.lv.tail_start_closest = (uint32_t)x.tail_start_closest;
  q.lv.tail_small = (uint32_t)x.tail_small;
  CUDA_TRY(cudaMemsetAsync(q.ctl.p, 0, q.ctl.n * sizeof(uint32_t), st));
  CUDA_TRY(cudaMemsetAsync(x.query_stats_dev.p, 0, CRT_STAT_SLOTS * sizeof(unsigned long long), st));
  launches++;
  const Frame fr{};
  if (ray_type == CRTB200_RAY_SHADOW)
    return traverse(x, fl, true, q, st, fr, 0, QueryShadow{qb}, false, x.blocks_query_shadow, nullptr, launches);
  return traverse(x, fl, true, q, st, fr, 0, QueryClosest{qb}, ray_type == CRTB200_RAY_PRIMARY, x.blocks_query_closest, nullptr,
                  launches);
}

// The query scratch of GPU x, allocated on first use: work cursors | hand-off counters (ctl, the layout of a frame's
// queue set), hand-off records for every lane of a query grid up to k_coop's capacity (ovf, all "not published"),
// device counters and the early pass's side stream.
static int query_scratch(Gpu &x) {
  QueueSet &q = x.query;
  if (x.query_ready) return CRTB200_OK;
  int occ = 0;
  CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_closest<QueryClosest, true, false, CRT_REFILL_CLOSEST, CRT_LOOP_MODE, true, false>, CRT_TRAV_BLOCK, 0));
  x.blocks_query_closest = std::max(1, occ) * x.sm_count;
  CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_shadow<QueryShadow, 0, CRT_REFILL_SHADOW, CRT_LOOP_MODE, true, false>, CRT_TRAV_BLOCK, 0));
  x.blocks_query_shadow = std::max(1, occ) * x.sm_count;
  const uint64_t lanes = (uint64_t)std::max(x.blocks_query_closest, x.blocks_query_shadow) * CRT_TRAV_BLOCK;
  const uint64_t cap = std::min<uint64_t>(lanes, (uint64_t)x.tail_cap * x.blocks_coop * CRT_COOP_WARPS);
  CUDA_TRY(q.ovf.ensure(3 * cap));
  CUDA_TRY(cudaMemset(q.ovf.p, 0xFF, 3 * cap * sizeof(uint4)));
  CUDA_TRY(cudaStreamSynchronize(nullptr));  // (the query runs on the caller's stream, which may not wait for stream 0)
  const size_t n_work = CRT_CTL_STRIDE * (CRT_MAX_LEVELS + 2), n_ovf = CRT_CTL_STRIDE * (CRT_MAX_LEVELS + 1);
  CUDA_TRY(q.ctl.ensure(n_work + n_ovf));
  CUDA_TRY(x.query_stats_dev.ensure(CRT_STAT_SLOTS));
  int lo = 0, hi = 0;
  CUDA_TRY(cudaDeviceGetStreamPriorityRange(&lo, &hi));
  // (each part is created once: a call that failed half-way is completed by the next one)
  CUDA_TRY(q.coop_stream.create(cudaStreamNonBlocking, lo));
  CUDA_TRY(q.coop_fork.create(cudaEventDisableTiming));
  CUDA_TRY(q.coop_join.create(cudaEventDisableTiming));
  q.work = q.ctl.p;
  q.lv.ovf = q.ovf.p;
  q.lv.ovf_ctl = q.ctl.p + n_work;
  q.lv.ovf_cap = (uint32_t)cap;
  q.lv.stats = x.query_stats_dev.p;
  x.query_ready = true;
  return CRTB200_OK;
}

// Host destinations of crtb200_render: each chunk's band of rows is copied back on the chunk's own stream right after
// its k_store, so the device->host copy of band k overlaps the traversal of the other chunks.
struct HostOut {
  float *rgb = nullptr;
  uint8_t *rgb8 = nullptr;
  crtb200_hit *hits = nullptr;
};

// A step of a progressive session (DESIGN.md 3.10.1): global samples [s0, s0 + n) through the chunk loop of
// enqueue_frame, into the accumulator of the GPU it runs on.  ap: the stop rule of an adaptive session (DESIGN.md
// 3.10.2), whose passes compact the active pixels before each sample and run k_adapt_step; null for a plain session.
struct AccumPass {
  uint32_t s0, n;
  const AdaptParams *ap;
};

// What a frame renders and where its pixels go; callers set the fields they use.
struct FrameReq {
  FrameReq(const crtb200_camera *cam, const crtb200_options *o, const crtb200_sampling &sampling)
      : cam(cam), o(o), sampling(sampling) {}
  const crtb200_camera *cam;
  const crtb200_options *o;
  crtb200_sampling sampling;  // use_gi = 0: unsampled; frame_index is the frame's Philox key word
  float *d_rgb = nullptr;  // device destinations (any may be null)
  uint8_t *d_rgb8 = nullptr;
  HitRec *d_hits = nullptr;
  float *d_slab = nullptr;          // a tile shard's compact slab (crtb200_render_device)
  const HostOut *host = nullptr;    // crtb200_render: band copies where the frame allows them (ctx->bands_copied)
  bool batch_continuation = false;  // a frame after the first of crtb200_render_frames
  const AccumPass *acc = nullptr;   // a step of a progressive session
  // crtb200_shade_rays_device: level 0 is this GPU's range of n_rays caller rays (cam is null), one pass with sample word
  // `sample`; colours and hits go to rays->rgb / rays->hits
  const ShadeRays *rays = nullptr;
  uint32_t n_rays = 0, sample = 0;
};

// level-0 work items of tile shard `index` of `count`: 8x4-pixel tiles dealt round-robin, 32 items each
static uint32_t shard_item_count(const Gpu &g, uint32_t index, uint32_t count) {
  const uint32_t tiles = ((g.sc.width + 7) / 8) * ((g.sc.height + 3) / 4);
  return (tiles > index ? (tiles - index + count - 1) / count : 0) * 32u;
}

// a Frame over the 8x4-pixel tiles of tile shard `index` of `count`, with the mask of the last plan_mask
static Frame frame_tiles(const Gpu &g, uint32_t index, uint32_t count) {
  Frame fr{};
  fr.tiles_x = (g.sc.width + 7) / 8;
  fr.n_tiles = fr.tiles_x * ((g.sc.height + 3) / 4);
  fr.shard_index = index;
  fr.shard_count = count;
  fr.mask = g.mask_needed ? g.mask.p : nullptr;
  return fr;
}

// One sample pass of one chunk (sample fr.sample): the level loop, the shadow pass, k_accumulate, k_resolve and the
// kernel that ends a sample of a GI frame or a progressive step.  Level 0 reads the request's source l0 (CameraRays or
// ShadeRays); primary0: its rays take the primary ray's back-face rule.
template <class L0>
static int sample_pass(Gpu &g, const FrameReq &r, const Flavour &fl, Frame &fr, QueueSet &q, uint32_t levels, const L0 &l0,
                       bool primary0, crtb200_ctx *timed, uint32_t &launches) {
  const cudaStream_t qs = q.stream;
  const int grid_simple = g.sm_count * 8;
  const bool adapt_step = r.acc && r.acc->ap;
  CUDA_TRY(cudaMemsetAsync(q.ctl.p, 0, q.ctl.n * sizeof(uint32_t), qs));
  if (adapt_step) {
    // level 0 of this pass runs over the pixels still sampling; the host keeps n_items0 as the bound
    fr.list = fr.n_list = nullptr;
    CUDA_TRY(cudaMemsetAsync(q.acount.p, 0, sizeof(uint32_t), qs));
    k_adapt_compact<<<grid_simple, 256, 0, qs>>>(fr, g.acc_sumsq.p, q.alist.p, q.acount.p);
    launches++;
    fr.list = q.alist.p;
    fr.n_list = q.acount.p;
  }
  q.lv.tail_iters = fl.handoff ? (uint32_t)(g.tail_iters + 1) : 0u;
  q.lv.skip_zero_terms = (r.o->traversal == 0 && r.o->count_work != 1) ? 1u : 0u;
  q.lv.tail_start = (uint32_t)g.tail_start;
  q.lv.tail_start_closest = (uint32_t)g.tail_start_closest;
  q.lv.tail_small = (uint32_t)g.tail_small;
  // (levels above 0 read the queue, whatever the request's level 0: k_shade / k_resolve over CameraRays run them)
  for (uint32_t l = 0; l < levels; l++) {
    const int rc = l == 0 ? traverse_frame(g, fl, fr, q, 0, l0, primary0, timed, launches)
                          : traverse_frame(g, fl, fr, q, l, QueueRays{}, false, timed, launches);
    if (rc) return rc;
    as_const(fl.gi, [&](auto gi) {
      if (l == 0)
        k_shade<gi><<<grid_simple, 256, 0, qs>>>(g.sc, fr, q.lv, 0u, l0);
      else
        k_shade<gi><<<grid_simple, 256, 0, qs>>>(g.sc, fr, q.lv, l, CameraRays{});
    });
    launches += 2;
  }
  const int rc = traverse_frame(g, fl, fr, q, 0, ShadowPairs{}, false, timed, launches);
  if (rc) return rc;
  k_accumulate<<<grid_simple, 256, 0, qs>>>(g.sc, fr, q.lv);
  launches += 2;
  // (GI frames resolve the last level too: its diffuse hits combine D with G background children)
  for (uint32_t l = fl.gi ? levels : levels - 1; l-- > 0;) {
    as_const(fl.gi, [&](auto gi) {
      if (l == 0)
        k_resolve<gi><<<grid_simple, 256, 0, qs>>>(g.sc, fr, q.lv, 0u, l0);
      else
        k_resolve<gi><<<grid_simple, 256, 0, qs>>>(g.sc, fr, q.lv, l, CameraRays{});
    });
    launches++;
  }
  // (a batch of caller rays is one pass with an arbitrary sample word: nothing to average)
  const bool sample_acc = fl.gi && std::is_same<L0, CameraRays>::value;
  if (adapt_step)
    k_adapt_step<<<grid_simple, 256, 0, qs>>>(g.sc, fr, q.lv, *r.acc->ap, g.acc_sum.p, g.acc_sumsq.p, g.acc_hit.p);
  else if (r.acc)
    k_accum_step<<<grid_simple, 256, 0, qs>>>(g.sc, fr, q.lv, g.acc_sum.p, g.acc_sumsq.p, g.acc_hit.p);
  else if (sample_acc)
    k_sample_acc<<<grid_simple, 256, 0, qs>>>(g.sc, fr, q.lv, q.acc.p, q.hit0.p);
  if (r.acc || sample_acc) launches++;
  return CRTB200_OK;
}

// the band of image rows that chunk `chunk` (level-0 items [begin, begin + n)) has stored, to the host destinations:
// behind the chunk's stream qs, on the band stream when there is one
static int copy_band(crtb200_ctx *c, const Gpu &g, const FrameReq &r, cudaStream_t qs, uint32_t chunk, uint32_t begin, uint32_t n,
                     uint32_t row_items, bool band_stream) {
  const uint32_t W = g.sc.width, H = g.sc.height;
  const uint32_t row0 = (begin / row_items) * 4u;
  const uint32_t row1 = std::min<uint32_t>(H, ((begin + n + row_items - 1) / row_items) * 4u);
  const size_t off = (size_t)row0 * W, cnt = (size_t)(row1 - row0) * W;
  cudaStream_t cs = qs;
  if (band_stream) {
    CUDA_TRY(cudaEventRecord(c->chunk_done[chunk], qs));
    CUDA_TRY(cudaStreamWaitEvent(c->band_stream, c->chunk_done[chunk], 0));
    cs = c->band_stream;
  }
  const HostOut &h = *r.host;
  if (h.rgb) CUDA_TRY(cudaMemcpyAsync(h.rgb + off * 3, r.d_rgb + off * 3, cnt * 3 * sizeof(float), cudaMemcpyDeviceToHost, cs));
  if (h.rgb8) CUDA_TRY(cudaMemcpyAsync(h.rgb8 + off * 3, r.d_rgb8 + off * 3, cnt * 3, cudaMemcpyDeviceToHost, cs));
  if (h.hits) CUDA_TRY(cudaMemcpyAsync(h.hits + off, r.d_hits + off, cnt * sizeof(HitRec), cudaMemcpyDeviceToHost, cs));
  if (getenv("CRT_CHUNK_TIMES")) {
    if (c->dbg_ev.size() < 2 * (size_t)(chunk + 1)) c->dbg_ev.resize(2 * (size_t)(chunk + 1));
    CUDA_TRY(c->dbg_ev[2 * chunk].create(cudaEventDefault));
    CUDA_TRY(c->dbg_ev[2 * chunk + 1].create(cudaEventDefault));
    CUDA_TRY(cudaEventRecord(c->dbg_ev[2 * chunk], qs));
    CUDA_TRY(cudaEventRecord(c->dbg_ev[2 * chunk + 1], cs));
    c->dbg_chunks = chunk + 1;
  }
  return CRTB200_OK;
}

// Enqueue GPU g's part of one frame on `st`; c->bands_copied then says whether the frame's host destinations are copied
// already.  Only the context's first GPU records the frame's span and per-launch events: nothing reads another GPU's.
static int enqueue_frame(crtb200_ctx *c, Gpu &g, const FrameReq &r, cudaStream_t st) {
  const bool first = &g == c->gpus[0].get();
  const crtb200_options *o = r.o;
  const AccumPass *acc = r.acc;
  if (!g.have_scene) return fail(CRTB200_ERR_STATE, "no scene uploaded");
  if (o->max_depth > 31) return fail(CRTB200_ERR_ARG, "max_depth > 31 is not supported");
  if (o->n_rects && !o->rects) return fail(CRTB200_ERR_ARG, "n_rects > 0 but rects is null");
  if (o->traversal > 1) return fail(CRTB200_ERR_ARG, "unknown traversal mode");
  if (o->count_work > 2) return fail(CRTB200_ERR_ARG, "unknown count_work mode");
  const Flavour fl = frame_flavour(g, o, r.sampling);
  const uint32_t shard_count = o->shard_count ? o->shard_count : 1;
  if (o->shard_index >= shard_count) return fail(CRTB200_ERR_ARG, "shard_index >= shard_count");
  int rc = r.rays ? CRTB200_OK : plan_mask(g, o);
  if (rc) return rc;
  Frame fr = frame_tiles(g, o->shard_index, shard_count);
  if (r.cam) {
    for (int k = 0; k < 3; k++) fr.cam.pos[k] = r.cam->position[k];
    for (int k = 0; k < 9; k++) fr.cam.rot[k] = r.cam->rotation[k];
  }
  fr.max_depth = o->max_depth;
  // GI frames (sampling contract, DESIGN.md 3.10): spp sample-major passes per chunk, each the whole level loop
  const bool gi = fl.gi, secondary = g.has_reflective || g.has_refractive || gi;
  fr.resolve = secondary ? 1u : 0u;
  fr.shadow_bias = o->shadow_bias;
  fr.reflection_bias = o->reflection_bias;
  fr.refraction_bias = o->refraction_bias;
  fr.gi = gi ? 1u : 0u;
  fr.gi_samples = gi ? r.sampling.gi_samples : 0u;
  fr.spp = gi && !r.rays ? r.sampling.rays_per_pixel : 1u;
  fr.seed = r.sampling.seed;
  fr.frame_index = r.sampling.frame_index;
  fr.mc_bias = r.sampling.monte_carlo_bias;
  const uint32_t shard_items = r.rays ? r.n_rays : shard_item_count(g, o->shard_index, shard_count);
  // unsharded frames: chunks are whole rows of tiles, so a chunk owns a contiguous band of image rows
  const uint32_t row_items = (shard_count == 1 && !r.rays) ? fr.tiles_x * 32u : 32u;
  rc = plan_queues(c, g, r.sampling, std::max(shard_items, 32u), o->max_depth, row_items, r.host != nullptr);
  if (rc) return rc;
  const uint32_t levels = secondary ? o->max_depth + 1 : 1;
  // sample passes s_begin, s_begin + 1, ... (caller rays: one, with any sample word)
  const uint32_t s_begin = acc ? acc->s0 : (r.rays ? r.sample : 0u), n_passes = acc ? acc->n : fr.spp;
  // Band copies need chunks that own whole rows of tiles: with a small queue budget or a deep refractive scene a chunk
  // is smaller than a tile row, two chunks on different streams would then share a 4-row band and a band copy could
  // pick up the other chunk's stale pixels.  Then the caller copies the whole frame after the join instead.
  const bool band_copies = r.host && shard_count == 1 && g.cap_items % row_items == 0;

  // frames after the first of a batch (crtb200_render_frames) keep accumulating into the same counters and time span
  if (!r.batch_continuation) CUDA_TRY(cudaMemsetAsync(g.stats_dev.p, 0, CRT_STAT_SLOTS * sizeof(unsigned long long), st));
#if CRT_PHASE_CLOCKS
  CUDA_TRY(cudaMemsetAsync(g.stats_dev.p + CRT_STAT_WARP_SPAN + 3, 0xFF, sizeof(unsigned long long), st));  // atomicMin slots
  CUDA_TRY(cudaMemsetAsync(g.stats_dev.p + CRT_STAT_WARP_SPAN + 7, 0xFF, sizeof(unsigned long long), st));
#endif
  if (first) {
    c->kev_used = 0;
    c->kev_kind.clear();
    if (!r.batch_continuation) CUDA_TRY(cudaEventRecord(c->ev[0], st));
  }
  // fork: every set's stream waits for the caller's stream, chunks go round-robin, the caller's stream joins at the end
  const uint32_t n_sets = g.cap_sets;
  crtb200_ctx *const timed = first && n_sets == 1 && !r.batch_continuation ? c : nullptr;
  CUDA_TRY(cudaEventRecord(g.fork_ev, st));
  for (uint32_t k = 0; k < n_sets; k++) CUDA_TRY(cudaStreamWaitEvent(g.sets[k].stream, g.fork_ev, 0));
  uint32_t launches = 0, chunk = 0;
  // band copies leave on their own stream, so a set starts its next chunk while its last band is still in flight
  const bool band_stream = band_copies && n_sets > 1 && !getenv("CRT_NO_BAND_STREAM");
  if (band_stream) {
    CUDA_TRY(c->band_stream.create(cudaStreamNonBlocking));
    CUDA_TRY(c->band_done.create(cudaEventDisableTiming));
    if (c->chunk_done.size() < g.n_chunks) c->chunk_done.resize(g.n_chunks);
    for (Event &e : c->chunk_done) CUDA_TRY(e.create(cudaEventDisableTiming));
  }
  for (uint32_t begin = 0; begin < shard_items; begin += g.cap_items, chunk++) {
    QueueSet &q = g.sets[chunk % n_sets];
    fr.item_begin = begin;
    fr.n_items0 = std::min(g.cap_items, shard_items - begin);
    if (gi && !acc && !r.rays) {
      CUDA_TRY(q.acc.ensure(g.cap_items));
      CUDA_TRY(q.hit0.ensure(g.cap_items));
    }
    if (acc && acc->ap) {
      CUDA_TRY(q.alist.ensure(g.cap_items));
      CUDA_TRY(q.acount.ensure(1));
    }
    for (uint32_t k = 0; k < n_passes; k++) {
      fr.sample = s_begin + k;
      rc = r.rays ? sample_pass(g, r, fl, fr, q, levels, *r.rays, r.rays->stat == CRT_STAT_RAYS_PRIMARY, timed, launches)
                  : sample_pass(g, r, fl, fr, q, levels, CameraRays{}, true, timed, launches);
      if (rc) return rc;
    }
    if (r.rays) {
      k_store_rays<<<g.sm_count * 8, 256, 0, q.stream>>>(g.sc, fr, q.lv, *r.rays);
      launches++;
    } else if (!acc) {
      k_store<<<g.sm_count * 8, 256, 0, q.stream>>>(g.sc, fr, q.lv, r.d_rgb, r.d_rgb8, r.d_hits, r.d_slab);
      launches++;
    }
    if (band_copies) {
      rc = copy_band(c, g, r, q.stream, chunk, begin, fr.n_items0, row_items, band_stream);
      if (rc) return rc;
    }
  }
  if (band_stream) {
    CUDA_TRY(cudaEventRecord(c->band_done, c->band_stream));
    CUDA_TRY(cudaStreamWaitEvent(st, c->band_done, 0));
  }
  for (uint32_t k = 0; k < n_sets; k++) {
    CUDA_TRY(cudaEventRecord(g.sets[k].done, g.sets[k].stream));
    CUDA_TRY(cudaStreamWaitEvent(st, g.sets[k].done, 0));
  }
  if (first) CUDA_TRY(cudaEventRecord(c->ev[1], st));
  CUDA_TRY(cudaGetLastError());
  g.launches = launches;
  if (first) {
    c->last.levels = levels;
    c->last_samples = acc ? acc->n : fr.spp;
    c->bands_copied = band_copies;
  }
  return CRTB200_OK;
}

// Multi-GPU frame (crtb200_create_multi): shard i of n goes to GPU i; every GPU stores into the SAME destination
// buffers (device memory of the first GPU, peer-mapped on the others), and the caller copies the assembled frame to the
// host after the join.  A tile shard of a multi-process frame runs on the first GPU alone.
static int enqueue_any(crtb200_ctx *c, const FrameReq &r, cudaStream_t st) {
  const uint32_t n = (uint32_t)c->gpus.size();
  c->frame_gpus = r.o->shard_count > 1 ? 1u : n;
  if (c->frame_gpus == 1) return enqueue_frame(c, *c->gpus[0], r, st);
  const int rc = fan_out(c, n, st, true, [&](uint32_t i, Gpu &g, cudaStream_t s) {
    crtb200_options oi = *r.o;
    oi.shard_index = i;
    oi.shard_count = n;
    FrameReq ri = r;
    ri.o = &oi;
    ri.host = nullptr;
    return enqueue_frame(c, g, ri, s);
  });
  if (rc) return rc;
  CUDA_TRY(cudaEventRecord(c->ev[1], st));  // the frame ends when the last GPU has stored its shard
  return CRTB200_OK;
}

// The counters in a GPU's CRT_STAT_* slots (stats_dev or query_stats_dev), on the current device
static int read_counts(const unsigned long long *slots, Counts &out) {
  unsigned long long st[CRT_STAT_SLOTS];
  CUDA_TRY(cudaMemcpy(st, slots, sizeof(st), cudaMemcpyDeviceToHost));
#if CRT_PHASE_CLOCKS
  for (int k = 0; k < 2; k++) {
    const unsigned long long *p = st + CRT_STAT_PHASE + 8 * k;
    const double tot = (double)(p[0] + p[1] + p[2] + p[3] + p[4]);
    fprintf(stderr, "[phase clocks] %s: refill %.1f%% slow %.1f%% node %.1f%% tri %.1f%% other %.1f%% | node iterations %llu, tri phases (MODE 2) / ranges stolen (k_*_s) %llu, rounds %llu\n",
            k ? "k_shadow " : "k_closest", 100.0 * p[0] / tot, 100.0 * p[1] / tot, 100.0 * p[2] / tot, 100.0 * p[3] / tot, 100.0 * p[4] / tot,
            p[5], p[6], p[7]);
    {
      unsigned long long hist[2][32];
      cudaMemcpyFromSymbol(hist, g_iter_hist, sizeof(hist));
      fprintf(stderr, "[phase clocks] %s rays by log2(node iterations + 1) (cumulative over frames):", k ? "k_shadow " : "k_closest");
      for (int b = 0; b < 20; b++) fprintf(stderr, " %llu", hist[k][b]);
      fprintf(stderr, "\n");
    }
    {
      unsigned long long tail[2][2];
      cudaMemcpyFromSymbol(tail, g_tail, sizeof(tail));
      const double clk = (double)(p[0] + p[1] + p[2] + p[3] + p[4]);
      fprintf(stderr, "[phase clocks] %s after the queue ran dry (cumulative): %.1f%% of warp time, %.1f of 32 lanes busy on average\n", k ? "k_shadow " : "k_closest",
              100.0 * (double)tail[k][0] / clk, tail[k][0] ? (double)tail[k][1] / (double)tail[k][0] : 0.0);
    }
    if (getenv("CRT_WARP_DUMP")) {
      static unsigned long long rec[2][8192][6];
      cudaMemcpyFromSymbol(rec, g_warp_rec, sizeof(rec));
      unsigned long long t0 = ~0ull;
      for (int w = 0; w < 8192; w++) if (rec[k][w][1] && rec[k][w][0] < t0) t0 = rec[k][w][0];
      std::vector<std::pair<unsigned long long, int>> ends;
      for (int w = 0; w < 8192; w++) if (rec[k][w][1]) ends.push_back({rec[k][w][1] - t0, w});
      std::sort(ends.begin(), ends.end());
      fprintf(stderr, "[warp dump] %s: %zu warps; end-time percentiles (us): p10 %.0f p50 %.0f p90 %.0f p99 %.0f max %.0f\n", k ? "k_shadow " : "k_closest", ends.size(),
              ends[ends.size() / 10].first * 1e-3, ends[ends.size() / 2].first * 1e-3, ends[ends.size() * 9 / 10].first * 1e-3,
              ends[ends.size() * 99 / 100].first * 1e-3, ends.back().first * 1e-3);
      for (size_t i = ends.size() >= 6 ? ends.size() - 6 : 0; i < ends.size(); i++) {
        const unsigned long long *r = rec[k][ends[i].second];
        fprintf(stderr, "[warp dump]   warp %d: start %.0f us end %.0f us rounds %llu node-iterations %llu clk-after-dry %llu stolen %llu\n", ends[i].second,
                (r[0] - t0) * 1e-3, (r[1] - t0) * 1e-3, r[2], r[3], r[4], r[5]);
      }
    }
    const unsigned long long *g = st + CRT_STAT_WARP_SPAN + 4 * k;  // sum of warp lifetimes, warps, last end, first start (globaltimer ns)
    if (g[1])
      fprintf(stderr, "[phase clocks] %s: %llu warps, mean warp lifetime %.1f us, kernel span %.1f us (first warp start -> last warp end; one launch per frame only)\n",
              k ? "k_shadow " : "k_closest", g[1], 1e-3 * (double)g[0] / (double)g[1], 1e-3 * (double)(g[2] - g[3]));
  }
#endif
  crtb200_stats &x = out.s;
  x.rays_primary = st[CRT_STAT_RAYS_PRIMARY];
  x.rays_shadow = st[CRT_STAT_RAYS_SHADOW];
  x.rays_reflection = st[CRT_STAT_RAYS_REFLECTION];
  x.rays_refraction = st[CRT_STAT_RAYS_REFRACTION];
  x.node_tests_closest = st[CRT_STAT_NODES_CLOSEST];
  x.triangle_tests_closest = st[CRT_STAT_TRIS_CLOSEST];
  x.node_tests_shadow = st[CRT_STAT_NODES_SHADOW];
  x.triangle_tests_shadow = st[CRT_STAT_TRIS_SHADOW];
  x.handoff_closest = st[CRT_STAT_HANDOFF_CLOSEST];
  x.handoff_shadow = st[CRT_STAT_HANDOFF_SHADOW];
  x.shadow_rays_zero_term = st[CRT_STAT_ZERO_TERM];
  out.side = SideCounts{st[CRT_STAT_DIFFUSE], st[CRT_STAT_PX_SAMPLES], st[CRT_STAT_STOPPED]};
#if CRT_COOP_STATS
  fprintf(stderr, "[coop stats] closest: %llu walks, %llu iterations, %llu box tests, %llu triangle tests | shadow: %llu walks, %llu iterations, %llu box tests, %llu triangle tests\n",
          st[CRT_STAT_HANDOFF_CLOSEST], st[CRT_STAT_COOP_DEBUG], st[CRT_STAT_COOP_DEBUG + 1], st[CRT_STAT_COOP_DEBUG + 2],
          st[CRT_STAT_HANDOFF_SHADOW], st[CRT_STAT_COOP_DEBUG + 3], st[CRT_STAT_COOP_DEBUG + 4], st[CRT_STAT_COOP_DEBUG + 5]);
#endif
  return CRTB200_OK;
}

// a record added into running totals: counters, launches and times summed (a GPU's counters carry no time), levels the
// deepest
static void add_counts(Counts &t, const Counts &x) {
  crtb200_stats &a = t.s;
  const crtb200_stats &b = x.s;
  a.rays_primary += b.rays_primary;
  a.rays_shadow += b.rays_shadow;
  a.rays_reflection += b.rays_reflection;
  a.rays_refraction += b.rays_refraction;
  a.node_tests_closest += b.node_tests_closest;
  a.triangle_tests_closest += b.triangle_tests_closest;
  a.node_tests_shadow += b.node_tests_shadow;
  a.triangle_tests_shadow += b.triangle_tests_shadow;
  a.handoff_closest += b.handoff_closest;
  a.handoff_shadow += b.handoff_shadow;
  a.shadow_rays_zero_term += b.shadow_rays_zero_term;
  a.kernel_launches += b.kernel_launches;
  a.device_ms += b.device_ms;
  a.closest_ms += b.closest_ms;
  a.shadow_ms += b.shadow_ms;
  a.coop_closest_ms += b.coop_closest_ms;
  a.coop_shadow_ms += b.coop_shadow_ms;
  a.levels = std::max(a.levels, b.levels);
  t.side.diffuse += x.side.diffuse;
  t.side.px_samples += x.side.px_samples;
  t.side.stopped += x.side.stopped;
}

// The last render's statistics into c->last / c->last_side: counters and launches summed over the GPUs that rendered
// it, times of the first GPU (span fork to join, per-launch events)
static int collect_stats(crtb200_ctx *c) {
  Counts t;
  for (uint32_t i = 0; i < c->frame_gpus; i++) {
    Gpu &g = *c->gpus[i];
    CUDA_TRY(cudaSetDevice(g.device));
    if (i) CUDA_TRY(cudaStreamSynchronize(g.stream));
    Counts x;
    const int rc = read_counts(g.stats_dev.p, x);
    if (rc) return rc;
    x.s.kernel_launches = g.launches;
    add_counts(t, x);
  }
  CUDA_TRY(cudaSetDevice(c->gpus[0]->device));
  t.s.levels = c->last.levels;
  float ms = 0.f;
  CUDA_TRY(cudaEventElapsedTime(&ms, c->ev[0], c->ev[1]));
  t.s.device_ms = ms;
  for (size_t k = 0; k < c->kev_kind.size() && 2 * k + 1 < c->kev_used; k++) {
    float kms = 0.f;
    CUDA_TRY(cudaEventElapsedTime(&kms, c->kev[2 * k], c->kev[2 * k + 1]));
    // closest_ms / shadow_ms include their k_coop part, which is also reported on its own
    if (c->kev_kind[k] == 0 || c->kev_kind[k] == 2) t.s.closest_ms += kms;
    if (c->kev_kind[k] == 1 || c->kev_kind[k] == 3) t.s.shadow_ms += kms;
    if (c->kev_kind[k] == 2) t.s.coop_closest_ms += kms;
    if (c->kev_kind[k] == 3) t.s.coop_shadow_ms += kms;
    if (getenv("CRT_KERNEL_TIMES"))  // tools: one line per traversal launch of the frame, in launch order
      fprintf(stderr, "[kernel times] %s %.3f ms\n", c->kev_kind[k] == 0 ? "k_closest" : c->kev_kind[k] == 1 ? "k_shadow" : "k_coop", kms);
  }
  c->last = t.s;
  c->last_side = t.side;
  return CRTB200_OK;
}

extern "C" {

}  // extern "C"

// crtb200_render of frame `frame` of a batch: the sampling's Philox key word is frame_index + frame
static int render(crtb200_ctx *c, const crtb200_camera *cam, const crtb200_options *o, uint32_t frame, float *rgb_out,
                  uint8_t *rgb8_out, crtb200_hit *hits_out, crtb200_stats *stats) {
  Gpu &g = *c->gpus[0];
  const auto t0 = std::chrono::steady_clock::now();
  CUDA_TRY(cudaSetDevice(g.device));
  if (!g.have_scene) return fail(CRTB200_ERR_STATE, "no scene uploaded");
  const size_t px = (size_t)g.sc.width * g.sc.height;
  if (hits_out) CUDA_TRY(c->hits.ensure(px));
  if (hits_out) CUDA_TRY(cudaMemsetAsync(c->hits.p, 0xFF, px * sizeof(HitRec), g.stream));
  c->last = crtb200_stats{};
  // Rectangle grids that leave pixels uncovered keep the previous frame there (colorBuffer persistence), so the whole
  // persistent frame is copied after the render; otherwise each chunk's band is copied as soon as it is stored.
  const HostOut host{rgb_out, rgb8_out, hits_out};
  int rc = plan_mask(g, o);
  if (rc) return rc;
  FrameReq r(cam, o, c->sampling);
  r.sampling.frame_index += frame;
  r.d_rgb = c->frame.p;
  r.d_rgb8 = rgb8_out ? c->frame8.p : nullptr;
  r.d_hits = hits_out ? c->hits.p : nullptr;
  if (o->shard_count <= 1 && !g.mask_needed && (rgb_out || rgb8_out || hits_out)) r.host = &host;
  rc = enqueue_any(c, r, g.stream);
  if (rc) return rc;
  if (!c->bands_copied) {
    if (rgb_out) CUDA_TRY(cudaMemcpyAsync(rgb_out, c->frame.p, px * 3 * sizeof(float), cudaMemcpyDeviceToHost, g.stream));
    if (rgb8_out) CUDA_TRY(cudaMemcpyAsync(rgb8_out, c->frame8.p, px * 3, cudaMemcpyDeviceToHost, g.stream));
    if (hits_out) CUDA_TRY(cudaMemcpyAsync(hits_out, c->hits.p, px * sizeof(HitRec), cudaMemcpyDeviceToHost, g.stream));
  }
  const double enqueue_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
  CUDA_TRY(cudaStreamSynchronize(g.stream));
  const double sync_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
  rc = collect_stats(c);
  if (rc) return rc;
  c->last.total_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
  if (c->bands_copied && c->dbg_chunks && getenv("CRT_CHUNK_TIMES")) {
    fprintf(stderr, "[chunk times] host: enqueue %.3f ms, synchronised %.3f ms, stats read %.3f ms; device frame %.3f ms\n", enqueue_ms, sync_ms,
            c->last.total_ms, c->last.device_ms);
    for (uint32_t k = 0; k < c->dbg_chunks; k++) {
      float a = 0.f, b = 0.f;
      cudaEventElapsedTime(&a, c->ev[0], c->dbg_ev[2 * k]);
      cudaEventElapsedTime(&b, c->ev[0], c->dbg_ev[2 * k + 1]);
      fprintf(stderr, "[chunk times]   chunk %u (up to %u items, set %u): stored at %.3f ms, band on the host at %.3f ms\n", k, g.cap_items, k % g.cap_sets, a, b);
    }
    c->dbg_chunks = 0;
  }
  if (stats) *stats = c->last;
  return CRTB200_OK;
}

extern "C" {

int crtb200_render(crtb200_ctx *c, const crtb200_camera *cam, const crtb200_options *o, float *rgb_out,
                   uint8_t *rgb8_out, crtb200_hit *hits_out, crtb200_stats *stats) {
  ErrScope scope(c);
  if (!c || !cam || !o) return fail(CRTB200_ERR_ARG, "null argument");
  return render(c, cam, o, 0, rgb_out, rgb8_out, hits_out, stats);
}

// The animation loop of app/animation.cpp:24-38 (setCamera + render per frame), batched and pipelined: no host
// synchronisation between frames, two frames in flight -- frame f + 1 is rendered while frame f's pixels travel to the
// host on a copy stream.  Rectangle lists that leave pixels uncovered need colorBuffer persistence from frame to frame
// (one buffer, in order), and tile shards write no full frame: those take the frame-by-frame path.  GI frames: frame f
// takes Philox key word frame_index + f.
int crtb200_render_frames(crtb200_ctx *c, const crtb200_camera *cams, uint32_t n_frames, const crtb200_options *o,
                          float *rgb_out, uint8_t *rgb8_out, crtb200_stats *stats) {
  ErrScope scope(c);
  if (!c || !cams || !o) return fail(CRTB200_ERR_ARG, "null argument");
  Gpu &g = *c->gpus[0];
  if (!g.have_scene) return fail(CRTB200_ERR_STATE, "no scene uploaded");
  CUDA_TRY(cudaSetDevice(g.device));
  const size_t px = (size_t)g.sc.width * g.sc.height;
  const auto t0 = std::chrono::steady_clock::now();
  int rc = plan_mask(g, o);
  if (rc) return rc;
  if (g.mask_needed || o->shard_count > 1 || o->count_work != 0 || n_frames < 2) {
    Counts total;
    for (uint32_t f = 0; f < n_frames; f++) {
      Counts x;
      rc = render(c, cams + f, o, f, rgb_out ? rgb_out + f * px * 3 : nullptr, rgb8_out ? rgb8_out + f * px * 3 : nullptr, nullptr, &x.s);
      if (rc) return rc;
      x.side = c->last_side;
      add_counts(total, x);
    }
    total.s.total_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    c->last_side = total.side;
    if (stats) *stats = total.s;
    return CRTB200_OK;
  }
  CUDA_TRY(c->frame_b.ensure(px * 3));
  if (rgb8_out) CUDA_TRY(c->frame8_b.ensure(px * 3));
  CUDA_TRY(c->copy_stream.create(cudaStreamNonBlocking));
  for (int k = 0; k < 2; k++) {
    CUDA_TRY(c->rendered[k].create(cudaEventDisableTiming));
    CUDA_TRY(c->copied[k].create(cudaEventDisableTiming));
  }
  c->last = crtb200_stats{};
  uint32_t launches = 0;
  for (uint32_t f = 0; f < n_frames; f++) {
    const int k = (int)(f & 1u);
    float *d_rgb = k ? c->frame_b.p : c->frame.p;
    uint8_t *d_rgb8 = rgb8_out ? (k ? c->frame8_b.p : c->frame8.p) : nullptr;
    if (f >= 2) CUDA_TRY(cudaStreamWaitEvent(g.stream, c->copied[k], 0));  // this pair's previous frame has left the device
    FrameReq r(cams + f, o, c->sampling);
    r.sampling.frame_index += f;
    r.d_rgb = d_rgb;
    r.d_rgb8 = d_rgb8;
    r.batch_continuation = f > 0;
    rc = enqueue_any(c, r, g.stream);
    if (rc) return rc;
    launches += g.launches;
    CUDA_TRY(cudaEventRecord(c->rendered[k], g.stream));
    CUDA_TRY(cudaStreamWaitEvent(c->copy_stream, c->rendered[k], 0));
    if (rgb_out) CUDA_TRY(cudaMemcpyAsync(rgb_out + f * px * 3, d_rgb, px * 3 * sizeof(float), cudaMemcpyDeviceToHost, c->copy_stream));
    if (rgb8_out) CUDA_TRY(cudaMemcpyAsync(rgb8_out + f * px * 3, d_rgb8, px * 3, cudaMemcpyDeviceToHost, c->copy_stream));
    CUDA_TRY(cudaEventRecord(c->copied[k], c->copy_stream));
  }
  CUDA_TRY(cudaStreamSynchronize(g.stream));
  CUDA_TRY(cudaStreamSynchronize(c->copy_stream));
  if ((n_frames & 1u) == 0u) {  // the last frame went into the second pair: it is the persistent colour buffer now
    std::swap(c->frame, c->frame_b);
    std::swap(c->frame8, c->frame8_b);
  }
  rc = collect_stats(c);
  if (rc) return rc;
  c->last.kernel_launches = launches;
  c->last.total_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
  if (stats) *stats = c->last;
  return CRTB200_OK;
}

int crtb200_render_device(crtb200_ctx *c, const crtb200_camera *cam, const crtb200_options *o, float *d_rgb_out,
                          uint8_t *d_rgb8_out, void *stream) {
  ErrScope scope(c);
  if (!c || !cam || !o) return fail(CRTB200_ERR_ARG, "null argument");
  CUDA_TRY(cudaSetDevice(c->gpus[0]->device));
  const uint32_t shard_count = o->shard_count ? o->shard_count : 1;
  c->last = crtb200_stats{};
  c->last_pending = true;
  FrameReq r(cam, o, c->sampling);
  if (shard_count > 1 && !o->shard_full_frame) {
    // sharded: d_rgb_out is the shard's compact slab (crtb200_shard_items x 3 floats), see crtb200_assemble_shards
    if (d_rgb8_out) return fail(CRTB200_ERR_ARG, "sharded rendering writes a float slab only");
    r.d_slab = d_rgb_out;
  } else {  // (shard_full_frame: the shard's pixels at their place in a full frame, peer-mapped, crtb200_ipc_open)
    r.d_rgb = d_rgb_out;
    r.d_rgb8 = d_rgb8_out;
  }
  return enqueue_any(c, r, (cudaStream_t)stream);  // (a tile shard goes to enqueue_frame)
}

// ---- progressive sessions (DESIGN.md 3.10.1) ---------------------------------------------------------------------
// One kernel over the whole tile shard of every GPU of the context: Frame with item_begin 0 and the session's rects;
// launch(x, fr, stream) enqueues GPU x's kernel.  Queues, device counters, the last render's statistics and the
// context's sampling stay as they are.  The pass runs on the first GPU's stream (fan_out).
static int shard_pass(crtb200_ctx *c, const std::function<void(Gpu &, const Frame &, cudaStream_t)> &launch) {
  const uint32_t n = (uint32_t)c->gpus.size();
  return fan_out(c, n, c->gpus[0]->stream, false, [&](uint32_t i, Gpu &x, cudaStream_t st) {
    const int rc = plan_mask(x, &c->acc_opt);
    if (rc) return rc;
    Frame fr = frame_tiles(x, i, n);
    fr.n_items0 = shard_item_count(x, i, n);
    launch(x, fr, st);
    CUDA_TRY(cudaGetLastError());
    return (int)CRTB200_OK;
  });
}

// device staging of a save / load: frame-layout S, Q, hit records and counts on the first GPU
struct AccumStaging {
  DevBuf<float> sum, sumsq;
  DevBuf<HitRec> hit;
  DevBuf<uint32_t> bad, counts;
  DevBuf<unsigned long long> tot;
};

// k_accum_load on every GPU from the staged arrays (all empty: an adaptive begin's flags), then the totals the session
// keeps on the host.  Inputs that do not fit the scene or `passes` end the session.
static int accum_load_pass(crtb200_ctx *c, AccumStaging &stg, uint32_t passes) {
  Gpu &g = *c->gpus[0];
  CUDA_TRY(stg.bad.ensure(2));
  CUDA_TRY(stg.tot.ensure(3));
  CUDA_TRY(cudaMemsetAsync(stg.bad.p, 0, 2 * sizeof(uint32_t), g.stream));
  CUDA_TRY(cudaMemsetAsync(stg.tot.p, 0, 3 * sizeof(unsigned long long), g.stream));
  const int rc = shard_pass(c, [&](Gpu &x, const Frame &fr, cudaStream_t st) {
    k_accum_load<<<x.sm_count * 8, 256, 0, st>>>(x.sc, fr, stg.sum.p, stg.sumsq.p, stg.hit.p, stg.counts.p, passes, x.n_triangles,
                                                  c->acc_adaptive, c->acc_ap, x.acc_sum.p, x.acc_sumsq.p, x.acc_hit.p,
                                                  stg.bad.p, stg.tot.p);
  });
  if (rc) return rc;
  uint32_t bad[2];
  unsigned long long tot[3];
  CUDA_TRY(cudaMemcpyAsync(bad, stg.bad.p, sizeof(bad), cudaMemcpyDeviceToHost, g.stream));
  CUDA_TRY(cudaMemcpyAsync(tot, stg.tot.p, sizeof(tot), cudaMemcpyDeviceToHost, g.stream));
  CUDA_TRY(cudaStreamSynchronize(g.stream));
  if (bad[0] || bad[1]) {
    accum_release(c);
    return fail(CRTB200_ERR_ARG, bad[0] ? "hit records name triangles the uploaded scene does not have; the session has ended"
                                        : "a count exceeds passes, or is 0 inside the rects while passes > 0; the session has ended");
  }
  c->acc_covered = tot[0];
  c->acc_active_px = tot[1];
  c->acc_px_samples = tot[2];
  return CRTB200_OK;
}

// plain (ad == nullptr) or adaptive session begin; the caller holds the ErrScope
static int accum_begin(crtb200_ctx *c, const crtb200_camera *cam, const crtb200_options *o, const crtb200_sampling *s,
                       const crtb200_adaptive *ad) {
  if (!c || !cam || !o || !s) return fail(CRTB200_ERR_ARG, "null argument");
  Gpu &g = *c->gpus[0];
  CUDA_TRY(cudaSetDevice(g.device));
  if (!g.have_scene) return fail(CRTB200_ERR_STATE, "no scene uploaded");
  if (!s->use_gi) return fail(CRTB200_ERR_ARG, "a progressive session needs sampling.use_gi = 1");
  if (ad && ad->min_samples < 2) return fail(CRTB200_ERR_ARG, "adaptive: min_samples must be at least 2");
  if (ad && ad->max_samples < ad->min_samples) return fail(CRTB200_ERR_ARG, "adaptive: max_samples < min_samples");
  if (ad && !(ad->abs_error >= 0.f && ad->rel_error >= 0.f))
    return fail(CRTB200_ERR_ARG, "adaptive: the error bounds must be >= 0 and not NaN");
  if (s->gi_samples > 1024) return fail(CRTB200_ERR_ARG, "gi_samples must be at most 1024");
  if (o->shard_count > 1 || o->shard_index != 0)
    return fail(CRTB200_ERR_ARG, "progressive sessions are not tile-sharded (several GPUs: crtb200_create_multi)");
  if (o->max_depth > 31 || (o->n_rects && !o->rects) || o->traversal > 1 || o->count_work > 2)
    return fail(CRTB200_ERR_ARG, "bad options (max_depth > 31, null rects, or unknown traversal / count_work mode)");
  accum_release(c);
  c->acc_cam = *cam;
  c->acc_opt = *o;
  c->acc_rects.assign(o->rects, o->rects + o->n_rects);
  c->acc_opt.rects = o->n_rects ? c->acc_rects.data() : nullptr;
  c->acc_smp = *s;
  c->acc_smp.use_gi = 1;
  c->acc_smp.rays_per_pixel = 1;  // unused: a step says how many samples it renders
  const uint32_t n = (uint32_t)c->gpus.size();
  for (uint32_t i = 0; i < n; i++) {
    Gpu &x = *c->gpus[i];
    const size_t items = std::max<size_t>(1, shard_item_count(g, i, n));
    cudaError_t e = cudaSetDevice(x.device);
    if (e == cudaSuccess) e = x.acc_sum.ensure(items);
    if (e == cudaSuccess) e = x.acc_sumsq.ensure(items);
    if (e == cudaSuccess) e = x.acc_hit.ensure(items);
    if (e == cudaSuccess) e = cudaMemsetAsync(x.acc_sum.p, 0, items * sizeof(float4), x.stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(x.acc_sumsq.p, 0, items * sizeof(float4), x.stream);
    // no hit until sample 0 has run: a save at 0 samples must not look up a triangle
    if (e == cudaSuccess) e = cudaMemsetAsync(x.acc_hit.p, 0xFF, items * sizeof(uint2), x.stream);
    if (e != cudaSuccess) {
      cudaGetLastError();
      accum_release(c);
      return fail(e == cudaErrorMemoryAllocation ? CRTB200_ERR_MEMORY : CRTB200_ERR_CUDA,
                  std::string("progressive accumulator (40 bytes per pixel) on device ") + std::to_string(x.device) + ": " +
                      cudaGetErrorString(e));
    }
  }
  CUDA_TRY(cudaSetDevice(g.device));
  c->acc_active = true;
  std::vector<uint8_t> m;
  c->acc_covered = c->acc_rects.empty() ? (uint64_t)g.sc.width * g.sc.height
                                        : rect_coverage(g.sc.width, g.sc.height, c->acc_rects, m);
  if (!ad) return CRTB200_OK;
  c->acc_adaptive = true;
  c->acc_ap = AdaptParams{ad->min_samples, ad->max_samples, ad->abs_error, ad->rel_error};
  // every covered pixel starts active: the flags are set on the device, shard by shard
  AccumStaging flags;
  const int rc = accum_load_pass(c, flags, 0);
  if (rc) accum_release(c);
  return rc;
}

int crtb200_accum_begin(crtb200_ctx *c, const crtb200_camera *cam, const crtb200_options *o, const crtb200_sampling *s) {
  ErrScope scope(c);
  return accum_begin(c, cam, o, s, nullptr);
}

int crtb200_accum_begin_adaptive(crtb200_ctx *c, const crtb200_camera *cam, const crtb200_options *o,
                                 const crtb200_sampling *s, const crtb200_adaptive *ad) {
  ErrScope scope(c);
  if (!ad) return fail(CRTB200_ERR_ARG, "null argument");
  return accum_begin(c, cam, o, s, ad);
}

int crtb200_accum_step(crtb200_ctx *c, uint32_t n_samples, crtb200_stats *stats) {
  ErrScope scope(c);
  if (!c) return fail(CRTB200_ERR_ARG, "ctx is null");
  Gpu &g = *c->gpus[0];
  CUDA_TRY(cudaSetDevice(g.device));
  if (!c->acc_active) return fail(CRTB200_ERR_STATE, "no progressive session (crtb200_accum_begin)");
  if (n_samples == 0 || (uint64_t)c->acc_done + n_samples > 0xFFFFFFFFull) return fail(CRTB200_ERR_ARG, "n_samples must be at least 1");
  const auto t0 = std::chrono::steady_clock::now();
  c->last = crtb200_stats{};
  const AccumPass a{c->acc_done, n_samples, c->acc_adaptive ? &c->acc_ap : nullptr};
  FrameReq r(&c->acc_cam, &c->acc_opt, c->acc_smp);
  r.acc = &a;
  int rc = enqueue_any(c, r, g.stream);
  if (rc) return rc;
  CUDA_TRY(cudaStreamSynchronize(g.stream));
  rc = collect_stats(c);
  if (rc) return rc;
  c->acc_done += n_samples;
  if (c->acc_adaptive) {
    c->acc_px_samples += c->last_side.px_samples;
    c->acc_active_px -= c->last_side.stopped;
  }
  c->last.total_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
  if (stats) *stats = c->last;
  return CRTB200_OK;
}

int crtb200_accum_read(crtb200_ctx *c, float *rgb_out, uint8_t *rgb8_out, crtb200_hit *hits_out, uint32_t *samples_done) {
  ErrScope scope(c);
  if (!c) return fail(CRTB200_ERR_ARG, "ctx is null");
  Gpu &g = *c->gpus[0];
  CUDA_TRY(cudaSetDevice(g.device));
  if (!c->acc_active) return fail(CRTB200_ERR_STATE, "no progressive session (crtb200_accum_begin)");
  if (c->acc_done == 0) return fail(CRTB200_ERR_STATE, "the progressive session has no samples yet");
  const size_t px = (size_t)g.sc.width * g.sc.height;
  if (hits_out) CUDA_TRY(c->hits.ensure(px));
  if (hits_out) CUDA_TRY(cudaMemsetAsync(c->hits.p, 0xFF, px * sizeof(HitRec), g.stream));
  const int rc = shard_pass(c, [&](Gpu &x, const Frame &fr, cudaStream_t st) {
    k_accum_read<<<x.sm_count * 8, 256, 0, st>>>(x.sc, fr, x.acc_sum.p, x.acc_hit.p, c->frame.p,
                                                  rgb8_out ? c->frame8.p : nullptr, hits_out ? c->hits.p : nullptr);
  });
  if (rc) return rc;
  if (rgb_out) CUDA_TRY(cudaMemcpyAsync(rgb_out, c->frame.p, px * 3 * sizeof(float), cudaMemcpyDeviceToHost, g.stream));
  if (rgb8_out) CUDA_TRY(cudaMemcpyAsync(rgb8_out, c->frame8.p, px * 3, cudaMemcpyDeviceToHost, g.stream));
  if (hits_out) CUDA_TRY(cudaMemcpyAsync(hits_out, c->hits.p, px * sizeof(HitRec), cudaMemcpyDeviceToHost, g.stream));
  CUDA_TRY(cudaStreamSynchronize(g.stream));
  if (samples_done) *samples_done = c->acc_done;
  return CRTB200_OK;
}

// k_accum_save on every GPU into the staged arrays (any may be empty)
static int accum_save_pass(crtb200_ctx *c, AccumStaging &stg) {
  return shard_pass(c, [&](Gpu &x, const Frame &fr, cudaStream_t st) {
    k_accum_save<<<x.sm_count * 8, 256, 0, st>>>(x.sc, fr, x.acc_sum.p, x.acc_sumsq.p, x.acc_hit.p, stg.sum.p, stg.sumsq.p,
                                                  stg.hit.p, stg.counts.p);
  });
}

int crtb200_accum_save(crtb200_ctx *c, float *sum_out, float *sumsq_out, crtb200_hit *hit0_out, uint32_t *samples_done) {
  ErrScope scope(c);
  if (!c) return fail(CRTB200_ERR_ARG, "ctx is null");
  Gpu &g = *c->gpus[0];
  CUDA_TRY(cudaSetDevice(g.device));
  if (!c->acc_active) return fail(CRTB200_ERR_STATE, "no progressive session (crtb200_accum_begin)");
  const size_t px = (size_t)g.sc.width * g.sc.height;
  AccumStaging stg;
  if (sum_out) {
    CUDA_TRY(stg.sum.ensure(px * 3));
    CUDA_TRY(cudaMemsetAsync(stg.sum.p, 0, px * 3 * sizeof(float), g.stream));
  }
  if (sumsq_out) {
    CUDA_TRY(stg.sumsq.ensure(px * 3));
    CUDA_TRY(cudaMemsetAsync(stg.sumsq.p, 0, px * 3 * sizeof(float), g.stream));
  }
  if (hit0_out) {
    CUDA_TRY(stg.hit.ensure(px));
    CUDA_TRY(cudaMemsetAsync(stg.hit.p, 0xFF, px * sizeof(HitRec), g.stream));
  }
  const int rc = accum_save_pass(c, stg);
  if (rc) return rc;
  if (sum_out) CUDA_TRY(cudaMemcpyAsync(sum_out, stg.sum.p, px * 3 * sizeof(float), cudaMemcpyDeviceToHost, g.stream));
  if (sumsq_out) CUDA_TRY(cudaMemcpyAsync(sumsq_out, stg.sumsq.p, px * 3 * sizeof(float), cudaMemcpyDeviceToHost, g.stream));
  if (hit0_out) CUDA_TRY(cudaMemcpyAsync(hit0_out, stg.hit.p, px * sizeof(HitRec), cudaMemcpyDeviceToHost, g.stream));
  CUDA_TRY(cudaStreamSynchronize(g.stream));
  if (samples_done) *samples_done = c->acc_done;
  return CRTB200_OK;
}

// plain or adaptive load (counts: null = samples_done everywhere); the caller holds the ErrScope
static int accum_load(crtb200_ctx *c, const float *sum, const float *sumsq, const crtb200_hit *hit0, const uint32_t *counts,
                      uint32_t samples_done) {
  if (!c || !sum || !sumsq || !hit0) return fail(CRTB200_ERR_ARG, "null argument");
  Gpu &g = *c->gpus[0];
  CUDA_TRY(cudaSetDevice(g.device));
  if (!c->acc_active) return fail(CRTB200_ERR_STATE, "no progressive session (crtb200_accum_begin)");
  if (counts && !c->acc_adaptive) return fail(CRTB200_ERR_ARG, "a counts map can only be loaded into an adaptive session");
  const size_t px = (size_t)g.sc.width * g.sc.height;
  AccumStaging stg;
  CUDA_TRY(stg.sum.ensure(px * 3));
  CUDA_TRY(stg.sumsq.ensure(px * 3));
  CUDA_TRY(stg.hit.ensure(px));
  CUDA_TRY(cudaMemcpyAsync(stg.sum.p, sum, px * 3 * sizeof(float), cudaMemcpyHostToDevice, g.stream));
  CUDA_TRY(cudaMemcpyAsync(stg.sumsq.p, sumsq, px * 3 * sizeof(float), cudaMemcpyHostToDevice, g.stream));
  CUDA_TRY(cudaMemcpyAsync(stg.hit.p, hit0, px * sizeof(HitRec), cudaMemcpyHostToDevice, g.stream));
  if (counts) {
    CUDA_TRY(stg.counts.ensure(px));
    CUDA_TRY(cudaMemcpyAsync(stg.counts.p, counts, px * sizeof(uint32_t), cudaMemcpyHostToDevice, g.stream));
  }
  const int rc = accum_load_pass(c, stg, samples_done);
  if (rc) return rc;
  c->acc_done = samples_done;
  return CRTB200_OK;
}

int crtb200_accum_load(crtb200_ctx *c, const float *sum, const float *sumsq, const crtb200_hit *hit0, uint32_t samples_done) {
  ErrScope scope(c);
  return accum_load(c, sum, sumsq, hit0, nullptr, samples_done);
}

int crtb200_accum_load_counts(crtb200_ctx *c, const float *sum, const float *sumsq, const crtb200_hit *hit0,
                              const uint32_t *counts, uint32_t passes) {
  ErrScope scope(c);
  return accum_load(c, sum, sumsq, hit0, counts, passes);
}

int crtb200_accum_progress(crtb200_ctx *c, crtb200_progress *p) {
  ErrScope scope(c);
  if (!c || !p) return fail(CRTB200_ERR_ARG, "null argument");
  if (!c->acc_active) return fail(CRTB200_ERR_STATE, "no progressive session (crtb200_accum_begin)");
  *p = crtb200_progress{};
  p->passes = c->acc_done;
  p->covered_pixels = c->acc_covered;
  p->active_pixels = c->acc_adaptive ? c->acc_active_px : c->acc_covered;
  p->pixel_samples = c->acc_adaptive ? c->acc_px_samples : c->acc_covered * c->acc_done;
  return CRTB200_OK;
}

int crtb200_accum_counts(crtb200_ctx *c, uint32_t *counts_out) {
  ErrScope scope(c);
  if (!c || !counts_out) return fail(CRTB200_ERR_ARG, "null argument");
  Gpu &g = *c->gpus[0];
  CUDA_TRY(cudaSetDevice(g.device));
  if (!c->acc_active) return fail(CRTB200_ERR_STATE, "no progressive session (crtb200_accum_begin)");
  const size_t px = (size_t)g.sc.width * g.sc.height;
  AccumStaging stg;
  CUDA_TRY(stg.counts.ensure(px));
  CUDA_TRY(cudaMemsetAsync(stg.counts.p, 0, px * sizeof(uint32_t), g.stream));
  const int rc = accum_save_pass(c, stg);
  if (rc) return rc;
  CUDA_TRY(cudaMemcpyAsync(counts_out, stg.counts.p, px * sizeof(uint32_t), cudaMemcpyDeviceToHost, g.stream));
  CUDA_TRY(cudaStreamSynchronize(g.stream));
  return CRTB200_OK;
}

int crtb200_accum_end(crtb200_ctx *c) {
  ErrScope scope(c);
  if (!c) return fail(CRTB200_ERR_ARG, "ctx is null");
  Gpu &g = *c->gpus[0];
  CUDA_TRY(cudaSetDevice(g.device));
  accum_release(c);
  return CRTB200_OK;
}

int crtb200_last_stats(crtb200_ctx *c, crtb200_stats *stats) {
  ErrScope scope(c);
  if (!c || !stats) return fail(CRTB200_ERR_ARG, "null argument");
  Gpu &g = *c->gpus[0];
  CUDA_TRY(cudaSetDevice(g.device));
  if (c->last_pending) {
    CUDA_TRY(cudaEventSynchronize(c->ev[1]));
    int rc = collect_stats(c);
    if (rc) return rc;
    c->last_pending = false;
  }
  *stats = c->last;
  return CRTB200_OK;
}

int crtb200_shard_items(crtb200_ctx *c, uint32_t shard_count, uint32_t *items) {
  ErrScope scope(c);
  if (!c || !items || shard_count == 0) return fail(CRTB200_ERR_ARG, "bad argument");
  Gpu &g = *c->gpus[0];
  if (!g.have_scene) return fail(CRTB200_ERR_STATE, "no scene uploaded");
  *items = shard_item_count(*c->gpus[0], 0, shard_count);  // shard 0 is the largest
  return CRTB200_OK;
}

int crtb200_ipc_alloc(int device, size_t bytes, void **d_ptr_out) {
  if (!d_ptr_out || bytes == 0) return fail(CRTB200_ERR_ARG, "bad argument");
  CUDA_TRY(cudaSetDevice(device));
  CUDA_TRY(cudaMalloc(d_ptr_out, bytes));
  CUDA_TRY(cudaMemset(*d_ptr_out, 0, bytes));
  return CRTB200_OK;
}
int crtb200_ipc_free(int device, void *d_ptr) {
  if (!d_ptr) return CRTB200_OK;
  CUDA_TRY(cudaSetDevice(device));
  CUDA_TRY(cudaFree(d_ptr));
  return CRTB200_OK;
}
int crtb200_ipc_export(void *d_ptr, uint8_t handle_out[CRTB200_IPC_HANDLE_BYTES]) {
  if (!d_ptr || !handle_out) return fail(CRTB200_ERR_ARG, "null argument");
  static_assert(sizeof(cudaIpcMemHandle_t) == CRTB200_IPC_HANDLE_BYTES, "IPC handle size");
  cudaIpcMemHandle_t h;
  CUDA_TRY(cudaIpcGetMemHandle(&h, d_ptr));
  std::memcpy(handle_out, &h, sizeof(h));
  return CRTB200_OK;
}
int crtb200_ipc_open(int device, const uint8_t handle[CRTB200_IPC_HANDLE_BYTES], void **d_ptr_out) {
  if (!handle || !d_ptr_out) return fail(CRTB200_ERR_ARG, "null argument");
  cudaIpcMemHandle_t h;
  std::memcpy(&h, handle, sizeof(h));
  CUDA_TRY(cudaSetDevice(device));
  CUDA_TRY(cudaIpcOpenMemHandle(d_ptr_out, h, cudaIpcMemLazyEnablePeerAccess));
  return CRTB200_OK;
}
int crtb200_ipc_close(int device, void *d_ptr) {
  if (!d_ptr) return CRTB200_OK;
  CUDA_TRY(cudaSetDevice(device));
  CUDA_TRY(cudaIpcCloseMemHandle(d_ptr));
  return CRTB200_OK;
}

int crtb200_assemble_shards(crtb200_ctx *c, const float *d_slabs, uint32_t shard_count, float *d_rgb_out,
                            uint8_t *d_rgb8_out, void *stream) {
  ErrScope scope(c);
  if (!c || !d_slabs || shard_count == 0) return fail(CRTB200_ERR_ARG, "bad argument");
  Gpu &g = *c->gpus[0];
  if (!g.have_scene) return fail(CRTB200_ERR_STATE, "no scene uploaded");
  CUDA_TRY(cudaSetDevice(g.device));
  uint32_t items = 0;
  crtb200_shard_items(c, shard_count, &items);
  // rectangle lists that leave pixels uncovered: the assembled frame keeps what d_rgb_out held there (colorBuffer
  // persistence), exactly like the unsharded path -- the mask is the one of the last render's rectangle list.
  // k_assemble sets the shard of each item itself.
  const Frame fr = frame_tiles(g, 0, shard_count);
  k_assemble<<<g.sm_count * 8, 256, 0, (cudaStream_t)stream>>>(g.sc, fr, d_slabs, items, shard_count, d_rgb_out, d_rgb8_out);
  CUDA_TRY(cudaGetLastError());
  return CRTB200_OK;
}

int crtb200_generate_rays_device(crtb200_ctx *c, const crtb200_camera *cam, float *d_rays_out, void *stream) {
  ErrScope scope(c);
  if (!c || !cam) return fail(CRTB200_ERR_ARG, "null argument");
  Gpu &g = *c->gpus[0];
  if (!g.have_scene) return fail(CRTB200_ERR_STATE, "no scene uploaded");
  CUDA_TRY(cudaSetDevice(g.device));
  int rc = check_device_ptr(g, d_rays_out, 4, "d_rays_out");
  if (rc) return rc;
  DCamera dc;
  for (int k = 0; k < 3; k++) dc.pos[k] = cam->position[k];
  for (int k = 0; k < 9; k++) dc.rot[k] = cam->rotation[k];
  k_generate_rays<<<g.sm_count * 8, 256, 0, (cudaStream_t)stream>>>(g.sc, dc, d_rays_out);
  CUDA_TRY(cudaGetLastError());
  return CRTB200_OK;
}

int crtb200_generate_rays(crtb200_ctx *c, const crtb200_camera *cam, float *rays_out) {
  ErrScope scope(c);
  if (!c || !cam || !rays_out) return fail(CRTB200_ERR_ARG, "null argument");
  Gpu &g = *c->gpus[0];
  if (!g.have_scene) return fail(CRTB200_ERR_STATE, "no scene uploaded");
  CUDA_TRY(cudaSetDevice(g.device));
  const size_t n = (size_t)g.sc.width * g.sc.height;
  if (n == 0) return CRTB200_OK;
  DevBuf<float> d;
  CUDA_TRY(d.ensure(n * 6));
  const int rc = crtb200_generate_rays_device(c, cam, d.p, g.stream);
  if (rc) return rc;
  CUDA_TRY(cudaMemcpyAsync(rays_out, d.p, n * 6 * sizeof(float), cudaMemcpyDeviceToHost, g.stream));
  CUDA_TRY(cudaStreamSynchronize(g.stream));
  return CRTB200_OK;
}

int crtb200_scene_trees(crtb200_ctx *c, crtb200_trees *t) {
  ErrScope scope(c);
  if (!c || !t) return fail(CRTB200_ERR_ARG, "null argument");
  Gpu &g = *c->gpus[0];
  if (!c->trees_built) return fail(CRTB200_ERR_STATE, "the context's scene was not uploaded with crtb200_upload_geometry");
  CUDA_TRY(cudaSetDevice(g.device));
  const crtb200_trees &k = c->kd_counts;
  t->n_meshes = k.n_meshes;
  t->n_mesh_nodes = k.n_mesh_nodes;
  t->n_mesh_leaf_refs = k.n_mesh_leaf_refs;
  t->n_top_nodes = k.n_top_nodes;
  t->n_top_leaf_refs = k.n_top_leaf_refs;
  t->reserved = 0;
  t->peak_scratch_bytes = k.peak_scratch_bytes;
  t->build_ms = k.build_ms;
  if (t->meshes && k.n_meshes) std::memcpy(t->meshes, c->kd_meshes.data(), k.n_meshes * sizeof(crtb200_mesh));
  cudaError_t e = cudaSuccess;
  auto get = [&](void *dst, const void *src, size_t bytes) {
    if (dst && bytes && e == cudaSuccess) e = cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, g.stream);
  };
  get(t->mesh_nodes, c->kd_nodes.p, (size_t)k.n_mesh_nodes * sizeof(crtb200_kdnode));
  get(t->mesh_leaf_refs, c->kd_refs.p, (size_t)k.n_mesh_leaf_refs * 4);
  get(t->top_nodes, c->kd_nodes.p + k.n_mesh_nodes, (size_t)k.n_top_nodes * sizeof(crtb200_kdnode));
  get(t->top_leaf_refs, g.top_refs.p, (size_t)k.n_top_leaf_refs * 4);
  if (e == cudaSuccess) e = cudaStreamSynchronize(g.stream);
  CUDA_TRY(e);
  return CRTB200_OK;
}

int crtb200_debug_scene_layout(crtb200_ctx *c, int device_index, crtb200_scene_layout *l) {
  ErrScope scope(c);
  if (!c || !l) return fail(CRTB200_ERR_ARG, "null argument");
  if (device_index < 0 || (size_t)device_index >= c->gpus.size()) return fail(CRTB200_ERR_ARG, "device_index out of range");
  Gpu &x = *c->gpus[device_index];
  if (!x.have_scene) return fail(CRTB200_ERR_STATE, "no scene uploaded");
  static_assert(sizeof(DMesh) == 20, "crtb200_scene_layout.meshes holds 5 words per mesh");
  l->n_nodes = x.n_nodes;
  l->n_leaf_refs = x.n_leaf_refs;
  l->n_top_refs = x.n_top_refs;
  l->n_meshes = x.sc.n_meshes;
  l->top_begin = x.sc.top_begin;
  l->top_end = x.sc.top_end;
  l->nested_ok = x.nested_ok ? 1u : 0u;
  l->reserved = 0;
  CUDA_TRY(cudaSetDevice(x.device));
  cudaError_t e = cudaSuccess;
  auto get = [&](void *dst, const void *src, size_t bytes) {
    if (dst && bytes && e == cudaSuccess) e = cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, x.stream);
  };
  get(l->nodes, x.nodes_p, (size_t)x.n_nodes * 32);
  get(l->leaf_refs, x.leaf_refs_p, (size_t)x.n_leaf_refs * 4);
  get(l->top_refs, x.top_refs.p, (size_t)x.n_top_refs * 4);
  get(l->meshes, x.meshes.p, (size_t)x.sc.n_meshes * sizeof(DMesh));
  if (e == cudaSuccess) e = cudaStreamSynchronize(x.stream);
  cudaSetDevice(c->gpus[0]->device);
  CUDA_TRY(e);
  return CRTB200_OK;
}

int crtb200_debug_scene_geometry(crtb200_ctx *c, int device_index, float *tri_geom_out, float *vertex_normal_out) {
  ErrScope scope(c);
  if (!c) return fail(CRTB200_ERR_ARG, "null argument");
  if (device_index < 0 || (size_t)device_index >= c->gpus.size()) return fail(CRTB200_ERR_ARG, "device_index out of range");
  Gpu &x = *c->gpus[device_index];
  if (!x.have_scene) return fail(CRTB200_ERR_STATE, "no scene uploaded");
  CUDA_TRY(cudaSetDevice(x.device));
  cudaError_t e = cudaSuccess;
  if (tri_geom_out && x.n_triangles)
    e = cudaMemcpyAsync(tri_geom_out, x.tri_geom_p, (size_t)x.n_triangles * 3 * sizeof(float4), cudaMemcpyDeviceToHost, x.stream);
  if (vertex_normal_out && c->n_vertices && e == cudaSuccess)  // float4 (n, 0) per vertex -> 3 floats
    e = cudaMemcpy2DAsync(vertex_normal_out, 3 * sizeof(float), x.vtx_normal.p, sizeof(float4), 3 * sizeof(float), c->n_vertices,
                          cudaMemcpyDeviceToHost, x.stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(x.stream);
  cudaSetDevice(c->gpus[0]->device);
  CUDA_TRY(e);
  return CRTB200_OK;
}

int crtb200_debug_powf5(crtb200_ctx *c, const float *x, uint32_t n, float *out) {
  ErrScope scope(c);
  if (!c || !x || !out) return fail(CRTB200_ERR_ARG, "null argument");
  if (n == 0) return CRTB200_OK;
  Gpu &g = *c->gpus[0];
  CUDA_TRY(cudaSetDevice(g.device));
  DevBuf<float> dx, dy;
  CUDA_TRY(dx.ensure(n));
  CUDA_TRY(dy.ensure(n));
  CUDA_TRY(cudaMemcpyAsync(dx.p, x, (size_t)n * 4, cudaMemcpyHostToDevice, g.stream));
  k_powf5<<<g.sm_count * 8, 256, 0, g.stream>>>(dx.p, n, dy.p);
  CUDA_TRY(cudaGetLastError());
  CUDA_TRY(cudaMemcpyAsync(out, dy.p, (size_t)n * 4, cudaMemcpyDeviceToHost, g.stream));
  CUDA_TRY(cudaStreamSynchronize(g.stream));
  return CRTB200_OK;
}

// the checks of a ray batch that need no pointer attributes (crtb200_trace_rays_device and its host wrapper)
static int check_batch(crtb200_ctx *c, const crtb200_ray_batch *b) {
  if (!c || !b || !b->rays) return fail(CRTB200_ERR_ARG, "null argument");
  Gpu &g = *c->gpus[0];
  if (!g.have_scene) return fail(CRTB200_ERR_STATE, "no scene uploaded");
  if (b->n >= 0x80000000u) return fail(CRTB200_ERR_ARG, "a ray batch holds fewer than 2^31 rays");
  if (b->ray_type > CRTB200_RAY_REFRACTION) return fail(CRTB200_ERR_ARG, "bad ray type (primary, shadow, reflection or refraction)");
  if (b->traversal > 1) return fail(CRTB200_ERR_ARG, "unknown traversal mode");
  if (b->count_work > 2) return fail(CRTB200_ERR_ARG, "unknown count_work mode");
  if (b->ray_type == CRTB200_RAY_SHADOW ? (!b->max_distance || !b->occluded) : !b->hits)
    return fail(CRTB200_ERR_ARG, "missing output / distance array");
  return CRTB200_OK;
}

int crtb200_trace_rays_device(crtb200_ctx *c, const crtb200_ray_batch *b, void *stream) {
  ErrScope scope(c);
  int rc = check_batch(c, b);
  if (rc || b->n == 0) return rc;
  Gpu &g = *c->gpus[0];
  CUDA_TRY(cudaSetDevice(g.device));
  const bool shadow = b->ray_type == CRTB200_RAY_SHADOW;
  if ((rc = check_device_ptr(g, b->rays, 4, "rays"))) return rc;
  if (shadow && ((rc = check_device_ptr(g, b->max_distance, 4, "max_distance")) || (rc = check_device_ptr(g, b->occluded, 1, "occluded"))))
    return rc;
  if (!shadow && (rc = check_device_ptr(g, b->hits, 4, "hits"))) return rc;
  static_assert(sizeof(HitRec) == sizeof(crtb200_hit), "hit records are written in the public layout");
  // contiguous ranges, one per GPU (a batch smaller than the GPU list uses its first n GPUs)
  const uint32_t n = (uint32_t)std::min<size_t>(c->gpus.size(), b->n);
  for (uint32_t i = 0; i < n; i++) {
    CUDA_TRY(cudaSetDevice(c->gpus[i]->device));
    if ((rc = query_scratch(*c->gpus[i]))) return rc;
  }
  CUDA_TRY(cudaSetDevice(g.device));
  for (Event &e : c->query_ev) CUDA_TRY(e.create(cudaEventDefault));
  const cudaStream_t st = (cudaStream_t)stream;
  const Flavour fl = query_flavour(g, b);
  c->query_pending = false;
  CUDA_TRY(cudaEventRecord(c->query_ev[0], st));
  uint32_t launches = 0;
  rc = fan_out(c, n, st, false, [&](uint32_t i, Gpu &x, cudaStream_t xs) {
    const uint64_t begin = (uint64_t)b->n * i / n, end = (uint64_t)b->n * (i + 1) / n;
    const QueryBatch qb{b->rays + 6 * begin, shadow ? b->max_distance + begin : nullptr,
                        shadow ? nullptr : reinterpret_cast<HitRec *>(b->hits + begin), shadow ? b->occluded + begin : nullptr,
                        (uint32_t)(end - begin)};
    int e = enqueue_query(x, fl, b->ray_type, qb, xs, launches);
    if (e == CRTB200_OK && cudaGetLastError() != cudaSuccess) e = fail(CRTB200_ERR_CUDA, "a query launch failed");
    return e;
  });
  if (rc) return rc;
  CUDA_TRY(cudaEventRecord(c->query_ev[1], st));
  c->query_last = crtb200_stats{};
  uint64_t *rays[4] = {&c->query_last.rays_primary, &c->query_last.rays_shadow, &c->query_last.rays_reflection,
                       &c->query_last.rays_refraction};
  *rays[b->ray_type] = b->n;
  c->query_last.kernel_launches = launches;
  c->query_gpus = n;
  c->query_pending = true;
  return CRTB200_OK;
}

int crtb200_last_query_stats(crtb200_ctx *c, crtb200_stats *stats) {
  ErrScope scope(c);
  if (!c || !stats) return fail(CRTB200_ERR_ARG, "null argument");
  CUDA_TRY(cudaSetDevice(c->gpus[0]->device));
  if (c->query_pending) {
    CUDA_TRY(cudaEventSynchronize(c->query_ev[1]));
    float ms = 0.f;
    CUDA_TRY(cudaEventElapsedTime(&ms, c->query_ev[0], c->query_ev[1]));
    Counts t{c->query_last, {}};
    t.s.device_ms = ms;
    for (uint32_t i = 0; i < c->query_gpus; i++) {
      Counts x;
      CUDA_TRY(cudaSetDevice(c->gpus[i]->device));
      const int rc = read_counts(c->gpus[i]->query_stats_dev.p, x);
      if (rc) return rc;
      add_counts(t, x);
    }
    CUDA_TRY(cudaSetDevice(c->gpus[0]->device));
    c->query_last = t.s;
    c->query_pending = false;
  }
  *stats = c->query_last;
  return CRTB200_OK;
}

int crtb200_trace_rays(crtb200_ctx *c, const float *rays, uint32_t n, uint32_t ray_type, uint32_t traversal,
                       const float *max_distance, crtb200_hit *hits_out, uint8_t *occluded_out) {
  ErrScope scope(c);
  crtb200_ray_batch b{n, ray_type, traversal, 0, rays, max_distance, hits_out, occluded_out};
  int rc = check_batch(c, &b);
  if (rc || n == 0) return rc;
  Gpu &g = *c->gpus[0];
  CUDA_TRY(cudaSetDevice(g.device));
  const bool shadow = ray_type == CRTB200_RAY_SHADOW;
  DevBuf<float> d_rays, d_dist;
  DevBuf<crtb200_hit> d_hits;
  DevBuf<uint8_t> d_occ;
  CUDA_TRY(d_rays.ensure((size_t)n * 6));
  CUDA_TRY(cudaMemcpyAsync(d_rays.p, rays, (size_t)n * 6 * sizeof(float), cudaMemcpyHostToDevice, g.stream));
  if (shadow) {
    CUDA_TRY(d_dist.ensure(n));
    CUDA_TRY(d_occ.ensure(n));
    CUDA_TRY(cudaMemcpyAsync(d_dist.p, max_distance, (size_t)n * sizeof(float), cudaMemcpyHostToDevice, g.stream));
  } else {
    CUDA_TRY(d_hits.ensure(n));
  }
  b.rays = d_rays.p;
  b.max_distance = d_dist.p;
  b.hits = d_hits.p;
  b.occluded = d_occ.p;
  if ((rc = crtb200_trace_rays_device(c, &b, g.stream))) return rc;
  if (shadow)
    CUDA_TRY(cudaMemcpyAsync(occluded_out, d_occ.p, n, cudaMemcpyDeviceToHost, g.stream));
  else
    CUDA_TRY(cudaMemcpyAsync(hits_out, d_hits.p, (size_t)n * sizeof(crtb200_hit), cudaMemcpyDeviceToHost, g.stream));
  CUDA_TRY(cudaStreamSynchronize(g.stream));
  return CRTB200_OK;
}

// Caller rays through the frame pipeline (DESIGN.md 3.13): each GPU's contiguous range is a frame request whose level 0
// is that range (enqueue_frame's chunk loop, sample_pass's level loop), fanned out as frames are.
int crtb200_shade_rays_device(crtb200_ctx *c, const crtb200_shade_batch *b, void *stream) {
  ErrScope scope(c);
  if (!c || !b || !b->rays || !b->rgb) return fail(CRTB200_ERR_ARG, "null argument");
  if (b->n >= 0x80000000u) return fail(CRTB200_ERR_ARG, "a ray batch holds fewer than 2^31 rays");
  if (b->ray_type != CRTB200_RAY_PRIMARY && b->ray_type != CRTB200_RAY_REFLECTION && b->ray_type != CRTB200_RAY_REFRACTION)
    return fail(CRTB200_ERR_ARG, "bad ray type (primary, reflection or refraction)");
  if (b->traversal > 1) return fail(CRTB200_ERR_ARG, "unknown traversal mode");
  if (b->count_work > 2) return fail(CRTB200_ERR_ARG, "unknown count_work mode");
  if (b->max_depth > 31) return fail(CRTB200_ERR_ARG, "max_depth > 31 is not supported");
  Gpu &g = *c->gpus[0];
  if (!g.have_scene) return fail(CRTB200_ERR_STATE, "no scene uploaded");
  if (b->n == 0) return CRTB200_OK;
  CUDA_TRY(cudaSetDevice(g.device));
  int rc;
  if ((rc = check_device_ptr(g, b->rays, 4, "rays")) || (rc = check_device_ptr(g, b->rgb, 4, "rgb")) ||
      (b->hits && (rc = check_device_ptr(g, b->hits, 4, "hits"))))
    return rc;
  crtb200_options o{};
  o.max_depth = b->max_depth;
  o.shadow_bias = b->shadow_bias;
  o.reflection_bias = b->reflection_bias;
  o.refraction_bias = b->refraction_bias;
  o.traversal = b->traversal;
  o.count_work = b->count_work;
  const uint32_t stat = b->ray_type == CRTB200_RAY_PRIMARY ? CRT_STAT_RAYS_PRIMARY
                        : b->ray_type == CRTB200_RAY_REFLECTION ? CRT_STAT_RAYS_REFLECTION : CRT_STAT_RAYS_REFRACTION;
  const cudaStream_t st = (cudaStream_t)stream;
  c->last = crtb200_stats{};
  c->last_pending = true;
  // contiguous ranges, one per GPU, as crtb200_trace_rays_device splits a batch; a range keeps its global p
  const uint32_t n = (uint32_t)std::min<size_t>(c->gpus.size(), b->n);
  c->frame_gpus = n;
  rc = fan_out(c, n, st, true, [&](uint32_t i, Gpu &x, cudaStream_t xs) {
    const uint64_t begin = (uint64_t)b->n * i / n, end = (uint64_t)b->n * (i + 1) / n;
    const ShadeRays sr{b->rays + 6 * begin, b->rgb + 3 * begin, b->hits ? reinterpret_cast<HitRec *>(b->hits + begin) : nullptr,
                       b->first_index + (uint32_t)begin, stat};
    FrameReq r(nullptr, &o, c->sampling);
    r.rays = &sr;
    r.n_rays = (uint32_t)(end - begin);
    r.sample = b->sample;
    return enqueue_frame(c, x, r, xs);
  });
  if (rc) return rc;
  if (n > 1) CUDA_TRY(cudaEventRecord(c->ev[1], st));  // the call ends when the last GPU has stored its range
  return CRTB200_OK;
}

}  // extern "C"
