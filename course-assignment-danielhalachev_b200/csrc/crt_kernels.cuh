// crt_kernels.cuh -- the wavefront pipeline kernels (sm_100a).
//
//   K1  primary-ray generation      fused into k_closest<CameraRays> / k_shade (level 0) + standalone k_generate_rays
//   K2  k_closest                   persistent closest-hit traversal, one ray per lane, stack-free two-level KD walk
//   K4/K5 k_shade                   per-hit: barycentrics, smooth normal, texture sample, material switch,
//                                   reflect / refract + Fresnel, compaction of children into the next level's queue
//   K3  k_shadow                    persistent any-hit traversal, one (diffuse hit, light) pair per lane -> visibility;
//                                   K2 and K3 run one loop (walk_loop) with a walk kind each
//   K2b/K3b k_coop                  the walks K2 / K3 hand off once their queue is dry: one warp per walk, a LIFO of
//                                   subtrees in shared memory; an early pass runs next to the traversal kernel
//                                   (k_mark tells it that the kernel has ended), a final pass behind both
//   K3c k_accumulate                in-order light sum per diffuse hit
//   K6  k_resolve                   bottom-up combine of the ray tree in the reference's expression order
//   K7  k_store                     level-0 colours -> framebuffer (f32 + PPMColor u8); k_store_rays for caller rays
// k_closest, k_shadow, k_coop, k_shade and k_resolve take a ray source as a template and a kernel parameter (see "Ray
// sources"): a frame's queue (QueueRays), camera rays (CameraRays) and (hit, light) pairs (ShadowPairs), a caller's
// rays shaded through the frame pipeline (ShadeRays), a caller's closest-hit and shadow queries (QueryClosest /
// QueryShadow).
//
// Reference functions replaced are cited at each kernel.  No tensor cores: the path is pointer-chasing + scalar
// binary32 arithmetic; the B200-specific choices are the 32-byte-sector node records, L2-resident working set,
// persistent grids sized to 148 SMs x resident CTAs, warp-aggregated queue compaction (ballot / shuffle).
#pragma once
#include "crt_device.cuh"
#include "crt_powf5.h"
#include "crt_sampling.h"
#include <type_traits>

namespace crtd {

#define CRT_FULL_MASK 0xFFFFFFFFu
#ifndef CRT_TRAV_MIN_BLOCKS
#define CRT_TRAV_MIN_BLOCKS 4   // resident CTAs per SM the register allocation is bounded for
#endif
#ifndef CRT_TRAV_MIN_BLOCKS_SEC
// ... of k_closest's secondary-level instantiation.  A secondary level has ~18 warps' worth of rays per SM and is bound
// by the latency of each warp's instruction chain, not by occupancy: 3 blocks = 76-85 registers, no spills
// (run r2aj: hw11_room 2.79 -> 2.61 ms; the primary and shadow kernels lose 4-5 % with 3).
#define CRT_TRAV_MIN_BLOCKS_SEC 3
#endif
#define CRT_MAX_LEVELS 34

struct Frame {
  DCamera cam;
  uint32_t tiles_x, n_tiles;          // 8x4-pixel tiles over the whole image
  uint32_t shard_index, shard_count;  // tile t belongs to shard t % shard_count
  const uint8_t *mask;                // optional per-pixel coverage (rectangles that do not tile the image)
  uint32_t item_begin;                // first level-0 work item of this chunk (shard-local numbering)
  uint32_t n_items0;                  // level-0 work items in this chunk
  uint32_t max_depth;
  uint32_t resolve;                   // 1 when the frame has secondary levels: k_resolve will read the combine records
  float shadow_bias, reflection_bias, refraction_bias;
  // sampling contract (crt_sampling.h, DESIGN.md 3.10).  gi = 0: the unsampled frame, none of the fields below is read
  uint32_t gi, gi_samples;            // diffuse children per diffuse hit (G)
  uint32_t sample, spp;               // sample pass of this launch, samples per pixel
  uint32_t seed, frame_index;         // Philox key
  float mc_bias;                      // MONTE_CARLO_BIAS: diffuse ray origin = P + N * mc_bias
  // adaptive session passes (DESIGN.md 3.10.2): level-0 slot j holds the ray of shard item list[j], j < *n_list (both
  // written on the device by k_adapt_compact); null in every other launch
  const uint32_t *list, *n_list;
};

struct Levels {
  float4 *ray_o;      // xyz origin, w = parent node (unused; GI frames: bits of the ray's path key)  -- indexed by node id - offset[1]
  float4 *ray_d;      // xyz direction (normalised twice), w = ray type (GI frames: bits of the global pixel index)
  uint32_t *hit_tri;  // per node: global triangle id or CRT_INVALID
  float *hit_t;
  float4 *color;      // per node: resolved colour
  uint4 *comb;        // per node: {kind, childA, childB / material, bits(F)}
  float4 *dq;         // diffuse queue, 3 x float4 per item: {P, bits(node)} {N, base.r} {base.g, base.b, -, -}
  uint8_t *vis;       // per (diffuse item, light): 1 = the light is visible from the hit
  uint32_t *counts;   // [CRT_MAX_LEVELS] rays per level; [CRT_MAX_LEVELS] = diffuse queue length
  unsigned long long *stats;  // device counters of the frame, CRT_STAT_SLOTS of them (named below)
  uint32_t offset[CRT_MAX_LEVELS + 1];
  // tail hand-off (k_coop): once the work queue of a traversal kernel is dry, the walks still running are written to
  // ovf[] (3 x uint4 per record) and finished one WARP per ray; tail_iters = 0 switches this off
  uint4 *ovf;
  uint32_t *ovf_ctl;  // per traversal launch L (level, or CRT_MAX_LEVELS for the shadow pass) one 128-byte line at
                      // ovf_ctl + 32 L: [0] written, [8] / [16] next record index of the early / the final k_coop pass,
                      // [24] != 0 once the traversal kernel has ended
  uint32_t ovf_cap;     // walks k_coop can take per launch (CRT_TAIL_CAP = 8 per resident k_coop warp): hand-off stops there
  uint32_t tail_iters;  // 0 = off; else tail_iters - 1 = the floor of the hand-off threshold (see tail_policy)
  uint32_t tail_start;  // the threshold's value when the queue of a large launch has just run dry: shadow pass (512)
  uint32_t tail_start_closest;  // ... closest-hit launches
  uint32_t tail_small;  // launches of at most this many rays hand off at the floor from the start (see tail_policy)
  uint32_t skip_zero_terms;  // 1 (default traversal): shadow rays whose light term is exactly zero are answered without a walk
};

// slots of Levels::stats
enum : uint32_t {
  CRT_STAT_RAYS_PRIMARY = 0, CRT_STAT_RAYS_SHADOW = 1, CRT_STAT_RAYS_REFLECTION = 2, CRT_STAT_RAYS_REFRACTION = 3,
  CRT_STAT_NODES_CLOSEST = 4, CRT_STAT_TRIS_CLOSEST = 5, CRT_STAT_NODES_SHADOW = 6, CRT_STAT_TRIS_SHADOW = 7,
  CRT_STAT_PHASE = 8,       // CRT_PHASE_CLOCKS: 8 phase clocks / counts of k_closest, then 8 of k_shadow
  CRT_STAT_WARP_SPAN = 24,  // CRT_PHASE_CLOCKS: warp lifetimes, warps, last end, first start of k_closest, then k_shadow
  CRT_STAT_HANDOFF_CLOSEST = 32, CRT_STAT_HANDOFF_SHADOW = 33,  // walks handed to k_coop
  CRT_STAT_COOP_DEBUG = 34,  // CRT_COOP_STATS: iterations, box tests, triangle tests of k_coop closest, then shadow
  CRT_STAT_ZERO_TERM = 40,   // shadow rays answered without a walk
  CRT_STAT_DIFFUSE = 41, CRT_STAT_PX_SAMPLES = 42, CRT_STAT_STOPPED = 43,
  CRT_STAT_SLOTS = 48
};

// COMB_GI = {kind, first diffuse child (CRT_INVALID: beyond max_depth, every child is the background), diffuse item, G}
enum { COMB_FINAL = 0, COMB_REFLECT = 1, COMB_FRESNEL = 2, COMB_COPY = 3, COMB_GI = 4 };

// Jittered primary ray of sample fr.sample of pixel (row, col): r = R(p, s, 0, 0), x = col + unit(r[0]),
// y = row + unit(r[1]), then getRay unchanged.  Returns the root path key r[2].
CRT_DI uint32_t jittered_primary_ray(const Frame &fr, uint32_t W, uint32_t H, uint32_t row, uint32_t col, V3 &o, V3 &d) {
  const crt_s_u4 r = crt_s_philox(row * W + col, fr.sample, 0u, 0u, fr.seed, fr.frame_index);
  primary_ray_at(fr.cam, W, H, fadd((float)col, crt_s_unit(r.x)), fadd((float)row, crt_s_unit(r.y)), o, d);
  return r.z;
}

CRT_DI uint32_t lane_id() { return threadIdx.x & 31u; }
CRT_DI uint32_t lanemask_lt() {
  uint32_t m;
  asm("mov.u32 %0, %%lanemask_lt;" : "=r"(m));
  return m;
}

// Warp-aggregated allocation: every lane of the (fully converged) warp asks for n slots; one atomic per warp.
CRT_DI uint32_t warp_alloc(uint32_t *counter, uint32_t n) {
  uint32_t incl = n;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    uint32_t v = __shfl_up_sync(CRT_FULL_MASK, incl, d);
    if (lane_id() >= (uint32_t)d) incl += v;
  }
  uint32_t total = __shfl_sync(CRT_FULL_MASK, incl, 31);
  uint32_t base = 0;
  if (lane_id() == 31 && total) base = atomicAdd(counter, total);
  base = __shfl_sync(CRT_FULL_MASK, base, 31);
  return base + incl - n;
}

// Adds a per-lane counter, summed over the (fully converged) warp, to stats[slot]: one atomic per warp, none for a zero sum.
template <class T>
CRT_DI void warp_stat_add(const Levels &lv, const uint32_t slot, T v) {
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(CRT_FULL_MASK, v, d);
  if (lane_id() == 0 && v) atomicAdd(&lv.stats[slot], (unsigned long long)v);
}

// level-0 work item -> pixel.  Items are numbered tile-major (8x4 tiles) so a warp starts on one coherent tile.
// LIST: the caller may run in an adaptive pass (GI level-0 kernels), where item_begin + j stands for shard item list[j].
template <bool LIST = false>
CRT_DI bool item_pixel(const Frame &fr, const DScene &sc, uint32_t item, uint32_t &row, uint32_t &col) {
  if (LIST && fr.list) {
    const uint32_t j = item - fr.item_begin;
    if (j >= *fr.n_list) return false;
    item = fr.list[j];
  }
  const uint32_t local_tile = item >> 5, l = item & 31u;
  const unsigned long long gt = (unsigned long long)local_tile * fr.shard_count + fr.shard_index;
  if (gt >= fr.n_tiles) return false;
  const uint32_t ty = (uint32_t)gt / fr.tiles_x, tx = (uint32_t)gt % fr.tiles_x;
  col = tx * 8u + (l & 7u);
  row = ty * 4u + (l >> 3);
  if (col >= sc.width || row >= sc.height) return false;
  if (fr.mask && !fr.mask[(size_t)row * sc.width + col]) return false;
  return true;
}

// level-0 slots of this chunk's launches: the device count of an adaptive pass, else every item of the chunk
template <bool LIST>
CRT_DI uint32_t level0_items(const Frame &fr) { return (LIST && fr.list) ? *fr.n_list : fr.n_items0; }

// ------------------------------------------------------------------------------------------------------------
// MODE 2 building blocks: warp-cooperative triangle phase.
//
// ncu (profiles/r1c) showed the merged loop's triangle path running at ~8 of 32 lanes (its three edge tests at 3 / 2 / 1
// lanes) serialised with a ~16-lane node path in every iteration.  MODE 2 splits the round differently:
//   node phase   lanes that need an AABB step take one per iteration while at least CRT_NODE_MIN lanes do; a lane that
//                reaches a leaf parks with its triangle range pending
//   tri phase    the pending ranges of ALL parked lanes are concatenated (shuffle prefix sum) and dealt out 32 at a
//                time: slot g of the concatenation is tested by lane g % 32 against its OWNER's ray, which every lane
//                can read from the warp's shared-memory ray table.  Owners are found from a ballot of segment heads.
//                Candidates are handed back to their owners in slot order, i.e. in the reference's encounter order
//                (a lane has at most one pending leaf), so closest_offer sees exactly the sequence of KDTree.cpp:59-63.
// ------------------------------------------------------------------------------------------------------------
// CRT_PHASE_CLOCKS (debug builds for tools/ only): per-warp clock64 time spent in the refill / between-trees / node /
// triangle phases of the MODE 2 kernels, plus iteration counts, summed into stats[CRT_STAT_PHASE + 8 * kernel + i] and printed by
// crtb200_core.cu after every frame.
#ifndef CRT_PHASE_CLOCKS
#define CRT_PHASE_CLOCKS 0
#endif
#if CRT_PHASE_CLOCKS
CRT_DI unsigned long long crt_globaltimer() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
__device__ unsigned long long g_warp_rec[2][8192][6];  // per warp: start, end (globaltimer ns), rounds, node iterations, time after dry, stolen
__device__ unsigned long long g_tail[2][2];
__device__ unsigned long long g_iter_hist[2][32];  // debug: rays by floor(log2(node-phase iterations + 1)), [0] closest [1] shadow
#define CRT_PC_RAY_DONE(k, it) { atomicAdd(&g_iter_hist[k][31 - __clz((int)(it) + 1)], 1ull); }
#define CRT_PC_DECL long long pc_t = clock64(); unsigned long long pc_acc[8] = {0, 0, 0, 0, 0, 0, 0, 0}; const unsigned long long pc_g0 = crt_globaltimer(); \
  long long pc_tail_t = 0; unsigned long long pc_tail_time = 0, pc_tail_lanes = 0;
// after the work queue is exhausted: wall time of the warp's remaining life and busy-lane x time within it
#define CRT_PC_TAIL(exh, act) { if (exh) { const long long n_ = clock64(); if (pc_tail_t) { pc_tail_time += (unsigned long long)(n_ - pc_tail_t); \
  pc_tail_lanes += (unsigned long long)(n_ - pc_tail_t) * __popc(__ballot_sync(CRT_FULL_MASK, act)); } pc_tail_t = n_; } }
#define CRT_PC_MARK(i) { const long long n_ = clock64(); pc_acc[i] += (unsigned long long)(n_ - pc_t); pc_t = n_; }
#define CRT_PC_COUNT(i, v) { pc_acc[i] += (v); }
#define CRT_PC_FLUSH(base) { if (lane_id() == 0) { for (int i_ = 0; i_ < 8; i_++) atomicAdd(&lv.stats[(base) + i_], pc_acc[i_]); \
    const unsigned long long g1_ = crt_globaltimer(); const int kb_ = CRT_STAT_WARP_SPAN + ((base) - CRT_STAT_PHASE) / 2; \
    atomicAdd(&lv.stats[kb_], g1_ - pc_g0); atomicAdd(&lv.stats[kb_ + 1], 1ull); atomicMax(&lv.stats[kb_ + 2], g1_); \
    atomicMin(&lv.stats[kb_ + 3], pc_g0 ? pc_g0 : 1ull); \
    atomicAdd(&g_tail[((base) - CRT_STAT_PHASE) / 8][0], pc_tail_time); atomicAdd(&g_tail[((base) - CRT_STAT_PHASE) / 8][1], pc_tail_lanes); \
    const uint32_t w_ = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; if (w_ < 8192u) { unsigned long long *r_ = g_warp_rec[((base) - CRT_STAT_PHASE) / 8][w_]; \
      r_[0] = pc_g0; r_[1] = g1_; r_[2] = pc_acc[7]; r_[3] = pc_acc[5]; r_[4] = pc_tail_time; r_[5] = pc_acc[6]; } } }
#else
#define CRT_PC_TAIL(exh, act)
#define CRT_PC_RAY_DONE(k, it)
#define CRT_PC_DECL
#define CRT_PC_MARK(i)
#define CRT_PC_COUNT(i, v)
#define CRT_PC_FLUSH(base)
#endif

#ifndef CRT_NODE_MIN
#define CRT_NODE_MIN 16  // leave the node phase when fewer lanes than this still need an AABB step (and leaves wait)
#endif

// Node-phase exit threshold: with `na` lanes active, keep stepping while at least min(CRT_NODE_MIN, na / 2) lanes (but
// at least one) want an AABB step.  Lanes leave the node phase only by parking (leaf pending / cursor off its tree), so
// when the loop exits with fewer steppers than that, the triangle phase or trav_slow has work: no livelock.
CRT_DI uint32_t node_threshold(uint32_t na) {
  const uint32_t h = na >> 1;
  return h < 1u ? 1u : (h < (uint32_t)CRT_NODE_MIN ? h : (uint32_t)CRT_NODE_MIN);
}

struct __align__(16) WarpShare {
  float4 ro[32];         // ray origin of lane i, w = distance to the light (shadow rays)
  float4 rd[32];         // ray direction of lane i
  uint32_t refbase[32];  // owner lane i: first pending leaf reference minus its start slot
  uint32_t owner[32];    // window slot h holding a segment head -> owner lane
};

// Runs the triangle tests of every parked lane.  `pending` lanes have tv.tref..tv.tend set.  On return those ranges are
// consumed.  CLOSEST: candidates are offered to cl in order.  SHADOW: `occluded` is set for owners with a candidate whose
// hit point is within the light distance (AccelerationStructure.cpp:73-74).
template <bool SHADOW, bool PRIMARY, bool COUNT>
CRT_DI void tri_phase(const DScene &sc, WarpShare &ws, const bool pending, const bool flush, uint32_t &tref, const uint32_t tend,
                      Closest &cl, bool &occluded, uint32_t &n_tris) {
  const uint32_t lane = lane_id();
  const uint32_t cnt = pending ? tend - tref : 0u;
  uint32_t incl = cnt;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const uint32_t v = __shfl_up_sync(CRT_FULL_MASK, incl, d);
    if (lane >= (uint32_t)d) incl += v;
  }
  uint32_t total = __shfl_sync(CRT_FULL_MASK, incl, 31);
  const uint32_t start = incl - cnt;
  if (cnt) ws.refbase[lane] = tref - start;
  for (uint32_t base = 0; base < total; base += 32u) {
    // segment heads of this window: an owner whose range intersects [base, base + 32) marks its first slot in the window
    const bool in_win = cnt && start < base + 32u && start + cnt > base;
    const uint32_t hp = (in_win && start > base) ? start - base : 0u;
    const uint32_t heads = __reduce_or_sync(CRT_FULL_MASK, in_win ? (1u << hp) : 0u);
    if (in_win) ws.owner[hp] = lane;
    __syncwarp();
    const uint32_t g = base + lane;
    bool hit = false;
    float t = 0.0f;
    uint32_t tri = 0, own = 0;
    if (g < total) {
      own = ws.owner[31 - __clz(heads & (CRT_FULL_MASK >> (31u - lane)))];  // slot 0 of a window is always a head
      tri = ld_ref(&sc.leaf_refs[ws.refbase[own] + g]);
      const float4 g0 = ld_tri(&sc.tri_geom[3 * (size_t)tri]);
      const float4 g1 = ld_tri(&sc.tri_geom[3 * (size_t)tri + 1]);
      const float4 g2 = ld_tri(&sc.tri_geom[3 * (size_t)tri + 2]);
      const float4 o4 = ws.ro[own], d4 = ws.rd[own];
      Ray r;
      r.o = mk(o4.x, o4.y, o4.z);
      r.d = mk(d4.x, d4.y, d4.z);
      r.flags = PRIMARY ? 8u : 0u;
      V3 p;
      if (COUNT) n_tris++;
      hit = triangle_test(g0, g1, g2, r, t, p);
      if (SHADOW) hit = hit && vlen(vsub(p, r.o)) <= o4.w;
    }
    // hand the candidates to their owners in slot (= encounter) order
    uint32_t hm = __ballot_sync(CRT_FULL_MASK, hit);
    while (hm) {
      const int l = __ffs(hm) - 1;
      hm &= hm - 1u;
      const uint32_t o_l = __shfl_sync(CRT_FULL_MASK, own, l);
      if (SHADOW) {
        if (lane == o_l) occluded = true;
      } else {
        const uint32_t tri_l = __shfl_sync(CRT_FULL_MASK, tri, l);
        const float t_l = __shfl_sync(CRT_FULL_MASK, t, l);
        if (lane == o_l) closest_offer(cl, tri_l, t_l);
      }
    }
    __syncwarp();  // ws.owner is rewritten by the next window
  }
  if (cnt) {
    const uint32_t done = total > start ? total - start : 0u;  // slots of this owner that were dealt out
    tref += done < cnt ? done : cnt;
  }
}


// ------------------------------------------------------------------------------------------------------------
// Tail hand-off.  A ray is walked by one lane, and 2-3 % of the rays of a large-mesh frame need hundreds of node-phase
// iterations: once the queue is dry a traversal kernel used to wait 0.3-0.8 ms for its last few lanes (DESIGN.md 3.8).
// Now, once the queue is dry (every warp polls the global cursor, so a warp full of long walks learns it too), a lane
// whose walk has taken more node-phase iterations than a falling threshold (tail_threshold) hands it to k_coop, where
// a group of lanes finishes it; young walks keep going here (most end within a few iterations).  k_coop's capacity
// bounds how many walks are handed off per launch.  A walk's state goes into one 48-byte record
//   r0 = {ray id (queue node / visibility slot), cur, cend, resume}     r1 = {mref, mend, seen lo, seen hi}
//   r2 = {below, bits(mu), bits(best_t), best_tri}
// written at the top of a round, where no lane has a pending triangle range.  min_t is implied: best_t when that is
// below +inf, else +inf (closest_offer keeps it so).
// ------------------------------------------------------------------------------------------------------------
// Hand-off policy of one launch (uniform over the grid; `total` = rays of the launch, `lanes` = threads of the grid).
// A walk costs k_coop about five times the instructions it costs a lane here (profiles/r2_tuning.md), so k_coop pays
// only for walks whose serial latency would otherwise set the kernel's end, and only while it is not itself the
// bottleneck:
//   large launch (total > lanes)   the queue runs dry late, with walks of every age in flight.  Threshold = 512
//                                  node-phase iterations when the queue has just run dry, halved every 4 rounds
//                                  (~20 us) down to the floor: the longest walks go first, and k_coop's capacity
//                                  (Levels::ovf_cap) closes the hand-off.
//   small launch (total <= lanes)  every ray is in flight from the start and the kernel IS its tail.  With at most
//                                  tail_small rays k_coop can take every walk that turns out long: threshold = floor
//                                  from the start.  With more (the secondary levels of a whole reflective frame:
//                                  ~90 k rays, half of them long) k_coop would be the bottleneck: no hand-off.
// Returns the threshold start value, or CRT_INVALID for "no hand-off in this launch".
#ifndef CRT_TAIL_DECAY_SHIFT
#define CRT_TAIL_DECAY_SHIFT 2  // the threshold halves every 2^this rounds once the queue is dry
#endif
#ifndef CRT_TAIL_POLL_MASK
#define CRT_TAIL_POLL_MASK 3    // the queue's dry flag is polled every (this + 1)-th round ...
#endif
#ifndef CRT_TAIL_POLL_MASK_BIG
#define CRT_TAIL_POLL_MASK_BIG 7  // ... in launches with more than CRT_TAIL_BIG rays per grid lane
#endif
#ifndef CRT_TAIL_BIG
#define CRT_TAIL_BIG 32
#endif
// When a warp learns that the queue is dry decides when it starts handing off.  A launch with many rays per lane (a whole
// 4K frame: 55) still has the SMs full of work at that moment, and k_coop's instructions compete with it: polling every
// 8th round instead of every 4th is worth 4 % there; tile shards and small launches (2-14 rays per lane) lose 3-8 %
// with it (profiles/r2_tuning.md 5.8).
CRT_DI uint32_t tail_poll_mask(const uint32_t total) {
  return total / (gridDim.x * blockDim.x) >= (uint32_t)CRT_TAIL_BIG ? (uint32_t)CRT_TAIL_POLL_MASK_BIG : (uint32_t)CRT_TAIL_POLL_MASK;
}
CRT_DI uint32_t tail_policy(const Levels &lv, const uint32_t total, const bool shadow) {
  if (!lv.tail_iters) return CRT_INVALID;
  const uint32_t lanes = gridDim.x * blockDim.x;
  if (total > lanes) return shadow ? lv.tail_start : lv.tail_start_closest;
  return total <= lv.tail_small ? lv.tail_iters - 1u : CRT_INVALID;
}
CRT_DI uint32_t tail_threshold(const Levels &lv, const uint32_t start, const uint32_t dry_rounds) {
  const uint32_t sh = dry_rounds >> CRT_TAIL_DECAY_SHIFT, t = sh < 31u ? (start >> sh) : 0u;
  return t > lv.tail_iters - 1u ? t : lv.tail_iters - 1u;
}
// Every hot counter of a launch has a 128-byte line of its own (CRT_CTL_STRIDE words): the work cursor (one atomicAdd per
// refill of every warp), its "dry" flag, and the hand-off counters.  The warps poll the FLAG, which the warp that takes
// the last rays sets, so the 4 700 readers stay off the line the refills' atomics go to.
#define CRT_CTL_STRIDE 32u
#define CRT_DRY_FLAG 16u  // word offset of the dry flag behind a work cursor
CRT_DI bool queue_dry(const uint32_t *work_counter) {
  uint32_t v = 0;
  if (lane_id() == 0) v = *reinterpret_cast<const volatile uint32_t *>(work_counter + CRT_DRY_FLAG);
  return __shfl_sync(CRT_FULL_MASK, v, 0) != 0u;
}
CRT_DI void queue_mark_dry(uint32_t *work_counter) {
  if (lane_id() == 0) *reinterpret_cast<volatile uint32_t *>(work_counter + CRT_DRY_FLAG) = 1u;
}
// `closed` (warp-uniform) is set once the record buffer is full: the warp stops asking
CRT_DI bool tail_handoff(const Levels &lv, const uint32_t launch, const bool want, const uint32_t id, const Trav &tv,
                         const float best_t, const uint32_t best_tri, bool &closed) {
  const uint32_t wm = __ballot_sync(CRT_FULL_MASK, want);
  if (!wm) return false;
  uint32_t base = 0;
  if (lane_id() == 0) base = atomicAdd(&lv.ovf_ctl[CRT_CTL_STRIDE * launch], (uint32_t)__popc(wm));
  base = __shfl_sync(CRT_FULL_MASK, base, 0);
  const uint32_t r = base + __popc(wm & lanemask_lt());
  if (base + (uint32_t)__popc(wm) >= lv.ovf_cap) closed = true;
  if (!want || r >= lv.ovf_cap) return false;  // k_coop's capacity is used up: the lane keeps walking here
  // r0.x (the ray id, never CRT_INVALID) is also the record's "published" flag: k_coop's early pass runs concurrently
  // with this kernel and takes a record by exchanging r0.x back to CRT_INVALID, so r0 goes out last, behind a fence
  uint4 *rec = lv.ovf + 3 * (size_t)r;
  rec[1] = make_uint4(tv.mref, tv.mend, (uint32_t)tv.seen, (uint32_t)(tv.seen >> 32));
  rec[2] = make_uint4(tv.below, __float_as_uint(tv.mu), __float_as_uint(best_t), best_tri);
  __threadfence();
  rec[0] = make_uint4(id, tv.cur, tv.cend, tv.resume);
  return true;
}

// ------------------------------------------------------------------------------------------------------------
// The persistent traversal loop of K2 (k_closest) and K3 (k_shadow).
//
// Persistent warps, one ray per lane.  Every loop below has a WARP-UNIFORM trip count (its condition is a vote), so the
// 32 lanes stay converged under independent thread scheduling; per-lane work is predicated.  (A first version with
// per-lane `while (active)` loops ran at 1.8-5 active threads per instruction: ncu profiles/r1a.)  One outer round =
//   refill        when >= REFILL lanes are idle, one atomicAdd per warp hands them the next rays of the global cursor
//   between trees trav_slow for lanes whose cursor ran off a tree (next mesh of the top-level leaf / back to the top level)
//   node phase    trav_fast2: lanes that need an AABB step take one (two consecutive nodes at once) per iteration while
//                 at least node_threshold() lanes do; a lane that reaches a leaf parks with its triangle range pending
//   tri phase     tri_phase: the parked ranges, packed across the warp
// MODE: 2 = this loop.  (0 = while-while and 1 = merged single loop were the round-1 predecessors; their measurements are
// in profiles/r1_tuning.md, their code is gone.)
//
// A walk kind (ClosestWalk, ShadowWalk, each over a ray source) holds the per-lane state of a walk's answer and supplies
// the steps that differ.  `id` is the source's record id of the ray, where its answer goes and the hand-off record's id:
//   total, take(i, ray, id)  work items of the launch; the ray of item i (false: the item is answered without a walk)
//   begin(ray, i, id)        a new walk's answer state; tri_dist() = w of its entry in the warp's ray table
//   limit(), allow_behind()  the node phase's culling bound (node_test)
//   tri()                    the triangle phase; true when the lane's answer can no longer change
//   answer(), handoff()      the result of a finished walk; the record of a walk handed to k_coop (tail_handoff)
//   finish(lv)               the walk kind's own counters
//   SHADOW                   also the index of its CRT_PHASE_CLOCKS records; STAT_NODES / STAT_TRIS: its COUNT slots
// SKIPR, DEDUP: trav_slow's; COUNT: count node and triangle tests; HANDOFF: hand long walks to k_coop once the queue is
// dry; EARLY: end a walk as soon as tri() reports its answer final.
template <int REFILL, bool CULL, bool WIDE, bool SKIPR, int DEDUP, bool COUNT, bool HANDOFF, bool EARLY, class W>
CRT_DI void walk_loop(const DScene &sc, const Frame &fr, const Levels &lv, uint32_t *work_counter, WarpShare &ws, W &w) {
  const uint32_t total = w.total;
  const uint32_t lane = lane_id();
  const uint32_t tail_start = HANDOFF ? tail_policy(lv, total, W::SHADOW) : CRT_INVALID;
  const uint32_t poll_mask = tail_poll_mask(total);
  bool active = false, exhausted = false, closed = false;
  uint32_t id = 0, n_nodes = 0, n_tris = 0, round = 0, walk_iters = 0, dry_rounds = 0;
#if CRT_PHASE_CLOCKS
  uint32_t ray_iters = 0;
#endif
  Ray ray;
  Trav tv;
  ray.o = ray.d = ray.inv = mk(0.f, 0.f, 0.f);
  ray.flags = 0;
  trav_begin<WIDE>(tv, sc);
  CRT_PC_DECL
  for (;;) {
    CRT_PC_MARK(4)
    CRT_PC_COUNT(7, 1)
    const uint32_t idle = __ballot_sync(CRT_FULL_MASK, !active);
    if (!exhausted && __popc(idle) >= REFILL) {
      const uint32_t want = __popc(idle);
      uint32_t start = 0;
      if (lane == 0) start = atomicAdd(work_counter, want);
      start = __shfl_sync(CRT_FULL_MASK, start, 0);
      if (start + want >= total) {
        if (!exhausted && start < total) queue_mark_dry(work_counter);  // (the warp that takes the last rays)
        exhausted = true;
      }
      const uint32_t i = start + __popc(idle & lanemask_lt());
      if (!active && i < total && w.take(sc, fr, lv, i, ray, id)) {
        ray_prepare(ray, W::PRIMARY);
        trav_begin<WIDE>(tv, sc);
        w.begin(ray, i, id);
        active = true;
        walk_iters = 0;
#if CRT_PHASE_CLOCKS
        ray_iters = 0;
#endif
        ws.ro[lane] = make_float4(ray.o.x, ray.o.y, ray.o.z, w.tri_dist());
        ws.rd[lane] = make_float4(ray.d.x, ray.d.y, ray.d.z, 0.f);
      }
    }
    if (HANDOFF && tail_start != CRT_INVALID) {
      if (!exhausted && (++round & poll_mask) == 0u) exhausted = queue_dry(work_counter);
      if (exhausted && !closed) {
        const uint32_t thr = tail_threshold(lv, tail_start, dry_rounds++);
        if (w.handoff(lv, active && walk_iters >= thr, id, tv, closed)) active = false;
      }
    }
    if (!__any_sync(CRT_FULL_MASK, active)) {
      if (exhausted) break;
      continue;
    }
    CRT_PC_MARK(0)
    CRT_PC_TAIL(exhausted, active)
    // ---- between-trees bookkeeping for lanes whose cursor ran off a tree (rare) ----
    for (;;) {
      const bool slow = active && tv.tref == tv.tend && tv.cur == tv.cend;
      if (!__any_sync(CRT_FULL_MASK, slow)) break;
      if (slow && trav_slow<SKIPR, DEDUP, CULL>(tv, sc, ray) == TRAV_DONE) {
        w.answer(lv, id);
        active = false;
        CRT_PC_RAY_DONE(W::SHADOW, ray_iters)
      }
    }
    CRT_PC_MARK(1)
    // ---- node phase: one AABB step per iteration while enough lanes want one ----
    bool need = active && tv.tref == tv.tend;
    const uint32_t thr = node_threshold(__popc(__ballot_sync(CRT_FULL_MASK, active)));
    // A lane's ray stays fixed through the phase (refill runs before it): when no stepping lane holds a ray of the
    // select-exact slab path (CRT_RAY_SLOW_MASK: axis-parallel or non-finite components, rare), the loop runs the box
    // test without that path, its flag test and its reconvergence point.
    const auto node_loop = [&](auto slow) {
      constexpr bool SLOW = decltype(slow)::value;
      uint32_t step = need;  // a 32-bit flag: a bool carried through the loop is repacked as a byte every iteration
      while ((uint32_t)__popc(__ballot_sync(CRT_FULL_MASK, step)) >= thr) {
        CRT_PC_COUNT(5, 1)
#if CRT_PHASE_CLOCKS
        if (step) ray_iters++;
#endif
        if (step) {
          walk_iters++;
          step = CRT_NODE_PAIR ? trav_fast2<COUNT, CULL, SLOW>(tv, sc, ray, n_nodes, cull_margins(ray, tv.mu), w.limit(), w.allow_behind())
                               : trav_fast<COUNT, CULL, SLOW>(tv, sc, ray, n_nodes, cull_margins(ray, tv.mu), w.limit(), w.allow_behind());
        }
      }
      need = step;
    };
    if (__any_sync(CRT_FULL_MASK, need && (ray.flags & CRT_RAY_SLOW_MASK)))
      node_loop(std::true_type());
    else
      node_loop(std::false_type());
    CRT_PC_MARK(2)
    // ---- triangle phase: all pending leaves, packed across the warp ----
    const bool parked = active && tv.tref != tv.tend;
    if (__any_sync(CRT_FULL_MASK, parked)) {
      CRT_PC_COUNT(6, 1)
      const bool done = w.template tri<COUNT>(sc, ws, parked, !__any_sync(CRT_FULL_MASK, need), tv, n_tris);
      if (EARLY && active && done) {  // early termination: the rest of the walk cannot change the answer
        tv.tref = tv.tend = 0;
        w.answer(lv, id);
        active = false;
        CRT_PC_RAY_DONE(W::SHADOW, ray_iters)
      }
    }
    CRT_PC_MARK(3)
  }
  CRT_PC_FLUSH(CRT_STAT_PHASE + 8 * W::SHADOW)
  w.finish(lv);
  if (COUNT) {
    warp_stat_add(lv, W::STAT_NODES, (unsigned long long)n_nodes);
    warp_stat_add(lv, W::STAT_TRIS, (unsigned long long)n_tris);
  }
}

// ------------------------------------------------------------------------------------------------------------
// K2: closest hit.  Replaces RayTracer::trace -> KDTree<ObjectKDTreeSubTree>::intersect -> KDTree<Triangle>::intersect
// (RayTracer.cpp:453-458, KDTree.cpp:127-166, 48-87).  Work item = one ray of the launch's source; the answer is its
// closest hit (a frame's: the ray node's hit_tri / hit_t).
//
// Ray sources (here the frame's QueueRays and CameraRays; ShadowPairs with K3, ShadeRays and the query sources at the end).
// A source says where the rays of a launch come from and where their answers go.  k_closest / k_shadow walk its items
// and k_coop reads the walks they hand off through the same source object, so a walk and its hand-off read the same
// ray bits.  Per-kernel flags (F: JITTER of k_closest, ZERO_TERMS of k_shadow, GI of k_shade / k_resolve) reach it as
// member-template arguments; the back-face rule (PRIMARY) is the kernel's own flag.
//   SHADOW                                   its rays are shadow rays (k_shadow) or closest-hit rays (k_closest)
//   level(l)                                 the level of a launch at `l`; 0 for the caller's rays, whose launches are
//                                            level 0 by construction (also the hand-off line of a closest-hit launch)
//   items<F>(fr, lv, level), base(lv, level) closest hit: work items of the launch, record id of item 0 (id = base + i)
//   take<F>(sc, fr, lv, base, i, ray)        closest hit: the ray of item i; false: not a ray of the launch
//   base(lv), items(sc, base)                shadow: a word of the launch take() reads, work items
//   take<F>(sc, fr, lv, base, i, ray, dist, id, n)  shadow: the ray of item i, its distance bound and record id; false:
//                                            answered without a walk (n += 1)
//   ray(sc, fr, lv, id, ray, dist)           the ray of record id again (k_coop); shadow: with its distance bound
//   limit(ray, dist), declined(lv, n)        shadow: the culling bound (CULL); counts the items take() declined
//   answer(sc, lv, id, cl) / answer(lv, id, occluded)  where a closest hit / an occlusion answer goes
// The level-0 sources of a frame request (CameraRays, ShadeRays) also feed level 0 of k_shade / k_resolve:
//   valid<GI>(sc, fr, i)                     level-0 slot i holds a ray
//   level0<GI>(sc, fr, i, valid, o, d, key, pix, n)  valid: slot i holds a ray; then its ray, GI: its root path key and
//                                            pixel index, and n += 1
//   ray_stat()                               the CRT_STAT_RAYS_* slot its rays count in
// ------------------------------------------------------------------------------------------------------------
// The frame's rays of level > 0: node base + i of the queue.  Its launches are the frame's secondary levels (k_closest's
// CRT_TRAV_MIN_BLOCKS_SEC).
struct QueueRays {
  static constexpr bool SHADOW = false;
  CRT_DI uint32_t level(const uint32_t l) const { return l; }
  template <bool>
  CRT_DI uint32_t items(const Frame &, const Levels &lv, const uint32_t level) const { return lv.counts[level]; }
  CRT_DI uint32_t base(const Levels &lv, const uint32_t level) const { return lv.offset[level]; }
  template <bool>
  CRT_DI bool take(const DScene &, const Frame &, const Levels &lv, const uint32_t base, const uint32_t i, Ray &ray) const {
    const float4 o = lv.ray_o[base - lv.offset[1] + i];
    const float4 d = lv.ray_d[base - lv.offset[1] + i];
    ray.o = mk(o.x, o.y, o.z);
    ray.d = mk(d.x, d.y, d.z);
    return true;
  }
  CRT_DI void ray(const DScene &, const Frame &, const Levels &lv, const uint32_t id, Ray &ray, float &) const {
    const float4 o = lv.ray_o[id - lv.offset[1]], d = lv.ray_d[id - lv.offset[1]];
    ray.o = mk(o.x, o.y, o.z);
    ray.d = mk(d.x, d.y, d.z);
  }
  CRT_DI void answer(const DScene &, const Levels &lv, const uint32_t id, const Closest &cl) const {
    lv.hit_tri[id] = cl.best_tri;
    lv.hit_t[id] = cl.best_t;
  }
};

// Level 0 of a frame: the pixel of the tile mapping and its camera ray, jittered in GI frames; answered into the frame's
// hit records like the queue's rays.  The walk's JITTER is a template flag, so that the unsampled primary kernels keep
// their register allocation; k_coop tests fr.gi at run time, so one k_coop serves both.  The level stays a kernel
// parameter: k_shade / k_resolve over camera rays run every level of a frame (levels > 0 read the queue, not the source).
struct CameraRays : QueueRays {
  template <bool JITTER>
  CRT_DI uint32_t items(const Frame &fr, const Levels &, const uint32_t) const { return level0_items<JITTER>(fr); }
  template <bool JITTER>
  CRT_DI bool take(const DScene &sc, const Frame &fr, const Levels &, const uint32_t, const uint32_t i, Ray &ray) const {
    uint32_t row, col;
    if (!item_pixel<JITTER>(fr, sc, fr.item_begin + i, row, col)) return false;
    if (JITTER)
      jittered_primary_ray(fr, sc.width, sc.height, row, col, ray.o, ray.d);
    else
      primary_ray(fr.cam, sc.width, sc.height, row, col, ray.o, ray.d);
    return true;
  }
  CRT_DI void ray(const DScene &sc, const Frame &fr, const Levels &lv, const uint32_t id, Ray &ray, float &) const {
    uint32_t row, col;
    item_pixel<true>(fr, sc, fr.item_begin + (id - lv.offset[0]), row, col);  // valid: the main kernel started this ray
    if (fr.gi)
      jittered_primary_ray(fr, sc.width, sc.height, row, col, ray.o, ray.d);
    else
      primary_ray(fr.cam, sc.width, sc.height, row, col, ray.o, ray.d);
  }
  template <bool GI>
  CRT_DI bool valid(const DScene &sc, const Frame &fr, const uint32_t i) const {
    uint32_t row, col;
    return item_pixel<GI>(fr, sc, fr.item_begin + i, row, col);
  }
  // (keeps the statement structure k_shade had before the sources existed: the register allocation of k_shade<false>
  // depends on it)
  template <bool GI>
  CRT_DI void level0(const DScene &sc, const Frame &fr, const uint32_t i, bool &valid, V3 &o, V3 &d, uint32_t &key,
                     uint32_t &pix, uint32_t &n) const {
    uint32_t row, col;
    valid = item_pixel<GI>(fr, sc, fr.item_begin + i, row, col);
    if (valid) {
      if (GI) {
        key = jittered_primary_ray(fr, sc.width, sc.height, row, col, o, d);
        pix = row * sc.width + col;
      } else {
        primary_ray(fr.cam, sc.width, sc.height, row, col, o, d);
      }
      n++;
    }
  }
  CRT_DI uint32_t ray_stat() const { return CRT_STAT_RAYS_PRIMARY; }
};

// A closest-hit walk over the rays of source Src; the answer is the closest hit of the ray.
template <bool P, bool JITTER, class Src>
struct ClosestWalk {
  static constexpr bool PRIMARY = P, SHADOW = false;
  static constexpr uint32_t STAT_NODES = CRT_STAT_NODES_CLOSEST, STAT_TRIS = CRT_STAT_TRIS_CLOSEST;
  const uint32_t level, total, base;
  Closest cl;
  const DScene &sc;
  const Src &src;
  CRT_DI ClosestWalk(const DScene &s, const Frame &fr, const Levels &lv, const uint32_t lvl, const Src &r)
      : level(r.level(lvl)), total(r.template items<JITTER>(fr, lv, level)), base(r.base(lv, level)), sc(s), src(r) {
    closest_begin(cl);
  }
  CRT_DI bool take(const DScene &s, const Frame &fr, const Levels &lv, const uint32_t i, Ray &ray, uint32_t &) const {
    return src.template take<JITTER>(s, fr, lv, base, i, ray);
  }
  CRT_DI void begin(const Ray &, const uint32_t i, uint32_t &id) {
    closest_begin(cl);
    id = base + i;
  }
  CRT_DI float tri_dist() const { return 0.f; }
  // conservative culling: beyond the best finite hit; behind the origin once a finite hit exists (crt_device.cuh)
  CRT_DI float limit() const { return cl.min_t; }
  CRT_DI bool allow_behind() const { return cl.min_t < CRT_INF; }
  template <bool COUNT>
  CRT_DI bool tri(const DScene &s, WarpShare &ws, const bool parked, const bool flush, Trav &tv, uint32_t &n_tris) {
    bool dummy = false;
    tri_phase<false, PRIMARY, COUNT>(s, ws, parked, flush, tv.tref, tv.tend, cl, dummy, n_tris);
    return false;
  }
  CRT_DI void answer(const Levels &lv, const uint32_t id) const { src.answer(sc, lv, id, cl); }
  CRT_DI bool handoff(const Levels &lv, const bool want, const uint32_t id, const Trav &tv, bool &closed) const {
    return tail_handoff(lv, level, want, id, tv, cl.best_t, cl.best_tri, closed);
  }
  CRT_DI void finish(const Levels &) const {}
};

// Work item = one ray of src at `level`; PRIMARY: the primary ray's back-face rule (Ray.cpp:13).
template <class Src, bool PRIMARY, bool COUNT, int REFILL, int MODE, bool CULL, bool WIDE, bool JITTER = false>
__global__ void __launch_bounds__(CRT_TRAV_BLOCK, std::is_same<Src, QueueRays>::value ? CRT_TRAV_MIN_BLOCKS_SEC : CRT_TRAV_MIN_BLOCKS)
    k_closest(const DScene sc, const Frame fr, const Levels lv, const uint32_t level, uint32_t *__restrict__ work_counter, const Src src) {
  static_assert(MODE == 2, "only loop mode 2 is implemented");
  __shared__ WarpShare s_ws[CRT_TRAV_BLOCK / 32];
  WarpShare &ws = s_ws[threadIdx.x >> 5];
  ClosestWalk<PRIMARY, JITTER, Src> w(sc, fr, lv, level, src);
  walk_loop<REFILL, CULL, WIDE, false, (COUNT ? 0 : (WIDE ? 2 : 1)), COUNT, !COUNT, false>(sc, fr, lv, work_counter, ws, w);
}

// ------------------------------------------------------------------------------------------------------------
// Texture::getColor x4                                                          Texture.cpp:14-72
// ------------------------------------------------------------------------------------------------------------
CRT_DI V3 texture_color(const DScene &sc, const DTexture &t, const uint4 sh, float b0, float b1, float b2) {
  if (t.kind == 0u) return mk(t.color_a[0], t.color_a[1], t.color_a[2]);
  if (t.kind == 1u) {
    if (b0 < t.scalar || b1 < t.scalar || b2 < t.scalar) return mk(t.color_b[0], t.color_b[1], t.color_b[2]);
    return mk(t.color_a[0], t.color_a[1], t.color_a[2]);
  }
  float2 uv0 = make_float2(0.f, 0.f), uv1 = uv0, uv2 = uv0;
  if (sc.vtx_uv) {
    uv0 = sc.vtx_uv[sh.x];
    uv1 = sc.vtx_uv[sh.y];
    uv2 = sc.vtx_uv[sh.z];
  }
  // b0 * UV1 + b1 * UV2 + (b2 * UV0)                                            Texture.cpp:34-36, 63-65
  const float u = fadd(fadd(fmul(b0, uv1.x), fmul(b1, uv2.x)), fmul(b2, uv0.x));
  const float v = fadd(fadd(fmul(b0, uv1.y), fmul(b1, uv2.y)), fmul(b2, uv0.y));
  if (t.kind == 2u) {
    // static_cast<unsigned int>(uv / squareSize): x86 cvttss2si (64-bit) truncation; inputs are kept in range by the
    // scene contract (SURVEY App. A-10), where CUDA's saturating cvt.rzi.u32 agrees.
    const unsigned x = (unsigned)fdiv(u, t.scalar);
    const unsigned y = (unsigned)fdiv(v, t.scalar);
    if ((x & 1u) == (y & 1u)) return mk(t.color_a[0], t.color_a[1], t.color_a[2]);
    return mk(t.color_b[0], t.color_b[1], t.color_b[2]);
  }
  const int w = (int)t.width, h = (int)t.height;
  int x = (int)fmul(u, (float)w);
  int y = (int)fmul(fsub(1.0f, v), (float)h);
  x = x < 0 ? 0 : (x > w - 1 ? w - 1 : x);
  y = y < 0 ? 0 : (y > h - 1 ? h - 1 : y);
  const float *px = sc.texels + 3ull * (t.texel_offset + (unsigned long long)y * w + x);
  return mk(px[0], px[1], px[2]);
}

// ------------------------------------------------------------------------------------------------------------
// K4/K5: shade + spawn for one level.  Replaces the body of RayTracer::shootRay after trace() (RayTracer.cpp:430-450),
// the hit post-processing of KDTree<ObjectKDTreeSubTree>::intersect (KDTree.cpp:167-190), Triangle::
// getBarycentricCoordinates (Triangle.cpp:63-73), the set-up halves of calculateReflection / calculateRefraction
// (RayTracer.cpp:358-417) and Texture::getColor.  Children are compacted into level+1 with one atomic per warp.
// ------------------------------------------------------------------------------------------------------------
// The G diffuse children of a diffuse hit (P, shading normal N) of a GI frame, written to queue slots q0 .. q0 + G - 1:
// origin P + N * mc_bias, direction crt_s_diffuse_dir, path key of slot j, pixel index.  Out of line: the rejection
// loop's registers stay out of k_shade's allocation.
static __device__ __noinline__ void spawn_diffuse(const Frame &fr, const Levels &lv, const V3 P, const V3 N, const uint32_t pix,
                                                  const uint32_t key, const uint32_t q0, const uint32_t G) {
  const float n3[3] = {N.x, N.y, N.z};
  const V3 co = vadd(P, vscale(N, fr.mc_bias));
  for (uint32_t j = 0; j < G; j++) {
    float dd[3];
    crt_s_diffuse_dir(fr.seed, fr.frame_index, pix, fr.sample, key, j, n3, dd);
    lv.ray_o[q0 + j] = make_float4(co.x, co.y, co.z, __uint_as_float(crt_s_child_key(fr.seed, fr.frame_index, pix, fr.sample, key, j)));
    lv.ray_d[q0 + j] = make_float4(dd[0], dd[1], dd[2], __uint_as_float(pix));
  }
}

// GI: frames under the sampling contract (crt_sampling.h): jittered level 0, path keys carried in ray_o.w / pixel index in
// ray_d.w, and every diffuse hit also spawns G diffuse children (COMB_GI).  GI = false is the unsampled kernel.
template <bool GI, class L0>
CRT_DI void shade_level(const DScene &sc, const Frame &fr, const Levels &lv, const uint32_t level, const L0 &src) {
  const uint32_t total = (level == 0) ? level0_items<GI>(fr) : lv.counts[level];
  const uint32_t node_base = lv.offset[level];
  const uint32_t rounded = (total + 31u) & ~31u;
  uint32_t n_refl = 0, n_refr = 0, n_prim = 0, n_diff = 0;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < rounded; i += gridDim.x * blockDim.x) {
    bool valid = i < total;
    const uint32_t node = node_base + i;
    V3 o = mk(0, 0, 0), d = mk(0, 0, 0);
    uint32_t key = 0, pix = 0;  // GI: path key of this ray, global pixel index
    if (valid) {
      if (level == 0) {
        src.template level0<GI>(sc, fr, i, valid, o, d, key, pix, n_prim);
      } else {
        const float4 ro = lv.ray_o[node - lv.offset[1]];
        const float4 rd = lv.ray_d[node - lv.offset[1]];
        o = mk(ro.x, ro.y, ro.z);
        d = mk(rd.x, rd.y, rd.z);
        if (GI) {
          key = __float_as_uint(ro.w);
          pix = __float_as_uint(rd.w);
        }
      }
    }
    uint32_t want_children = 0, want_diffuse = 0;
    uint32_t kind = COMB_FINAL, mat_index = 0;
    V3 P = mk(0, 0, 0), N = mk(0, 0, 0), base = mk(0, 0, 0), out = mk(sc.bg[0], sc.bg[1], sc.bg[2]);
    V3 c0o = P, c0d = P, c1o = P, c1d = P;
    float fresnel = 0.0f;
    const V3 bg = mk(sc.bg[0], sc.bg[1], sc.bg[2]);
    const uint32_t tri = valid ? lv.hit_tri[node] : CRT_INVALID;
    if (valid && tri != CRT_INVALID) {
      const float t = lv.hit_t[node];
      const float4 g0 = __ldg(&sc.tri_geom[3 * (size_t)tri]);
      const float4 g1 = __ldg(&sc.tri_geom[3 * (size_t)tri + 1]);
      const float4 g2 = __ldg(&sc.tri_geom[3 * (size_t)tri + 2]);
      const uint4 sh = __ldg(&sc.tri_shade[tri]);
      const DMesh me = sc.meshes[sh.w];
      mat_index = me.material;
      const DMaterial mat = sc.materials[mat_index];
      P = vadd(o, vscale(d, t));  // Ray.cpp:22
      N = mk(g0.w, g1.w, g2.w);   // Ray.cpp:28
      float u = 0.0f, v = 0.0f;
      if (mat.smooth || mat.texture != CRT_INVALID) {
        // Triangle::getBarycentricCoordinates                                  Triangle.cpp:63-73
        const V3 v0 = mk(g0.x, g0.y, g0.z), v1 = mk(g1.x, g1.y, g1.z), v2 = mk(g2.x, g2.y, g2.z);
        const V3 v0p = vsub(P, v0), v0v1 = vsub(v1, v0), v0v2 = vsub(v2, v0);
        const float area = vlen(vcross(v0v1, v0v2));
        u = fdiv(vlen(vcross(v0p, v0v2)), area);
        v = fdiv(vlen(vcross(v0v1, v0p)), area);
        if (mat.smooth) {  // KDTree.cpp:180-185
          const float4 n0 = __ldg(&sc.vtx_normal[sh.x]), n1 = __ldg(&sc.vtx_normal[sh.y]), n2 = __ldg(&sc.vtx_normal[sh.z]);
          const float w = fsub(fsub(1.0f, u), v);
          N = vnorm(vadd(vadd(vscale(mk(n1.x, n1.y, n1.z), u), vscale(mk(n2.x, n2.y, n2.z), v)),
                         vscale(mk(n0.x, n0.y, n0.z), w)));
        }
      }
      const bool child_traced = level + 1 <= fr.max_depth;  // RayTracer.cpp:427-429
      if (mat.type == 0u) {                                 // Diffuse: calculateDiffusion
        want_diffuse = 1;
        base = (mat.texture != CRT_INVALID)
                   ? texture_color(sc, sc.textures[mat.texture], sh, u, v, fsub(fsub(1.0f, u), v))
                   : mk(mat.albedo[0], mat.albedo[1], mat.albedo[2]);
        if (GI) {  // G diffuse children; beyond max_depth none is traced and each contributes the background
          kind = COMB_GI;
          if (child_traced) want_children = fr.gi_samples;
        }
      } else if (mat.type == 1u) {  // Reflective: calculateReflection            RayTracer.cpp:366-373
        c0o = vadd(P, vscale(N, fr.reflection_bias));
        c0d = vnorm(vnorm(vreflect(d, N)));  // getNormalized() then shootRay's normalize
        if (child_traced) {
          want_children = 1;
          kind = COMB_REFLECT;
        } else {
          out = vadd(mk(0, 0, 0), mk(fmul(mat.albedo[0], bg.x), fmul(mat.albedo[1], bg.y), fmul(mat.albedo[2], bg.z)));
        }
      } else if (mat.type == 3u) {  // Refractive: calculateRefraction           RayTracer.cpp:381-416
        float eta1 = 1.0f, eta2 = mat.ior;
        V3 n = N;
        float idn = vdot(d, n);
        if (idn > 0.0f) {
          const float tmp = eta1;
          eta1 = eta2;
          eta2 = tmp;
          n = sscale(-1.0f, n);
          idn = -idn;
        }
        const float cos_a = -idn;
        const float sin_a = fsqrt(stdmax(0.0f, fsub(1.0f, fmul(cos_a, cos_a))));
        c0o = vadd(P, vscale(n, fr.reflection_bias));
        c0d = vnorm(vnorm(vreflect(d, n)));
        const float eta = fdiv(eta1, eta2);
        const float sin_b = fmul(eta, sin_a);
        if (sin_b < 1.0f) {
          const float r = fdiv(fsub(eta1, eta2), fadd(eta1, eta2));
          const float r0 = fmul(r, r);  // powf(r, 2) == r*r bit for bit (SURVEY section 7)
          fresnel = fadd(r0, fmul(fsub(1.0f, r0), crt_powf5(fsub(1.0f, cos_a))));
          const float cos_b = fsqrt(stdmax(0.0f, fsub(1.0f, fmul(sin_b, sin_b))));
          const V3 dir = vsub(sscale(eta, vadd(d, sscale(cos_a, n))), sscale(cos_b, n));
          c1o = vsub(P, vscale(n, fr.refraction_bias));
          c1d = vnorm(vnorm(dir));
          if (child_traced) {
            want_children = 2;
            kind = COMB_FRESNEL;
          } else {
            out = vadd(sscale(fresnel, bg), sscale(fsub(1.0f, fresnel), bg));
          }
        } else {
          if (child_traced) {
            want_children = 1;
            kind = COMB_COPY;
          } else {
            out = bg;
          }
        }
      }  // Constant / default: background                                       RayTracer.cpp:443-446
    }
    // ---- queue compaction: one atomic per warp per queue ----
    const uint32_t child = warp_alloc(&lv.counts[level + 1], want_children);
    const uint32_t dslot = warp_alloc(&lv.counts[CRT_MAX_LEVELS], want_diffuse);
    if (!valid) continue;
    if (GI && kind == COMB_GI) {
      const uint32_t cbase = want_children ? lv.offset[level + 1] + child : CRT_INVALID;
      if (want_children) spawn_diffuse(fr, lv, P, N, pix, key, cbase - lv.offset[1], want_children);
      n_diff += want_children;
      lv.comb[node] = make_uint4(COMB_GI, cbase, dslot, fr.gi_samples);
      float4 *q = lv.dq + 3 * (size_t)dslot;
      q[0] = make_float4(P.x, P.y, P.z, __uint_as_float(node));
      q[1] = make_float4(N.x, N.y, N.z, base.x);
      q[2] = make_float4(base.y, base.z, 0.f, 0.f);
    } else if (want_children) {
      const uint32_t cbase = lv.offset[level + 1] + child;
      const uint32_t q = cbase - lv.offset[1];
      // GI: children carry their path key (reflection = slot 0, refraction = slot 1) and the pixel index
      lv.ray_o[q] = make_float4(c0o.x, c0o.y, c0o.z, __uint_as_float(GI ? crt_s_child_key(fr.seed, fr.frame_index, pix, fr.sample, key, 0u) : node));
      lv.ray_d[q] = make_float4(c0d.x, c0d.y, c0d.z, __uint_as_float(GI ? pix : 2u));
      n_refl++;
      if (want_children == 2) {
        lv.ray_o[q + 1] = make_float4(c1o.x, c1o.y, c1o.z, __uint_as_float(GI ? crt_s_child_key(fr.seed, fr.frame_index, pix, fr.sample, key, 1u) : node));
        lv.ray_d[q + 1] = make_float4(c1d.x, c1d.y, c1d.z, __uint_as_float(GI ? pix : 3u));
        n_refr++;
      }
      lv.comb[node] = make_uint4(kind, cbase, kind == COMB_REFLECT ? mat_index : cbase + 1, __float_as_uint(fresnel));
    } else {
      if (fr.resolve) lv.comb[node] = make_uint4(COMB_FINAL, 0, 0, 0);  // diffuse-only frames never read it (16 B / ray saved)
      if (want_diffuse) {
        float4 *q = lv.dq + 3 * (size_t)dslot;
        q[0] = make_float4(P.x, P.y, P.z, __uint_as_float(node));
        q[1] = make_float4(N.x, N.y, N.z, base.x);
        q[2] = make_float4(base.y, base.z, 0.f, 0.f);
      } else {
        lv.color[node] = make_float4(out.x, out.y, out.z, 0.f);
      }
    }
  }
  // ray statistics (traced rays only, SURVEY 8(d)); n_prim: level-0 rays, counted under the source's type
  warp_stat_add(lv, src.ray_stat(), (unsigned long long)n_prim);
  warp_stat_add(lv, CRT_STAT_RAYS_REFLECTION, (unsigned long long)n_refl);
  warp_stat_add(lv, CRT_STAT_RAYS_REFRACTION, (unsigned long long)n_refr);
  if (GI) warp_stat_add(lv, CRT_STAT_DIFFUSE, (unsigned long long)n_diff);
}

// Level 0 reads src (CameraRays, ShadeRays), every other level the queue.
template <bool GI, class Src>
__global__ void __launch_bounds__(256) k_shade(const DScene sc, const Frame fr, const Levels lv, const uint32_t level, const Src src) {
  shade_level<GI>(sc, fr, lv, src.level(level), src);
}

// ------------------------------------------------------------------------------------------------------------
// K3: shadow any-hit.  Replaces RayTracer::hasIntersection -> ObjectKDTree::checkForIntersection (RayTracer.cpp:507-518,
// AccelerationStructure.cpp:56-94) for the shadow rays of RayTracer::calculateDiffusion (RayTracer.cpp:308-317).
// The reference runs a full closest-hit per mesh and accepts iff |P - o| <= distanceToLight; because that length is
// monotone in t, "closest passes" == "some candidate passes", so terminating on the first passing candidate is exact
// (SURVEY App. A-11).  Work item = one (diffuse hit, light) pair, light-major so a warp's lanes shoot towards the same
// light from neighbouring hits; the result is one visibility byte per pair.  (One item per pair, not per hit: the
// kernel's tail is its longest item, profiles/r1_tuning.md.)
// COUNT: 0 = no counters; 1 = count under the reference's visit-all rule (early termination disabled, same result);
// 2 = count the work this kernel really does with early termination.
// ------------------------------------------------------------------------------------------------------------
CRT_DI void shadow_ray_setup(const DScene &sc, const Frame &fr, const V3 P, const V3 N, const uint32_t light, Ray &ray,
                             float &dist, float &contrib) {
  const float PI = 3.14159274101257324219f;  // M_PIf                            RayTracer.cpp:27
  const DLight L = sc.lights[light];
  V3 ld = vsub(mk(L.pos[0], L.pos[1], L.pos[2]), P);  // RayTracer.cpp:309
  dist = vlen(ld);
  const float area = fmul(fmul(fmul(4.0f, dist), dist), PI);  // 4 * r * r * PI   RayTracer.cpp:311-312
  ld = vnorm(ld);
  const float angle = stdmax(0.0f, vdot(ld, N));
  contrib = fmul(fdiv(L.intensity, area), angle);  // (float(I) / area * angle)     RayTracer.cpp:320
  ray.o = vadd(P, vscale(N, fr.shadow_bias));        // RayTracer.cpp:316
  ray.d = ld;
}

// CULL only: no candidate beyond this parameter can satisfy |P - o| <= dist (|d| = 1 within 2 ulp; the slack covers the
// rounding of P and of the length, DESIGN.md section 3.6)
CRT_DI float shadow_limit(const Ray &ray, const float dist) {
  return dist * 1.0001f + 1e-4f + 1e-6f * (fabsf(ray.o.x) + fabsf(ray.o.y) + fabsf(ray.o.z));
}

// The diffuse hits of a frame towards each light: item i = pair (hit i % n_hits, light i / n_hits), record id = its
// visibility slot hit * n_lights + light.  ZERO_TERMS: a pair whose light term is exactly zero may be answered without
// a walk (not in the visit-all counting mode).
struct ShadowPairs {
  static constexpr bool SHADOW = true;
  CRT_DI uint32_t level(const uint32_t l) const { return l; }
  CRT_DI uint32_t base(const Levels &lv) const { return lv.counts[CRT_MAX_LEVELS]; }  // n_hits
  CRT_DI uint32_t items(const DScene &sc, const uint32_t n_hits) const { return n_hits * sc.n_lights; }
  template <bool ZERO_TERMS>
  CRT_DI bool take(const DScene &sc, const Frame &fr, const Levels &lv, const uint32_t n_hits, const uint32_t i, Ray &ray,
                   float &dist, uint32_t &slot, uint32_t &n_moot) const {
    const uint32_t light = i / n_hits, hit = i - light * n_hits;
    const float4 q0 = lv.dq[3 * (size_t)hit], q1 = lv.dq[3 * (size_t)hit + 1];
    float contrib;
    shadow_ray_setup(sc, fr, mk(q0.x, q0.y, q0.z), mk(q1.x, q1.y, q1.z), light, ray, dist, contrib);
    slot = hit * sc.n_lights + light;
    // A light term that is exactly zero needs no walk.  The reference traces the shadow ray of every (hit, light) pair
    // (RayTracer.cpp:314-317) and then adds `direct * albedo` with direct = float(I) / area * max(0, L.N)
    // (:313, :320-327): for a surface turned away from the light direct is +0, the term is (+-0, +-0, +-0) for any
    // finite albedo / texel, and x + (+-0) == x bit for bit (the sum starts at +0): visible or not, the pixel is the
    // same.  The pair still counts as a traced ray (ray counts are the reference's).
    bool moot = false;
    if (ZERO_TERMS && lv.skip_zero_terms && contrib == 0.0f) {
      const float4 q2 = lv.dq[3 * (size_t)hit + 2];
      const uint32_t nf = 0x7f800000u;
      moot = (__float_as_uint(q1.w) & nf) != nf && (__float_as_uint(q2.x) & nf) != nf && (__float_as_uint(q2.y) & nf) != nf;
    }
    if (moot) {
      lv.vis[slot] = 0;
      n_moot++;
    }
    return !moot;
  }
  CRT_DI void ray(const DScene &sc, const Frame &fr, const Levels &lv, const uint32_t id, Ray &ray, float &dist) const {
    const uint32_t hit = id / sc.n_lights, light = id - hit * sc.n_lights;
    const float4 q0 = lv.dq[3 * (size_t)hit], q1 = lv.dq[3 * (size_t)hit + 1];
    float contrib;
    shadow_ray_setup(sc, fr, mk(q0.x, q0.y, q0.z), mk(q1.x, q1.y, q1.z), light, ray, dist, contrib);
  }
  CRT_DI float limit(const Ray &ray, const float dist) const { return shadow_limit(ray, dist); }
  CRT_DI void answer(const Levels &lv, const uint32_t id, const bool occluded) const { lv.vis[id] = occluded ? 0 : 1; }
  CRT_DI void declined(const Levels &lv, const uint32_t n) const { warp_stat_add(lv, CRT_STAT_ZERO_TERM, n); }
};

// A shadow walk over the rays of source Src; the answer is whether a candidate lies within the ray's distance bound.
template <bool ZERO_TERMS, class Src>
struct ShadowWalk {
  static constexpr bool PRIMARY = false, SHADOW = true;
  static constexpr uint32_t STAT_NODES = CRT_STAT_NODES_SHADOW, STAT_TRIS = CRT_STAT_TRIS_SHADOW;
  const uint32_t base, total;
  uint32_t n_declined = 0;
  float dist = 0.0f, t_limit = 0.0f;
  bool occluded = false;
  const Src &src;
  CRT_DI ShadowWalk(const DScene &sc, const Levels &lv, const Src &r) : base(r.base(lv)), total(r.items(sc, base)), src(r) {}
  CRT_DI bool take(const DScene &sc, const Frame &fr, const Levels &lv, const uint32_t i, Ray &ray, uint32_t &id) {
    return src.template take<ZERO_TERMS>(sc, fr, lv, base, i, ray, dist, id, n_declined);
  }
  CRT_DI void begin(const Ray &ray, const uint32_t, uint32_t &) {
    t_limit = src.limit(ray, dist);
    occluded = false;
  }
  CRT_DI float tri_dist() const { return dist; }
  CRT_DI float limit() const { return t_limit; }
  CRT_DI bool allow_behind() const { return true; }
  template <bool COUNT>
  CRT_DI bool tri(const DScene &sc, WarpShare &ws, const bool parked, const bool flush, Trav &tv, uint32_t &n_tris) {
    Closest unused;
    tri_phase<true, false, COUNT>(sc, ws, parked, flush, tv.tref, tv.tend, unused, occluded, n_tris);
    return occluded;
  }
  CRT_DI void answer(const Levels &lv, const uint32_t id) const { src.answer(lv, id, occluded); }
  CRT_DI bool handoff(const Levels &lv, const bool want, const uint32_t id, const Trav &tv, bool &closed) const {
    return tail_handoff(lv, CRT_MAX_LEVELS, want, id, tv, 0.0f, CRT_INVALID, closed);
  }
  CRT_DI void finish(const Levels &lv) const { src.declined(lv, n_declined); }
};

// SKIPR: shadow rays ignore refractive meshes, as the reference does only when !useGI (AccelerationStructure.cpp:67-71);
// GI frames instantiate SKIPR = false.
template <class Src, int COUNT, int REFILL, int MODE, bool CULL, bool WIDE, bool SKIPR = true>
__global__ void __launch_bounds__(CRT_TRAV_BLOCK, CRT_TRAV_MIN_BLOCKS) k_shadow(const DScene sc, const Frame fr, const Levels lv,
                                                                             uint32_t *__restrict__ work_counter, const Src src) {
  static_assert(MODE == 2, "only loop mode 2 is implemented");
  __shared__ WarpShare s_ws[CRT_TRAV_BLOCK / 32];
  WarpShare &ws = s_ws[threadIdx.x >> 5];
  ShadowWalk<COUNT != 1, Src> w(sc, lv, src);
  walk_loop<REFILL, CULL, WIDE, SKIPR, (COUNT == 1 ? 0 : (WIDE ? 2 : 1)), (COUNT != 0), COUNT == 0, COUNT != 1>(
      sc, fr, lv, work_counter, ws, w);
}

// ------------------------------------------------------------------------------------------------------------
// K2b / K3b: k_coop -- a GROUP of lanes per handed-off walk (records written by tail_handoff).
//
// Why any order is allowed.  The reference's child boxes are the exact halves of the parent box (BoundingBox.h:60-69: one
// plane replaced by min + (max - min) / 2, which lies in [min, max] in binary32) and BoundingBox::hasIntersection is
// monotone in every plane under round-to-nearest (moving min down or max up can only lower t0 / raise t1 or widen the
// containment test of a parallel axis; a NaN never rejects).  So "leaf passes" implies "every ancestor passes": the
// leaves the reference visits (KDTree.cpp:53-72) are exactly the leaves whose OWN box passes, in tree order.
// crtb200_upload_scene verifies the nesting for the uploaded trees; without it nothing is handed off.  The set of
// tested triangles therefore does not depend on the order in which a subtree is explored, only the ORDER of the
// candidates does, and that order is restored from a key:
//   shadow rays   the answer is an OR over candidates (SURVEY App. A-11): no order needed
//   closest hit   KDTree.cpp:75-86 keeps the first candidate unless a later one has strictly smaller t.  Every candidate
//                 carries key = (leaf node index, leaf reference index) = its position in the reference's encounter
//                 order; a mesh walk reduces its candidates to (a) the minimum of (t, key) over candidates with
//                 t < +inf and (b) the candidate with the smallest key, and folds them into the ray's running Closest
//                 exactly as the in-order sequence of closest_offer calls would have.
//
// The walk.  A group of GW lanes (GW = 32, a warp, by default) keeps a LIFO of node indices in shared memory.
// One iteration pops up to GW nodes, one per lane; a lane loads its node, drops it when its whole subtree lies before
// the hand-off cursor (already walked), tests the box (node_test: the reference's slab test + the conservative culling
// of crt_device.cuh) and pushes both children of a passing inner node (first child = index + 1, second child = the
// node's `b` word).  The passing leaves of an iteration are tested together, their triangle lists packed GW slots at a
// time like tri_phase.  One iteration costs about two dependent memory round trips whatever its width, and a single
// ray's frontier is rarely wider than a dozen nodes (a walk's critical path is the tree's depth), so a whole warp per
// walk leaves most lanes idle.  Narrower groups (GW = 8 / 16: four / two walks per warp side by side) and a variant in
// which eight walks of a warp shared one frontier were built and measured: neither raised the throughput, both
// lengthened single walks (profiles/r2_tuning.md 2.1), so a walk gets the whole warp (GW = 32).
// Every group runs the same loop; group-uniform branches use the group's own lane mask for their shuffles and votes.
// ------------------------------------------------------------------------------------------------------------
#define CRT_COOP_CAP 512    // LIFO entries per warp (2 KB), shared out between its groups
#ifndef CRT_COOP_SPINS
#define CRT_COOP_SPINS 4000  // early pass: polls (0.5 us apart) for a record to be published before the group gives up
#endif
#define CRT_COOP_WARPS 4    // warps per CTA
#ifndef CRT_COOP_MIN_BLOCKS
#define CRT_COOP_MIN_BLOCKS 6  // resident CTAs per SM the register allocation is bounded for (24 warps = 96 walks per SM)
#endif
#ifndef CRT_COOP_STATS
#define CRT_COOP_STATS 0  // debug builds (tools/): iterations, box tests and triangle tests of k_coop into stats[CRT_STAT_COOP_DEBUG ..]
#endif
#ifndef CRT_COOP_GROUP
#define CRT_COOP_GROUP 32   // lanes per walk (8 and 16 measured: same throughput, longer walks; profiles/r2_tuning.md)
#endif
struct __align__(16) WarpCoop {
  uint32_t stack[CRT_COOP_CAP];
  uint32_t refbase[32], owner[32], leafidx[32];
};

struct CoopBest {            // per-lane partial result of one mesh walk (closest hit)
  float t;                   // (a) smallest t < +inf seen by this lane, ties by key
  unsigned long long key;
  uint32_t tri;
  unsigned long long fkey;   // (b) smallest key seen by this lane, whatever its t
  float ft;
  uint32_t ftri;
};
#define CRT_KEY_NONE 0xFFFFFFFFFFFFFFFFull

CRT_DI void coop_best_reset(CoopBest &cb) {
  cb.t = CRT_INF;
  cb.key = cb.fkey = CRT_KEY_NONE;
  cb.tri = cb.ftri = CRT_INVALID;
  cb.ft = 0.0f;
}

// fold the lanes' partial results of one mesh walk into the ray's running Closest (all lanes of the group end with the
// same cl); gm = the group's lane mask
template <int GW>
CRT_DI void coop_fold(const uint32_t gm, CoopBest &cb, Closest &cl) {
#pragma unroll
  for (int d = GW / 2; d > 0; d >>= 1) {
    const float t = __shfl_xor_sync(gm, cb.t, d);
    const unsigned long long key = __shfl_xor_sync(gm, cb.key, d);
    const uint32_t tri = __shfl_xor_sync(gm, cb.tri, d);
    if (t < cb.t || (t == cb.t && key < cb.key)) {
      cb.t = t;
      cb.key = key;
      cb.tri = tri;
    }
    const unsigned long long fkey = __shfl_xor_sync(gm, cb.fkey, d);
    const float ft = __shfl_xor_sync(gm, cb.ft, d);
    const uint32_t ftri = __shfl_xor_sync(gm, cb.ftri, d);
    if (fkey < cb.fkey) {
      cb.fkey = fkey;
      cb.ft = ft;
      cb.ftri = ftri;
    }
  }
  // = closest_offer over the mesh's candidates in key order: the first one is kept if nothing was kept before, and the
  // first one achieving the smallest t < +inf replaces it iff that t is strictly below the running minimum
  if (cb.fkey != CRT_KEY_NONE && cl.best_tri == CRT_INVALID) {
    cl.best_tri = cb.ftri;
    cl.best_t = cb.ft;
  }
  if (cb.key != CRT_KEY_NONE && cb.t < cl.min_t) {
    cl.min_t = cb.t;
    cl.best_t = cb.t;
    cl.best_tri = cb.tri;
  }
}

// Runs behind a traversal kernel on its stream: tells k_coop's early pass that nothing more will be published.
__global__ void k_mark(uint32_t *flag) {
  if (threadIdx.x == 0) *reinterpret_cast<volatile uint32_t *>(flag) = 1u;
}

// The body of k_coop.  Its walks come from, and their answers go to, the ray source of the traversal kernel that handed
// them off: src.ray rebuilds the ray of a record, src.limit bounds a shadow walk, src.answer writes the answer.
// SKIPR: shadow rays ignore refractive meshes (false in GI frames, see k_shadow)
template <bool SHADOW, bool PRIMARY, bool CULL, int GW, bool SKIPR, class Src>
CRT_DI void coop_walks(const DScene &sc, const Frame &fr, const Levels &lv, const uint32_t level, const uint32_t early, WarpCoop &wc,
                       const Src &src) {
  constexpr uint32_t NG = 32u / GW;            // walks per warp
  constexpr uint32_t CAP = CRT_COOP_CAP / NG;  // LIFO entries per walk
  static_assert(GW == 8 || GW == 16 || GW == 32, "group width");
  const uint32_t lane = lane_id(), gl = lane & (GW - 1u), g0 = lane & ~(GW - 1u);
  const uint32_t gm = (GW == 32 ? CRT_FULL_MASK : ((1u << GW) - 1u)) << g0;  // lanes of this group
  uint32_t *const stack = wc.stack + (g0 / GW) * CAP;
  uint32_t *const refbase = wc.refbase + g0, *const owner = wc.owner + g0, *const leafidx = wc.leafidx + g0;
  const uint32_t launch = SHADOW ? (uint32_t)CRT_MAX_LEVELS : level;
  // Two passes per traversal launch (DESIGN.md 3.8).  early = 1: launched next to the traversal kernel on a second
  // stream; its blocks become resident as the traversal kernel's blocks exit and take records while the last lanes
  // there are still walking.  Record r is waited for until it is published, the traversal kernel has ended (ovf_ctl
  // word 24 of its line, set by k_mark behind it) or CRT_COOP_SPINS polls have passed -- a bounded wait, so this pass can never hold
  // the GPU against the kernel it waits for.  early = 0: launched behind both; takes whatever is still published.
  volatile uint32_t *const ctl = lv.ovf_ctl + CRT_CTL_STRIDE * launch;
  const uint32_t n_rec = early ? lv.ovf_cap : min(ctl[0], lv.ovf_cap);
  if (!early && blockIdx.x == 0 && threadIdx.x == 0 && n_rec) atomicAdd(&lv.stats[SHADOW ? CRT_STAT_HANDOFF_SHADOW : CRT_STAT_HANDOFF_CLOSEST], (unsigned long long)n_rec);

  // group state: identical in all lanes of a group, except cb (per-lane partial results)
  bool busy = false, drained = false, in_mesh = false, occluded = false;
  uint32_t id = 0, sp = 0, from = 0;
  uint32_t cur = 0, cend = 0, resume = 0, mref = 0, mend = 0, below = 0;
  unsigned long long seen = 0ull;
  float dist = 0.0f, mu = CRT_INF, lim = CRT_INF;
  Ray ray;
  ray.o = ray.d = ray.inv = mk(0.f, 0.f, 0.f);
  ray.flags = 0;
  Closest cl;
  closest_begin(cl);
  CoopBest cb;
  coop_best_reset(cb);

#if CRT_COOP_STATS
  unsigned long long dbg_iters = 0, dbg_nodes = 0, dbg_tris = 0;
#endif
  for (;;) {
    // ---- 1. an idle group takes the next record ----
    while (!busy && !drained) {
      uint32_t r = 0, got = CRT_INVALID;
      if (gl == 0) {
        r = atomicAdd(const_cast<uint32_t *>(&ctl[early ? 8 : 16]), 1u);
        if (r < n_rec) {
          uint32_t *flag = reinterpret_cast<uint32_t *>(lv.ovf + 3 * (size_t)r);
          if (early) {
            for (uint32_t spins = 0; spins < (uint32_t)CRT_COOP_SPINS; spins++) {
              if (*reinterpret_cast<volatile uint32_t *>(flag) != CRT_INVALID) break;
              if (ctl[24]) break;  // the traversal kernel has ended: what is not published now never will be
              __nanosleep(500);
            }
          }
          got = atomicExch(flag, CRT_INVALID);  // take the record (the other pass may have been here first)
          __threadfence();
        }
      }
      r = __shfl_sync(gm, r, 0, GW);
      got = __shfl_sync(gm, got, 0, GW);
      if (r >= n_rec || (early && got == CRT_INVALID)) {
        drained = true;  // (early pass: an unpublished record ends the group; the final pass looks at every record)
      } else if (got != CRT_INVALID) {
        const uint4 r0 = __ldcg(&lv.ovf[3 * (size_t)r]), r1 = __ldcg(&lv.ovf[3 * (size_t)r + 1]), r2 = __ldcg(&lv.ovf[3 * (size_t)r + 2]);
        id = got;
        src.ray(sc, fr, lv, id, ray, dist);
        ray_prepare(ray, PRIMARY);
        // the walk's state where the main kernel left it
        cur = r0.y;
        cend = r0.z;
        resume = r0.w;
        mref = r1.x;
        mend = r1.y;
        seen = (unsigned long long)r1.z | ((unsigned long long)r1.w << 32);
        below = r2.x;
        mu = __uint_as_float(r2.y);
        cl.best_t = __uint_as_float(r2.z);
        cl.best_tri = r2.w;
        cl.min_t = (cl.best_tri != CRT_INVALID && cl.best_t < CRT_INF) ? cl.best_t : CRT_INF;
        if constexpr (SHADOW)
          lim = src.limit(ray, dist);
        else
          lim = cl.min_t;
        occluded = false;
        in_mesh = false;
        busy = true;
      }
    }
    if (!__any_sync(CRT_FULL_MASK, busy)) break;  // idle groups have just found the record list empty

    // ---- 2. between mesh walks: one step of the ray's itinerary (trav_fast / trav_slow's order of events, per group) ----
    if (busy && !in_mesh) {
      if (cur < cend) {
        if (below) {
          // (the rest of) a mesh tree: start at the root of the tree whose node range contains cur; subtrees that end at
          // or before cur are dropped by the walk
          uint32_t root = CRT_INVALID;
          for (uint32_t m0 = 0; m0 < sc.n_meshes && root == CRT_INVALID; m0 += GW) {
            const uint32_t m = m0 + gl;
            uint32_t nb = CRT_INVALID;
            if (m < sc.n_meshes) {
              const DMesh me = sc.meshes[m];
              if (cur >= me.node_begin && cur < me.node_end) nb = me.node_begin;
            }
            root = __reduce_min_sync(gm, nb);
          }
          from = cur;
          cur = cend;
          coop_best_reset(cb);
          if (root != CRT_INVALID) {
            if (gl == 0) stack[0] = root;
            sp = 1u;
            in_mesh = true;
            __syncwarp(gm);
          }
        } else {
          // one step in the top-level tree (a handful of nodes: every lane does the same step; never culled)
          const float4 lo = ld_node(&sc.nodes[2 * (size_t)cur]), hi = ld_node(&sc.nodes[2 * (size_t)cur + 1]);
          const uint32_t a = __float_as_uint(lo.w);
          const bool leaf = (a & CRT_LEAF_FLAG) != 0u;
          const bool pass = node_test<false>(lo, hi, ray, mk(CRT_INF, CRT_INF, CRT_INF), CRT_INF, false);
          cur = (pass || leaf) ? cur + 1u : a;
          if (pass && leaf) {
            mref = __float_as_uint(hi.w);
            mend = mref + (a & ~CRT_LEAF_FLAG);
            resume = cur;
            cur = cend;
            below = 1u;
          }
        }
      } else if (mref != mend) {
        const uint32_t m = __ldg(&sc.top_refs[mref++]);
        const DMesh me = sc.meshes[m];
        bool skip = SHADOW && SKIPR && sc.materials[me.material].type == 3u;  // shadow rays ignore refractive meshes (AccelerationStructure.cpp:67-71)
        if (sc.dedup_meshes == 1u) {  // (scenes with more than 64 meshes: the rest of a handed-off walk re-walks a mesh for
          const unsigned long long bit = 1ull << (m & 63u);  //  every listing, like the reference; same result)
          skip = skip || (seen & bit) != 0ull;
          seen |= bit;
        }
        if (!skip) {
          cur = me.node_begin;
          cend = me.node_end;
          mu = CULL ? cull_margin_for(ray, me.cull_margin) : CRT_INF;
        }
      } else if (below) {
        below = 0u;
        cur = resume;
        cend = sc.top_end;
      } else {
        // itinerary complete
        if (gl == 0) {
          if constexpr (SHADOW)
            src.answer(lv, id, false);
          else
            src.answer(sc, lv, id, cl);
        }
        busy = false;
      }
    }

    // ---- 3. one iteration of the mesh walk ----
    if (busy && in_mesh) {
      // pop up to GW entries; close to capacity fall back to one at a time (then the LIFO grows by at most one per step)
      const uint32_t n = (CAP - sp < 2u * GW + 40u) ? 1u : (sp < GW ? sp : GW);
      const bool have = gl < n;
      uint32_t j = 0;
      if (have) j = stack[sp - 1u - gl];
      sp -= n;
      __syncwarp(gm);
#if CRT_COOP_STATS
      if (gl == 0) dbg_iters++;
      if (have) dbg_nodes++;
#endif
      bool leaf_hit = false;
      uint32_t a = 0, b = CRT_INVALID, cnt = 0;
      if (have) {
        const float4 lo = ld_node(&sc.nodes[2 * (size_t)j]), hi = ld_node(&sc.nodes[2 * (size_t)j + 1]);
        a = __float_as_uint(lo.w);
        b = __float_as_uint(hi.w);
        const bool leaf = (a & CRT_LEAF_FLAG) != 0u;
        const uint32_t endj = leaf ? j + 1u : a;
        if (endj > from && node_test<CULL>(lo, hi, ray, cull_margins(ray, mu), lim, SHADOW || lim < CRT_INF)) {
          leaf_hit = leaf;
          if (!leaf) cnt = (b != CRT_INVALID) ? 2u : 1u;
        }
      }
      uint32_t incl = cnt;
#pragma unroll
      for (int d = 1; d < GW; d <<= 1) {
        const uint32_t v = __shfl_up_sync(gm, incl, d, GW);
        if (gl >= (uint32_t)d) incl += v;
      }
      const uint32_t total = __shfl_sync(gm, incl, GW - 1, GW);
      uint32_t at = sp + incl - cnt;
      if (cnt == 2u) stack[at++] = b;  // second child below the first: the first child's subtree is taken first
      if (cnt) stack[at] = j + 1u;
      sp += total;
      __syncwarp(gm);
      // triangles of the leaves that passed in this iteration, packed across the group (cf. tri_phase)
      if (__ballot_sync(gm, leaf_hit)) {
        const uint32_t tcnt = leaf_hit ? (a & ~CRT_LEAF_FLAG) : 0u;
        uint32_t tincl = tcnt;
#pragma unroll
        for (int d = 1; d < GW; d <<= 1) {
          const uint32_t v = __shfl_up_sync(gm, tincl, d, GW);
          if (gl >= (uint32_t)d) tincl += v;
        }
        const uint32_t ttotal = __shfl_sync(gm, tincl, GW - 1, GW);
        const uint32_t tstart = tincl - tcnt;
        if (tcnt) {
          refbase[gl] = b - tstart;
          leafidx[gl] = j;
        }
        for (uint32_t base = 0; base < ttotal; base += GW) {
          const bool in_win = tcnt && tstart < base + GW && tstart + tcnt > base;
          const uint32_t hp = (in_win && tstart > base) ? tstart - base : 0u;
          const uint32_t heads = __reduce_or_sync(gm, in_win ? (1u << hp) : 0u);
          if (in_win) owner[hp] = gl;
          __syncwarp(gm);
          const uint32_t slot = base + gl;
          bool hit = false;
          float t = 0.0f;
          if (slot < ttotal) {
#if CRT_COOP_STATS
            dbg_tris++;
#endif
            const uint32_t own = owner[31 - __clz(heads & (CRT_FULL_MASK >> (31u - gl)))];  // slot 0 of a window is always a head
            const uint32_t ref = refbase[own] + slot;
            const uint32_t tri = ld_ref(&sc.leaf_refs[ref]);
            const float4 t0 = ld_tri(&sc.tri_geom[3 * (size_t)tri]);
            const float4 t1 = ld_tri(&sc.tri_geom[3 * (size_t)tri + 1]);
            const float4 t2 = ld_tri(&sc.tri_geom[3 * (size_t)tri + 2]);
            V3 p;
            hit = triangle_test(t0, t1, t2, ray, t, p);
            if (SHADOW) {
              hit = hit && vlen(vsub(p, ray.o)) <= dist;
            } else if (hit) {
              const unsigned long long key = ((unsigned long long)leafidx[own] << 32) | ref;
              if (key < cb.fkey) {
                cb.fkey = key;
                cb.ft = t;
                cb.ftri = tri;
              }
              if (t < CRT_INF && (t < cb.t || (t == cb.t && key < cb.key))) {
                cb.t = t;
                cb.key = key;
                cb.tri = tri;
              }
            }
          }
          if (SHADOW) {
            if (__ballot_sync(gm, hit)) {
              occluded = true;
              break;
            }
          } else if (CULL) {
            // tighten the culling limit: smallest finite t of this window (t >= 0, so the int order is the float order;
            // -0.0 sorts first, which is still a correct bound)
            const int m = __reduce_min_sync(gm, (hit && t < CRT_INF) ? __float_as_int(t) : 0x7f800000);
            const float tm = __int_as_float(m);
            if (tm < lim) lim = tm;
          }
          __syncwarp(gm);
        }
      }
      if (SHADOW && occluded) {  // the first occluder ends the record (SURVEY App. A-11)
        if constexpr (SHADOW) {
          if (gl == 0) src.answer(lv, id, true);
        }
        busy = false;
        in_mesh = false;
        __syncwarp(gm);
      } else if (sp == 0u) {     // mesh walk complete
        if (!SHADOW) {
          coop_fold<GW>(gm, cb, cl);
          lim = cl.min_t;
        }
        in_mesh = false;
      }
    }
  }
#if CRT_COOP_STATS
  atomicAdd(&lv.stats[CRT_STAT_COOP_DEBUG + (SHADOW ? 3 : 0)], dbg_iters);
  atomicAdd(&lv.stats[CRT_STAT_COOP_DEBUG + (SHADOW ? 4 : 1)], dbg_nodes);
  atomicAdd(&lv.stats[CRT_STAT_COOP_DEBUG + (SHADOW ? 5 : 2)], dbg_tris);
#endif
}

// k_coop over the walks k_closest / k_shadow handed off from the rays of src at `level`
template <class Src, bool PRIMARY, bool CULL, int GW, bool SKIPR = true>
__global__ void __launch_bounds__(32 * CRT_COOP_WARPS, CRT_COOP_MIN_BLOCKS) k_coop(const DScene sc, const Frame fr, const Levels lv, const uint32_t level,
                                                                                 const uint32_t early, const Src src) {
  __shared__ WarpCoop s_wc[CRT_COOP_WARPS];
  coop_walks<Src::SHADOW, PRIMARY, CULL, GW, SKIPR>(sc, fr, lv, src.level(level), early, s_wc[threadIdx.x >> 5], src);
}

// K3c: the light loop of RayTracer::calculateDiffusion (RayTracer.cpp:308-330): per diffuse hit, walk the lights IN
// ORDER and add `direct * albedo` for the unshadowed ones, so the float sum is formed exactly like the reference's.
__global__ void __launch_bounds__(256) k_accumulate(const DScene sc, const Frame fr, const Levels lv) {
  const uint32_t n_hits = lv.counts[CRT_MAX_LEVELS];
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n_hits; i += gridDim.x * blockDim.x) {
    const float4 q0 = lv.dq[3 * (size_t)i], q1 = lv.dq[3 * (size_t)i + 1], q2 = lv.dq[3 * (size_t)i + 2];
    const V3 P = mk(q0.x, q0.y, q0.z), N = mk(q1.x, q1.y, q1.z), base = mk(q1.w, q2.x, q2.y);
    V3 acc = mk(0.f, 0.f, 0.f);
    for (uint32_t l = 0; l < sc.n_lights; l++) {
      if (lv.vis[(size_t)i * sc.n_lights + l]) {
        Ray ray;
        float dist, contrib;
        shadow_ray_setup(sc, fr, P, N, l, ray, dist, contrib);
        acc = vadd(acc, sscale(contrib, base));  // finalColor += direct * albedo   RayTracer.cpp:321-327
      }
    }
    lv.color[__float_as_uint(q0.w)] = make_float4(acc.x, acc.y, acc.z, 0.f);
  }
}

// ------------------------------------------------------------------------------------------------------------
// K6: resolve one level bottom-up.  The return path of the recursion, in the reference's expression order:
//   reflective : Color(0,0,0) += albedo (*) R                                    RayTracer.cpp:369-373
//   refractive : F * R + (1 - F) * T   |   R on total internal reflection       RayTracer.cpp:414, 416
// ------------------------------------------------------------------------------------------------------------
//   GI diffuse : (D + base (*) S) / float(G + 1), S = ((0 + L_0) + L_1) + ...,   D = the light sum k_accumulate left in
//                color[node], base from the diffuse item (sampling contract, DESIGN.md 3.10)
template <bool GI, class L0>
CRT_DI void resolve_level(const DScene &sc, const Frame &fr, const Levels &lv, const uint32_t level, const L0 &src) {
  const uint32_t total = (level == 0) ? level0_items<GI>(fr) : lv.counts[level];
  const uint32_t node_base = lv.offset[level];
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const uint32_t node = node_base + i;
    if (level == 0 && !src.template valid<GI>(sc, fr, i)) continue;
    const uint4 cb = lv.comb[node];
    if (cb.x == COMB_FINAL) continue;
    if (GI && cb.x == COMB_GI) {
      const float4 D = lv.color[node], q1 = lv.dq[3 * (size_t)cb.z + 1], q2 = lv.dq[3 * (size_t)cb.z + 2];
      V3 S = mk(0.f, 0.f, 0.f);
      for (uint32_t j = 0; j < cb.w; j++) {
        const float4 L = cb.y != CRT_INVALID ? lv.color[cb.y + j] : make_float4(sc.bg[0], sc.bg[1], sc.bg[2], 0.f);
        S = vadd(S, mk(L.x, L.y, L.z));
      }
      const float g1 = (float)(cb.w + 1u);
      lv.color[node] = make_float4(fdiv(fadd(D.x, fmul(q1.w, S.x)), g1), fdiv(fadd(D.y, fmul(q2.x, S.y)), g1),
                                   fdiv(fadd(D.z, fmul(q2.y, S.z)), g1), 0.f);
      continue;
    }
    const float4 A = lv.color[cb.y];
    V3 out;
    if (cb.x == COMB_REFLECT) {
      const DMaterial mat = sc.materials[cb.z];
      out = vadd(mk(0, 0, 0), mk(fmul(mat.albedo[0], A.x), fmul(mat.albedo[1], A.y), fmul(mat.albedo[2], A.z)));
    } else if (cb.x == COMB_FRESNEL) {
      const float4 B = lv.color[cb.z];
      const float F = __uint_as_float(cb.w);
      out = vadd(sscale(F, mk(A.x, A.y, A.z)), sscale(fsub(1.0f, F), mk(B.x, B.y, B.z)));
    } else {
      out = mk(A.x, A.y, A.z);
    }
    lv.color[node] = make_float4(out.x, out.y, out.z, 0.f);
  }
}

template <bool GI, class Src>
__global__ void __launch_bounds__(256) k_resolve(const DScene sc, const Frame fr, const Levels lv, const uint32_t level, const Src src) {
  resolve_level<GI>(sc, fr, lv, src.level(level), src);
}

// Sample pass fr.sample of a GI frame: acc = acc + c_s in sample order (acc starts at (0,0,0)); the last pass leaves
// acc / float(spp) in the level-0 colour, and sample 0's primary hit in the level-0 hit record, for k_store.  Counts
// the shadow rays of every pass but the last (k_store counts those of the last).
__global__ void __launch_bounds__(256) k_sample_acc(const DScene sc, const Frame fr, const Levels lv, float4 *__restrict__ acc,
                                                    uint2 *__restrict__ hit0) {
  if (blockIdx.x == 0 && threadIdx.x == 0 && fr.sample + 1u < fr.spp)
    atomicAdd(&lv.stats[CRT_STAT_RAYS_SHADOW], (unsigned long long)lv.counts[CRT_MAX_LEVELS] * sc.n_lights);
  const bool last = fr.sample + 1u == fr.spp;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < fr.n_items0; i += gridDim.x * blockDim.x) {
    const uint32_t node = lv.offset[0] + i;
    const float4 c = lv.color[node];
    const float4 a0 = fr.sample == 0 ? make_float4(0.f, 0.f, 0.f, 0.f) : acc[i];
    const V3 a = vadd(mk(a0.x, a0.y, a0.z), mk(c.x, c.y, c.z));
    if (fr.sample == 0 && !last) hit0[i] = make_uint2(lv.hit_tri[node], __float_as_uint(lv.hit_t[node]));
    if (last) {
      const float n = (float)fr.spp;
      lv.color[node] = make_float4(fdiv(a.x, n), fdiv(a.y, n), fdiv(a.z, n), 0.f);
      if (fr.sample != 0) {
        const uint2 h = hit0[i];
        lv.hit_tri[node] = h.x;
        lv.hit_t[node] = __uint_as_float(h.y);
      }
    } else {
      acc[i] = make_float4(a.x, a.y, a.z, 0.f);
    }
  }
}

// PPMColor: static_cast<unsigned short>(std::clamp(c, 0.0f, 1.0f) * 255)       Color.cpp:12-16
CRT_DI uint8_t quantize(float c) {
  c = (c < 0.0f) ? 0.0f : ((1.0f < c) ? 1.0f : c);
  const float s = fmul(c, 255.0f);
  return (uint8_t)(unsigned short)__float2uint_rz(s);  // NaN -> 0 like x86 cvttss2si's low 16 bits
}

// ------------------------------------------------------------------------------------------------------------
// K7: store.  colorBuffer[row][col] = color (RayTracer.cpp:106) + optional PPMColor bytes + optional hit records.
// With tile sharding and slab != nullptr the shard's pixels are ALSO written compactly (item order) for the gather.
// ------------------------------------------------------------------------------------------------------------
struct HitRec {
  int mesh, tri;
  float t;
};
// A global triangle in public numbering: h.mesh and h.tri (the triangle within its mesh), -1 and -1 for CRT_INVALID.
// h.t is the caller's.
CRT_DI void public_tri(const DScene &sc, uint32_t tri, HitRec &h) {
  h.mesh = h.tri = -1;
  if (tri != CRT_INVALID) {
    const uint32_t m = sc.tri_shade[tri].w;
    h.mesh = (int)m;
    h.tri = (int)(tri - sc.meshes[m].first_triangle);
  }
}
// The frame stores of k_store and k_accum_read.  colour(i) is level-0 item i's colour, hit(i) its HitRec; both are only
// called for items that are pixels of the frame (and hit only when `hits` is not null).
// A warp holds one 8x4 tile (items are tile-major and chunks start on tile boundaries).  When the whole tile is inside
// the frame its four 96-byte rows leave as 16-byte stores (24 lanes x float4; PPMColor: 12 lanes x 8 bytes), staged
// through shared memory: a third of the store instructions, and -- what matters when `rgb` is the frame of another GPU
// (crtb200_create_multi, shard_full_frame) -- NVLink packets of 16 bytes instead of 4.  Partial tiles, odd widths and
// unaligned frames take the scalar path.
template <class Colour, class Hit>
CRT_DI void store_items(const DScene &sc, const Frame &fr, float *__restrict__ rgb, uint8_t *__restrict__ rgb8,
                        HitRec *__restrict__ hits, float *__restrict__ slab, const Colour &colour, const Hit &hit) {
  __shared__ __align__(16) float s_f[8][96];
  __shared__ __align__(8) uint8_t s_b[8][96];
  const uint32_t lane = lane_id(), w = threadIdx.x >> 5;
  const bool aligned = (sc.width & 7u) == 0u && (fr.item_begin & 31u) == 0u && (reinterpret_cast<uintptr_t>(rgb) & 15u) == 0u &&
                       (reinterpret_cast<uintptr_t>(rgb8) & 7u) == 0u && (reinterpret_cast<uintptr_t>(slab) & 15u) == 0u;
  for (uint32_t base = blockIdx.x * blockDim.x + (threadIdx.x & ~31u); base < fr.n_items0; base += gridDim.x * blockDim.x) {
    const uint32_t i = base + lane;
    uint32_t row = 0, col = 0;
    const bool valid = i < fr.n_items0 && item_pixel(fr, sc, fr.item_begin + i, row, col);
    const float4 c = valid ? colour(i) : make_float4(0.f, 0.f, 0.f, 0.f);
    const bool whole = aligned && base + 32u <= fr.n_items0;                 // all 32 items exist (slab path)
    const bool full = whole && __all_sync(CRT_FULL_MASK, valid);             // ... and are pixels of the frame
    const size_t pix = (size_t)row * sc.width + col;
    if (whole && (slab || (full && rgb))) {
      s_f[w][3 * lane + 0] = c.x;
      s_f[w][3 * lane + 1] = c.y;
      s_f[w][3 * lane + 2] = c.z;
      __syncwarp();
      if (lane < 24u) {
        const float4 v = *reinterpret_cast<const float4 *>(&s_f[w][4 * lane]);
        if (slab) *reinterpret_cast<float4 *>(slab + 3 * (size_t)(fr.item_begin + base) + 4 * lane) = v;
        if (full && rgb) {
          const size_t p0 = (size_t)__shfl_sync(0x00FFFFFFu, (unsigned long long)pix, 0);  // tile origin
          *reinterpret_cast<float4 *>(rgb + 3 * (p0 + (size_t)(lane / 6u) * sc.width) + 4 * (lane % 6u)) = v;
        }
      }
      __syncwarp();
    }
    if (full && rgb8) {
      s_b[w][3 * lane + 0] = quantize(c.x);
      s_b[w][3 * lane + 1] = quantize(c.y);
      s_b[w][3 * lane + 2] = quantize(c.z);
      __syncwarp();
      if (lane < 12u) {
        const size_t p0 = (size_t)__shfl_sync(0x00000FFFu, (unsigned long long)pix, 0);
        *reinterpret_cast<uint2 *>(rgb8 + 3 * (p0 + (size_t)(lane / 3u) * sc.width) + 8 * (lane % 3u)) =
            *reinterpret_cast<const uint2 *>(&s_b[w][8 * lane]);
      }
      __syncwarp();
    }
    if (slab && !whole && i < fr.n_items0) {
      float *s = slab + 3 * (size_t)(fr.item_begin + i);
      s[0] = c.x;
      s[1] = c.y;
      s[2] = c.z;
    }
    if (!valid) continue;
    if (rgb && !full) {
      rgb[3 * pix + 0] = c.x;
      rgb[3 * pix + 1] = c.y;
      rgb[3 * pix + 2] = c.z;
    }
    if (rgb8 && !full) {
      rgb8[3 * pix + 0] = quantize(c.x);
      rgb8[3 * pix + 1] = quantize(c.y);
      rgb8[3 * pix + 2] = quantize(c.z);
    }
    if (hits) hits[pix] = hit(i);
  }
}

__global__ void __launch_bounds__(256) k_store(const DScene sc, const Frame fr, const Levels lv, float *__restrict__ rgb,
                                              uint8_t *__restrict__ rgb8, HitRec *__restrict__ hits,
                                              float *__restrict__ slab) {
  // shadow rays traced for this chunk = diffuse hits x lights (one per pair even when cos = 0, RayTracer.cpp:314-317)
  if (blockIdx.x == 0 && threadIdx.x == 0)
    atomicAdd(&lv.stats[CRT_STAT_RAYS_SHADOW], (unsigned long long)lv.counts[CRT_MAX_LEVELS] * sc.n_lights);
  store_items(
      sc, fr, rgb, rgb8, hits, slab, [&](uint32_t i) { return lv.color[lv.offset[0] + i]; },
      [&](uint32_t i) {
        const uint32_t tri = lv.hit_tri[lv.offset[0] + i];
        HitRec h;
        public_tri(sc, tri, h);
        h.t = tri == CRT_INVALID ? 0.0f : lv.hit_t[lv.offset[0] + i];
        return h;
      });
}

// ------------------------------------------------------------------------------------------------------------
// Progressive sessions (crtb200_accum_*, DESIGN.md 3.10.1 / 3.10.2).  The session's accumulator holds, per shard item
// (item_begin + i, so that chunks never collide), S = ((0 + c_0) + c_1) + ..., Q = ((0 + c_0 c_0) + c_1 c_1) + ... and
// sample 0's primary hit {global triangle, bits(t)}.  S and Q start at +0, so S is k_sample_acc's running sum bit for
// bit.  The unused w lanes hold the pixel's sample count n_p (S.w, as uint32 bits) and, in adaptive sessions, its active
// flag (Q.w: 1 = still sampling, 0 = stopped or not covered; plain sessions leave it 0).  A stopped pixel never starts
// again, so an active pixel has taken exactly the samples 0 .. passes - 1, and in a plain session n_p = passes.
// ------------------------------------------------------------------------------------------------------------
struct AdaptParams {
  uint32_t min_samples, max_samples;
  float abs_error, rel_error;
};

// Sample fr.sample of the pixel at shard item k, from level-0 node `node`: S += c, Q += c c, n_p += 1, and the hit at
// sample 0.  ADAPT: then the stop rule (crt_s_adapt_stop); returns true when it stops the pixel, whose flag it clears.
template <bool ADAPT>
CRT_DI bool accum_sample(const Frame &fr, const Levels &lv, uint32_t node, uint32_t k, const AdaptParams &ap,
                         float4 *__restrict__ sum, float4 *__restrict__ sumsq, uint2 *__restrict__ hit0) {
  const float4 c = lv.color[node], s = sum[k], q = sumsq[k];
  const V3 a = vadd(mk(s.x, s.y, s.z), mk(c.x, c.y, c.z));
  const V3 b = vadd(mk(q.x, q.y, q.z), mk(fmul(c.x, c.x), fmul(c.y, c.y), fmul(c.z, c.z)));
  const uint32_t n = __float_as_uint(s.w) + 1u;
  const float S[3] = {a.x, a.y, a.z}, Q[3] = {b.x, b.y, b.z};
  const bool stop = ADAPT && crt_s_adapt_stop(n, S, Q, ap.min_samples, ap.max_samples, ap.abs_error, ap.rel_error) != 0;
  sum[k] = make_float4(a.x, a.y, a.z, __uint_as_float(n));
  sumsq[k] = make_float4(b.x, b.y, b.z, (ADAPT && !stop) ? 1.f : 0.f);
  if (fr.sample == 0) hit0[k] = make_uint2(lv.hit_tri[node], __float_as_uint(lv.hit_t[node]));
  return stop;
}

// One sample pass of a plain session step, in place of k_sample_acc.  No k_store follows a step, so this counts the
// shadow rays of every pass.
__global__ void __launch_bounds__(256) k_accum_step(const DScene sc, const Frame fr, const Levels lv, float4 *__restrict__ sum,
                                                   float4 *__restrict__ sumsq, uint2 *__restrict__ hit0) {
  if (blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(&lv.stats[CRT_STAT_RAYS_SHADOW], (unsigned long long)lv.counts[CRT_MAX_LEVELS] * sc.n_lights);
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < fr.n_items0; i += gridDim.x * blockDim.x)
    accum_sample<false>(fr, lv, lv.offset[0] + i, fr.item_begin + i, AdaptParams{}, sum, sumsq, hit0);
}

// The following kernels run once over a GPU's whole shard (item_begin 0).  Frame-layout arrays (H*W*3 floats, H*W hits
// or counts) are in the primary's memory, peer-mapped on the other GPUs of a multi-GPU context, like k_store's frame.

// Read: S / float(n_p) (k_sample_acc's division), its PPMColor bytes and the kept hit into the frame, stored as k_store
// stores a frame
__global__ void __launch_bounds__(256) k_accum_read(const DScene sc, const Frame fr, const float4 *__restrict__ sum,
                                                   const uint2 *__restrict__ hit0, float *__restrict__ rgb,
                                                   uint8_t *__restrict__ rgb8, HitRec *__restrict__ hits) {
  store_items(
      sc, fr, rgb, rgb8, hits, nullptr,
      [&](uint32_t i) {
        const float4 s = sum[fr.item_begin + i];
        const float n = (float)__float_as_uint(s.w);
        return make_float4(fdiv(s.x, n), fdiv(s.y, n), fdiv(s.z, n), 0.f);
      },
      [&](uint32_t i) {
        const uint2 h = hit0[fr.item_begin + i];
        HitRec r;
        public_tri(sc, h.x, r);
        r.t = h.x == CRT_INVALID ? 0.0f : __uint_as_float(h.y);
        return r;
      });
}

// Save: the accumulator of the covered pixels into frame-layout arrays (public hit numbering, mesh = triangle = -1 for a
// miss, t bits kept either way; counts = n_p).  Any output may be null.
__global__ void __launch_bounds__(256) k_accum_save(const DScene sc, const Frame fr, const float4 *__restrict__ sum,
                                                   const float4 *__restrict__ sumsq, const uint2 *__restrict__ hit0,
                                                   float *__restrict__ sum_out, float *__restrict__ sumsq_out,
                                                   HitRec *__restrict__ hit_out, uint32_t *__restrict__ counts_out) {
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < fr.n_items0; i += gridDim.x * blockDim.x) {
    uint32_t row, col;
    if (!item_pixel(fr, sc, fr.item_begin + i, row, col)) continue;
    const uint32_t k = fr.item_begin + i;
    const size_t pix = (size_t)row * sc.width + col;
    if (sum_out) {
      const float4 s = sum[k];
      sum_out[3 * pix + 0] = s.x;
      sum_out[3 * pix + 1] = s.y;
      sum_out[3 * pix + 2] = s.z;
    }
    if (sumsq_out) {
      const float4 q = sumsq[k];
      sumsq_out[3 * pix + 0] = q.x;
      sumsq_out[3 * pix + 1] = q.y;
      sumsq_out[3 * pix + 2] = q.z;
    }
    if (hit_out) {
      const uint2 h = hit0[k];
      HitRec r;
      public_tri(sc, h.x, r);
      r.t = __uint_as_float(h.y);
      hit_out[pix] = r;
    }
    if (counts_out) counts_out[pix] = __float_as_uint(sum[k].w);
  }
}

// Load: the reverse of k_accum_save, or with sum_in == null (an adaptive begin) the counts and flags alone.  Per covered
// pixel: S, Q and the hit from the inputs; n_p from counts_in, or `passes` without it; adaptive sessions set the
// active flag iff n_p == passes and the rule does not stop the pixel at n_p.  The inputs come from a file: a hit record
// that names no triangle of the uploaded scene sets bad[0], a count above passes or 0 while passes > 0 sets bad[1].
// tot[0..2] += covered pixels, active pixels, sum of n_p.
__global__ void __launch_bounds__(256) k_accum_load(const DScene sc, const Frame fr, const float *__restrict__ sum_in,
                                                   const float *__restrict__ sumsq_in, const HitRec *__restrict__ hit_in,
                                                   const uint32_t *__restrict__ counts_in, uint32_t passes,
                                                   uint32_t n_triangles, const bool adaptive, const AdaptParams ap,
                                                   float4 *__restrict__ sum, float4 *__restrict__ sumsq,
                                                   uint2 *__restrict__ hit0, uint32_t *__restrict__ bad,
                                                   unsigned long long *__restrict__ tot) {
  uint32_t covered = 0, active = 0;
  unsigned long long samples = 0;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < fr.n_items0; i += gridDim.x * blockDim.x) {
    uint32_t row, col;
    if (!item_pixel(fr, sc, fr.item_begin + i, row, col)) continue;
    const uint32_t k = fr.item_begin + i;
    const size_t pix = (size_t)row * sc.width + col;
    float4 s = sum[k], q = sumsq[k];
    if (sum_in) {
      s = make_float4(sum_in[3 * pix + 0], sum_in[3 * pix + 1], sum_in[3 * pix + 2], 0.f);
      q = make_float4(sumsq_in[3 * pix + 0], sumsq_in[3 * pix + 1], sumsq_in[3 * pix + 2], 0.f);
      const HitRec r = hit_in[pix];
      uint32_t tri = CRT_INVALID;
      if (r.mesh >= 0) {
        const bool ok = (uint32_t)r.mesh < sc.n_meshes && r.tri >= 0 &&
                        (unsigned long long)sc.meshes[r.mesh].first_triangle + (uint32_t)r.tri < n_triangles &&
                        sc.tri_shade[sc.meshes[r.mesh].first_triangle + (uint32_t)r.tri].w == (uint32_t)r.mesh;
        if (!ok) {
          bad[0] = 1u;
          continue;
        }
        tri = sc.meshes[r.mesh].first_triangle + (uint32_t)r.tri;
      } else if (r.mesh != -1 || r.tri != -1) {
        bad[0] = 1u;
        continue;
      }
      hit0[k] = make_uint2(tri, __float_as_uint(r.t));
    }
    const uint32_t n = counts_in ? counts_in[pix] : passes;
    if (n > passes || (n == 0 && passes > 0)) {
      bad[1] = 1u;
      continue;
    }
    const float S[3] = {s.x, s.y, s.z}, Q[3] = {q.x, q.y, q.z};
    const bool act = adaptive && n == passes && !crt_s_adapt_stop(n, S, Q, ap.min_samples, ap.max_samples, ap.abs_error, ap.rel_error);
    sum[k] = make_float4(s.x, s.y, s.z, __uint_as_float(n));
    sumsq[k] = make_float4(q.x, q.y, q.z, act ? 1.f : 0.f);
    covered++;
    active += act ? 1u : 0u;
    samples += n;
  }
  covered = __reduce_add_sync(CRT_FULL_MASK, covered);
  active = __reduce_add_sync(CRT_FULL_MASK, active);
  for (int d = 16; d > 0; d >>= 1) samples += __shfl_xor_sync(CRT_FULL_MASK, samples, d);
  if (lane_id() == 0 && covered) {
    atomicAdd(&tot[0], (unsigned long long)covered);
    atomicAdd(&tot[1], (unsigned long long)active);
    atomicAdd(&tot[2], samples);
  }
}

// ------------------------------------------------------------------------------------------------------------
// Adaptive session passes (crtb200_accum_begin_adaptive, DESIGN.md 3.10.2)
// ------------------------------------------------------------------------------------------------------------
// Per pass and chunk: the shard items still sampling, into list[0 .. *n_list) (*n_list zeroed before).  One warp per
// 8x4 tile, one ballot and one atomicAdd, so a tile's active pixels stay adjacent and a level-0 warp starts coherent.
// The order of tiles in the list varies from run to run; nothing depends on it (path keys follow the ray's place in
// its tree, DESIGN.md 3.10).
__global__ void __launch_bounds__(256) k_adapt_compact(const Frame fr, const float4 *__restrict__ sumsq,
                                                      uint32_t *__restrict__ list, uint32_t *__restrict__ n_list) {
  const uint32_t lane = lane_id(), warps = gridDim.x * (blockDim.x >> 5);
  for (uint32_t t = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); 32u * t < fr.n_items0; t += warps) {
    const uint32_t i = 32u * t + lane;
    const bool active = i < fr.n_items0 && sumsq[fr.item_begin + i].w != 0.f;
    const uint32_t ball = __ballot_sync(CRT_FULL_MASK, active);
    if (!ball) continue;
    uint32_t base = 0;
    if (lane == 0) base = atomicAdd(n_list, (uint32_t)__popc(ball));
    base = __shfl_sync(CRT_FULL_MASK, base, 0);
    if (active) list[base + __popc(ball & lanemask_lt())] = fr.item_begin + i;
  }
}

// One adaptive pass, in place of k_accum_step: accum_sample with the stop rule at shard item list[j].  Counts the
// pass's shadow rays as k_accum_step does, its pixel-samples into stats[CRT_STAT_PX_SAMPLES] and the pixels it stopped into stats[CRT_STAT_STOPPED].
__global__ void __launch_bounds__(256) k_adapt_step(const DScene sc, const Frame fr, const Levels lv, const AdaptParams ap,
                                                   float4 *__restrict__ sum, float4 *__restrict__ sumsq,
                                                   uint2 *__restrict__ hit0) {
  const uint32_t n_act = *fr.n_list;
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    atomicAdd(&lv.stats[CRT_STAT_RAYS_SHADOW], (unsigned long long)lv.counts[CRT_MAX_LEVELS] * sc.n_lights);
    atomicAdd(&lv.stats[CRT_STAT_PX_SAMPLES], (unsigned long long)n_act);
  }
  const uint32_t stride = gridDim.x * blockDim.x;
  for (uint32_t base = blockIdx.x * blockDim.x + (threadIdx.x & ~31u); base < n_act; base += stride) {
    const uint32_t j = base + lane_id();
    const bool stop = j < n_act && accum_sample<true>(fr, lv, lv.offset[0] + j, fr.list[j], ap, sum, sumsq, hit0);
    const uint32_t stopped = __popc(__ballot_sync(CRT_FULL_MASK, stop));
    if (lane_id() == 0 && stopped) atomicAdd(&lv.stats[CRT_STAT_STOPPED], (unsigned long long)stopped);
  }
}

// Scatter gathered shard slabs (shard-major, item order) into a full frame: the rank-0 side of the NCCL gather.
// A warp moves one 8x4 tile: 384 contiguous slab bytes in, four 96-byte frame rows out (16-byte accesses both ways when
// the tile is whole and everything is aligned, like k_store).
__global__ void __launch_bounds__(256) k_assemble(const DScene sc, Frame fr, const float *__restrict__ slabs,
                                                 uint32_t items_per_shard, uint32_t shard_count,
                                                 float *__restrict__ rgb, uint8_t *__restrict__ rgb8) {
  __shared__ __align__(16) float s_f[8][96];
  __shared__ __align__(8) uint8_t s_b[8][96];
  const uint32_t lane = lane_id(), w = threadIdx.x >> 5;
  const bool aligned = (sc.width & 7u) == 0u && (items_per_shard & 31u) == 0u && (reinterpret_cast<uintptr_t>(rgb) & 15u) == 0u &&
                       (reinterpret_cast<uintptr_t>(rgb8) & 7u) == 0u && (reinterpret_cast<uintptr_t>(slabs) & 15u) == 0u;
  const unsigned long long total = (unsigned long long)items_per_shard * shard_count;
  for (unsigned long long base = blockIdx.x * (unsigned long long)blockDim.x + (threadIdx.x & ~31u); base < total;
       base += (unsigned long long)gridDim.x * blockDim.x) {
    const unsigned long long g = base + lane;
    const uint32_t shard = (uint32_t)(g / items_per_shard), i = (uint32_t)(g % items_per_shard);
    fr.shard_index = shard;
    fr.shard_count = shard_count;
    uint32_t row = 0, col = 0;
    const bool valid = g < total && item_pixel(fr, sc, i, row, col);
    const size_t pix = (size_t)row * sc.width + col;
    if (aligned && __all_sync(CRT_FULL_MASK, valid)) {  // (aligned => a warp's 32 items are one tile of one shard)
      const size_t p0 = (size_t)__shfl_sync(CRT_FULL_MASK, (unsigned long long)pix, 0);
      if (lane < 24u) *reinterpret_cast<float4 *>(&s_f[w][4 * lane]) = *reinterpret_cast<const float4 *>(slabs + 3 * base + 4 * lane);
      __syncwarp();
      if (rgb && lane < 24u)
        *reinterpret_cast<float4 *>(rgb + 3 * (p0 + (size_t)(lane / 6u) * sc.width) + 4 * (lane % 6u)) =
            *reinterpret_cast<const float4 *>(&s_f[w][4 * lane]);
      if (rgb8) {
        s_b[w][3 * lane + 0] = quantize(s_f[w][3 * lane + 0]);
        s_b[w][3 * lane + 1] = quantize(s_f[w][3 * lane + 1]);
        s_b[w][3 * lane + 2] = quantize(s_f[w][3 * lane + 2]);
        __syncwarp();
        if (lane < 12u)
          *reinterpret_cast<uint2 *>(rgb8 + 3 * (p0 + (size_t)(lane / 3u) * sc.width) + 8 * (lane % 3u)) =
              *reinterpret_cast<const uint2 *>(&s_b[w][8 * lane]);
      }
      __syncwarp();
      continue;
    }
    if (!valid) continue;
    const float *s = slabs + 3 * g;
    if (rgb) {
      rgb[3 * pix + 0] = s[0];
      rgb[3 * pix + 1] = s[1];
      rgb[3 * pix + 2] = s[2];
    }
    if (rgb8) {
      rgb8[3 * pix + 0] = quantize(s[0]);
      rgb8[3 * pix + 1] = quantize(s[1]);
      rgb8[3 * pix + 2] = quantize(s[2]);
    }
  }
}

// Test hook: crt_powf5 on the device, for the bit-equality test against the host libm's powf(x, 5).
__global__ void __launch_bounds__(256) k_powf5(const float *__restrict__ x, uint32_t n, float *__restrict__ out) {
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) out[i] = crt_powf5(x[i]);
}

// K1 standalone: RayTracer::getRay + shootRay's re-normalisation into a caller's array (crtb200_generate_rays_device).
__global__ void __launch_bounds__(256) k_generate_rays(const DScene sc, const DCamera cam, float *__restrict__ rays) {
  const uint32_t n = sc.width * sc.height;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    V3 o, d;
    primary_ray(cam, sc.width, sc.height, i / sc.width, i % sc.width, o, d);
    float *r = rays + 6 * (size_t)i;
    r[0] = o.x;
    r[1] = o.y;
    r[2] = o.z;
    r[3] = d.x;
    r[4] = d.y;
    r[5] = d.z;
  }
}

// ------------------------------------------------------------------------------------------------------------
// Caller-supplied ray batches (crtb200_trace_rays_device, DESIGN.md 3.12): RayTracer::trace (RayTracer.cpp:453-458) and
// the non-GI RayTracer::hasIntersection (RayTracer.cpp:507-518) for rays the caller holds in device memory, walked by
// k_closest / k_shadow and handed off to k_coop with the sources QueryClosest / QueryShadow.  Work item i = ray i of the
// batch = record id i; its answer goes straight to the caller's arrays.
// ------------------------------------------------------------------------------------------------------------
struct QueryBatch {
  const float *rays;          // n x 6: origin xyz, direction xyz
  const float *max_distance;  // n, shadow queries
  HitRec *hits;               // n, closest-hit queries (public numbering; miss: -1, -1, t = 0)
  uint8_t *occluded;          // n, shadow queries
  uint32_t n;
};

// Ray i of a batch: three 8-byte loads when the array is 8-byte aligned (a ray is 24 bytes)
CRT_DI void query_ray(const float *rays, const uint32_t i, Ray &ray) {
  const float *r = rays + 6 * (size_t)i;
  if ((reinterpret_cast<uintptr_t>(rays) & 7u) == 0u) {
    const float2 a = *reinterpret_cast<const float2 *>(r), b = *reinterpret_cast<const float2 *>(r + 2),
                 c = *reinterpret_cast<const float2 *>(r + 4);
    ray.o = mk(a.x, a.y, b.x);
    ray.d = mk(b.y, c.x, c.y);
  } else {
    ray.o = mk(r[0], r[1], r[2]);
    ray.d = mk(r[3], r[4], r[5]);
  }
}

// The culling bound of a caller's shadow ray.  shadow_limit assumes |d| = 1 within 2 ulp; a caller's direction may
// have any length, so the *beyond* skip is applied only when the computed |d| is within 8 ulp of 1 (then the true |d| is
// within 11 ulp of 1, far inside shadow_limit's 1e-4 relative slack); other rays keep *behind* alone (DESIGN.md 3.12).
CRT_DI float query_shadow_limit(const Ray &ray, const float dist) {
  return fabsf(fsub(vlen(ray.d), 1.0f)) <= 8.0f * CRT_FLT_EPSILON ? shadow_limit(ray, dist) : CRT_INF;
}

CRT_DI void query_store_hit(const DScene &sc, HitRec *hits, const uint32_t i, const uint32_t tri, const float t) {
  HitRec h;
  public_tri(sc, tri, h);
  h.t = tri == CRT_INVALID ? 0.0f : t;
  hits[i] = h;
}

// Closest hit of ray i (the walk's PRIMARY: CRTB200_RAY_PRIMARY batches).  Limits as the frame's: culling in parameter
// space holds for any direction length (DESIGN.md 3.12).
struct QueryClosest : QueryBatch {
  static constexpr bool SHADOW = false;
  CRT_DI uint32_t level(const uint32_t) const { return 0u; }
  template <bool>
  CRT_DI uint32_t items(const Frame &, const Levels &, const uint32_t) const { return n; }
  CRT_DI uint32_t base(const Levels &, const uint32_t) const { return 0u; }
  template <bool>
  CRT_DI bool take(const DScene &, const Frame &, const Levels &, const uint32_t, const uint32_t i, Ray &ray) const {
    query_ray(rays, i, ray);
    return true;
  }
  CRT_DI void ray(const DScene &, const Frame &, const Levels &, const uint32_t id, Ray &ray, float &) const { query_ray(rays, id, ray); }
  CRT_DI void answer(const DScene &sc, const Levels &, const uint32_t id, const Closest &cl) const {
    query_store_hit(sc, hits, id, cl.best_tri, cl.best_t);
  }
};

// Any hit of ray i within max_distance[i]: occluded iff some candidate has |P - o| <= max_distance (refractive meshes
// skipped, AccelerationStructure.cpp:67-74).  A query has no light term, so no walk is skipped for a zero term.
struct QueryShadow : QueryBatch {
  static constexpr bool SHADOW = true;
  CRT_DI uint32_t level(const uint32_t) const { return 0u; }
  CRT_DI uint32_t base(const Levels &) const { return 0u; }
  CRT_DI uint32_t items(const DScene &, const uint32_t) const { return n; }
  template <bool>
  CRT_DI bool take(const DScene &, const Frame &, const Levels &, const uint32_t, const uint32_t i, Ray &ray, float &dist,
                   uint32_t &id, uint32_t &) const {
    query_ray(rays, i, ray);
    dist = max_distance[i];
    id = i;
    return true;
  }
  CRT_DI void ray(const DScene &, const Frame &, const Levels &, const uint32_t id, Ray &ray, float &dist) const {
    query_ray(rays, id, ray);
    dist = max_distance[id];
  }
  CRT_DI float limit(const Ray &ray, const float dist) const { return query_shadow_limit(ray, dist); }
  CRT_DI void answer(const Levels &, const uint32_t id, const bool occ) const { occluded[id] = occ ? 1 : 0; }
  CRT_DI void declined(const Levels &, const uint32_t) const {}
};

// ------------------------------------------------------------------------------------------------------------
// Caller-supplied rays shaded through the frame pipeline (crtb200_shade_rays_device, DESIGN.md 3.13): RayTracer::shootRay
// (RayTracer.cpp:419-451) for a batch of rays.  Level 0 of a chunk is ray item_begin + i of the batch instead of a
// pixel: k_closest, k_coop, k_shade and k_resolve read it through the source ShadeRays; every later level, the shadow
// pass and k_accumulate are the frame's.  k_store_rays writes colour i and hit i.
// ------------------------------------------------------------------------------------------------------------
// Ray `item` of the range with shootRay's normalisation of the direction (RayTracer.cpp:420), applied once: the walk,
// its hand-off and k_shade read the same bits
CRT_DI void shade_ray(const float *rays, const uint32_t item, V3 &o, V3 &d) {
  Ray r;
  query_ray(rays, item, r);
  o = r.o;
  d = vnorm(r.d);
}

// This GPU's range of the batch; record id = level-0 queue node, answered into the frame's hit records.  Its
// launches are level 0 only.
struct ShadeRays {
  const float *rays;     // n x 6 (origin xyz, direction xyz)
  float *rgb;            // n x 3
  HitRec *hits;          // n, or null
  uint32_t first_index;  // GI: pixel index p of ray 0 of the range
  uint32_t stat;         // CRT_STAT_RAYS_* slot of the batch's ray type

  static constexpr bool SHADOW = false;
  CRT_DI uint32_t level(const uint32_t) const { return 0u; }
  template <bool>
  CRT_DI uint32_t items(const Frame &fr, const Levels &, const uint32_t) const { return fr.n_items0; }
  CRT_DI uint32_t base(const Levels &lv, const uint32_t level) const { return lv.offset[level]; }
  template <bool>
  CRT_DI bool take(const DScene &, const Frame &fr, const Levels &, const uint32_t, const uint32_t i, Ray &ray) const {
    shade_ray(rays, fr.item_begin + i, ray.o, ray.d);
    return true;
  }
  CRT_DI void ray(const DScene &, const Frame &fr, const Levels &lv, const uint32_t id, Ray &ray, float &) const {
    shade_ray(rays, fr.item_begin + (id - lv.offset[0]), ray.o, ray.d);
  }
  CRT_DI void answer(const DScene &, const Levels &lv, const uint32_t id, const Closest &cl) const {
    lv.hit_tri[id] = cl.best_tri;
    lv.hit_t[id] = cl.best_t;
  }
  template <bool GI>
  CRT_DI bool valid(const DScene &, const Frame &, const uint32_t) const { return true; }
  // GI: p = first_index + item, s = fr.sample, root path key = R(p, s, 0, 0).z (the word jittered_primary_ray returns)
  template <bool GI>
  CRT_DI void level0(const DScene &, const Frame &fr, const uint32_t i, bool &valid, V3 &o, V3 &d, uint32_t &key,
                     uint32_t &pix, uint32_t &n) const {
    shade_ray(rays, fr.item_begin + i, o, d);
    if (GI) {
      pix = first_index + fr.item_begin + i;
      key = crt_s_philox(pix, fr.sample, 0u, 0u, fr.seed, fr.frame_index).z;
    }
    valid = true;
    n++;
  }
  CRT_DI uint32_t ray_stat() const { return stat; }
};

// Colour i and hit i of the chunk's rays, in place of k_store: a warp's 32 colours leave as 24 16-byte stores when rgb is
// 16-byte aligned (chunks start at multiples of 32 rays, so every full warp's 384 bytes are then aligned too).  Counts
// the chunk's shadow rays as k_store does.
__global__ void __launch_bounds__(256) k_store_rays(const DScene sc, const Frame fr, const Levels lv, const ShadeRays sr) {
  __shared__ __align__(16) float s_f[8][96];
  if (blockIdx.x == 0 && threadIdx.x == 0)
    atomicAdd(&lv.stats[CRT_STAT_RAYS_SHADOW], (unsigned long long)lv.counts[CRT_MAX_LEVELS] * sc.n_lights);
  const uint32_t lane = lane_id(), w = threadIdx.x >> 5;
  const bool aligned = (reinterpret_cast<uintptr_t>(sr.rgb) & 15u) == 0u;
  for (uint32_t base = blockIdx.x * blockDim.x + (threadIdx.x & ~31u); base < fr.n_items0; base += gridDim.x * blockDim.x) {
    const uint32_t i = base + lane, k = fr.item_begin + i;
    const bool valid = i < fr.n_items0;
    const float4 c = valid ? lv.color[lv.offset[0] + i] : make_float4(0.f, 0.f, 0.f, 0.f);
    if (aligned && base + 32u <= fr.n_items0) {
      s_f[w][3 * lane + 0] = c.x;
      s_f[w][3 * lane + 1] = c.y;
      s_f[w][3 * lane + 2] = c.z;
      __syncwarp();
      if (lane < 24u)
        *reinterpret_cast<float4 *>(sr.rgb + 3 * (size_t)(fr.item_begin + base) + 4 * lane) = *reinterpret_cast<const float4 *>(&s_f[w][4 * lane]);
      __syncwarp();
    } else if (valid) {
      sr.rgb[3 * (size_t)k + 0] = c.x;
      sr.rgb[3 * (size_t)k + 1] = c.y;
      sr.rgb[3 * (size_t)k + 2] = c.z;
    }
    if (sr.hits && valid) {
      const uint32_t tri = lv.hit_tri[lv.offset[0] + i];
      HitRec h;
      public_tri(sc, tri, h);
      h.t = tri == CRT_INVALID ? 0.0f : lv.hit_t[lv.offset[0] + i];
      sr.hits[k] = h;
    }
  }
}

}  // namespace crtd
