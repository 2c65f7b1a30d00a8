// crt_build.cuh -- device KD build of crtb200_upload_geometry (DESIGN.md 3.11).
//
// Builds every mesh's TriangleKDTree(mesh, 25, 8) and the ObjectKDTree(scene, 25, 4) (AccelerationStructure.cpp:12-50)
// node for node as the host builder csrc/frontend/crt_kdtree.cpp does, level by level over the frontier of all trees at
// once, and writes the device layout crtb200_upload_scene writes from those trees (relayout_tree, mesh_cull_margin and
// the nesting rule of upload_one in crtb200_core.cu).  Every position comes from a scan, never from the order in which
// atomics arrive; the only atomics are order-free maxima / minima over (value, position) keys.
//
// Elements ("items"): the triangles of mesh 0, then of mesh 1, ... (item = item_base[m] + mesh-local index), followed by
// one item per mesh (n_items + m) whose box is that mesh's root box: the elements of the top-level tree (tree n_meshes).
// A level's listing holds one (element, node) pair per element of each node, in node order, elements ascending.
#pragma once
#include "../../include/crtb200.h"
#include "crt_device.cuh"

namespace crtd {

#define CRT_BUILD_MAX_DEPTH 25u  // TriangleKDTree(mesh, 25, 8), ObjectKDTree(scene, 25, 4): AccelerationStructure.h:10-11
#define CRT_BUILD_FLT_MAX 3.40282346638528859812e+38f

struct BBox {
  float mn[3], mx[3];
};
// one node of a level: its box, tree, and its elements' segment [seg, seg + cnt) of the level's listing
struct BNode {
  float mn[3], mx[3];
  uint32_t tree, seg, cnt, pad;
};

// std::min / std::max as written (BoundingBox.h:31-32): a NaN coordinate never enters a box
CRT_DI void bbox_grow(BBox &b, float x, float y, float z) {
  const float v[3] = {x, y, z};
#pragma unroll
  for (int i = 0; i < 3; i++) {
    b.mn[i] = (v[i] < b.mn[i]) ? v[i] : b.mn[i];
    b.mx[i] = (b.mx[i] < v[i]) ? v[i] : b.mx[i];
  }
}
CRT_DI BBox bbox_empty() {
  BBox b;
#pragma unroll
  for (int i = 0; i < 3; i++) {
    b.mn[i] = CRT_BUILD_FLT_MAX;
    b.mx[i] = -CRT_BUILD_FLT_MAX;
  }
  return b;
}
// KDTree.cpp:13-16
CRT_DI bool build_is_leaf(const BNode &n, uint32_t level, uint32_t n_meshes) {
  return level >= CRT_BUILD_MAX_DEPTH || n.cnt <= (n.tree < n_meshes ? 8u : 4u);
}
// BoundingBox::split, BoundingBox.h:60-69: child 0 takes mx[axis] = plane, child 1 mn[axis] = plane
// (the axis is selected, not used as an index: the node stays in registers)
CRT_DI float build_axis(const float *v, uint32_t axis) { return axis == 0 ? v[0] : (axis == 1 ? v[1] : v[2]); }
CRT_DI float build_plane(const BNode &n, uint32_t axis) {
  const float lo = build_axis(n.mn, axis), middle = fdiv(fsub(build_axis(n.mx, axis), lo), 2.0f);
  return fadd(lo, middle);
}
// BoundingBox::intersects, BoundingBox.h:75-83: inclusive on both sides
CRT_DI bool build_overlaps(const float *amn, const float *amx, const BBox &b) {
#pragma unroll
  for (int i = 0; i < 3; i++)
    if (amn[i] > b.mx[i] || amx[i] < b.mn[i]) return false;
  return true;
}
// mesh of an item: the last m with item_base[m] <= item (empty meshes share their successor's base)
CRT_DI uint32_t build_item_mesh(const uint32_t *item_base, uint32_t n_meshes, uint32_t item) {
  uint32_t lo = 0, hi = n_meshes;  // answer in [lo, hi)
  while (hi - lo > 1) {
    const uint32_t mid = (lo + hi) >> 1;
    if (item_base[mid] <= item) lo = mid; else hi = mid;
  }
  return lo;
}
// binary32 -> u32 key ordered as the float compares; -0.0 and +0.0 get the same key (they compare equal)
CRT_DI uint32_t build_order_key(float v) {
  const uint32_t u = __float_as_uint(v == 0.0f ? 0.0f : v);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
// Lanes of a warp with the same key fold their values, and the lowest of them does one atomicMax.  Every lane of the
// warp must call it (out-of-range lanes with key CRT_INVALID).
CRT_DI void build_warp_max(unsigned long long *slots, uint32_t key, uint32_t field, unsigned long long v) {
  const uint32_t peers = __match_any_sync(0xffffffffu, key);
  unsigned long long best = v;
#pragma unroll 1
  for (int src = 0; src < 32; src++) {
    const unsigned long long o = __shfl_sync(0xffffffffu, v, src);
    if ((peers >> src) & 1u) best = o > best ? o : best;
  }
  if (key != CRT_INVALID && (threadIdx.x & 31u) == (uint32_t)(__ffs(peers) - 1)) atomicMax(slots + 4ull * key + field, best);
}
CRT_DI void build_warp_min(unsigned long long *slots, uint32_t key, uint32_t field, unsigned long long v) {
  const uint32_t peers = __match_any_sync(0xffffffffu, key);
  unsigned long long best = v;
#pragma unroll 1
  for (int src = 0; src < 32; src++) {
    const unsigned long long o = __shfl_sync(0xffffffffu, v, src);
    if ((peers >> src) & 1u) best = o < best ? o : best;
  }
  if (key != CRT_INVALID && (threadIdx.x & 31u) == (uint32_t)(__ffs(peers) - 1)) atomicMin(slots + 6ull * key + field, best);
}

// ---- boxes -------------------------------------------------------------------------------------------------------
// BoundingBox(const Triangle&), BoundingBox.h:50-58: vertices 0, 1, 2.  Then the mesh root boxes (BoundingBox.h:26-34,
// the vertices of the mesh's triangles in triangle order) as an order-free reduction: per mesh and bound, the smallest
// (value key, mesh-local item) pair among the triangle boxes' bounds.  The serial fold keeps the FIRST of equal values,
// so the smallest position among equal keys is its result bit for bit; a bound that never beats the initial FLT_MAX
// (resp. -FLT_MAX) is no candidate.
__global__ void __launch_bounds__(256) k_build_item_boxes(const float4 *__restrict__ geom, const uint32_t *__restrict__ item_base,
                                                          const uint32_t *__restrict__ mesh_tri, uint32_t n_meshes, uint32_t n_items,
                                                          BBox *__restrict__ ebox, unsigned long long *__restrict__ mslots) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  uint32_t key = CRT_INVALID;
  unsigned long long k6[6];
#pragma unroll
  for (int f = 0; f < 6; f++) k6[f] = ~0ull;
  if (i < n_items) {
    const uint32_t m = build_item_mesh(item_base, n_meshes, i);
    const uint32_t local = i - item_base[m];
    const size_t t = (size_t)mesh_tri[m] + local;
    BBox b = bbox_empty();
#pragma unroll
    for (int k = 0; k < 3; k++) {
      const float4 p = geom[3 * t + k];
      bbox_grow(b, p.x, p.y, p.z);
    }
    ebox[i] = b;
    key = m;
#pragma unroll
    for (int a = 0; a < 3; a++) {
      if (b.mn[a] < CRT_BUILD_FLT_MAX) k6[a] = ((unsigned long long)build_order_key(b.mn[a]) << 32) | local;
      if (-CRT_BUILD_FLT_MAX < b.mx[a]) k6[3 + a] = ((unsigned long long)~build_order_key(b.mx[a]) << 32) | local;
    }
  }
#pragma unroll
  for (int f = 0; f < 6; f++) build_warp_min(mslots, key, f, k6[f]);
}

// Per mesh: its root box from the reduction's positions, written as the top-level tree's element n_items + m and as the
// root of mesh tree m (node m of level 0).  k_build_scene_box then folds the scene box (BoundingBox(scene),
// BoundingBox.h:36-48) over the mesh boxes in mesh order -- the serial fold over all triangles in order, regrouped: the
// first of equal values still wins -- and writes the top-level root (node n_meshes).
__global__ void __launch_bounds__(256) k_build_roots(const uint32_t *__restrict__ item_base, uint32_t n_meshes, uint32_t n_items,
                                                     BBox *__restrict__ ebox, const unsigned long long *__restrict__ mslots,
                                                     BNode *__restrict__ roots) {
  const uint32_t m = blockIdx.x * blockDim.x + threadIdx.x;
  if (m < n_meshes) {
    BBox b = bbox_empty();
#pragma unroll
    for (int f = 0; f < 6; f++) {
      const unsigned long long s = mslots[6ull * m + f];
      if (s == ~0ull) continue;
      const BBox &e = ebox[item_base[m] + (uint32_t)s];
      if (f < 3) b.mn[f] = e.mn[f]; else b.mx[f - 3] = e.mx[f - 3];
    }
    ebox[n_items + m] = b;
    BNode r;
    for (int a = 0; a < 3; a++) {
      r.mn[a] = b.mn[a];
      r.mx[a] = b.mx[a];
    }
    r.tree = m;
    r.seg = item_base[m];
    r.cnt = item_base[m + 1] - item_base[m];
    r.pad = 0;
    roots[m] = r;
  }
}
__global__ void k_build_scene_box(uint32_t n_meshes, uint32_t n_items, const BBox *__restrict__ ebox, BNode *__restrict__ roots) {
  BBox s = bbox_empty();
  for (uint32_t m = 0; m < n_meshes; m++) {
    const BBox &b = ebox[n_items + m];
    for (int a = 0; a < 3; a++) {
      s.mn[a] = (b.mn[a] < s.mn[a]) ? b.mn[a] : s.mn[a];
      s.mx[a] = (s.mx[a] < b.mx[a]) ? b.mx[a] : s.mx[a];
    }
  }
  BNode r;
  for (int a = 0; a < 3; a++) {
    r.mn[a] = s.mn[a];
    r.mx[a] = s.mx[a];
  }
  r.tree = n_meshes;
  r.seg = n_items;
  r.cnt = n_meshes;
  r.pad = 0;
  roots[n_meshes] = r;
}
__global__ void __launch_bounds__(256) k_build_listing0(const uint32_t *__restrict__ item_base, uint32_t n_meshes, uint32_t n_items,
                                                        uint32_t *__restrict__ lelem, uint32_t *__restrict__ lnode) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_items + n_meshes) return;
  lelem[i] = i;
  lnode[i] = i < n_items ? build_item_mesh(item_base, n_meshes, i) : n_meshes;
}

// ---- one level -----------------------------------------------------------------------------------------------------
// Per listing: which children of its (inner) node the element overlaps; thread nL writes the zero sentinel so that the
// exclusive scan's last entry is the total.
__global__ void __launch_bounds__(256) k_build_flags(const BNode *__restrict__ nodes, const uint32_t *__restrict__ lelem,
                                                     const uint32_t *__restrict__ lnode, uint32_t nL, uint32_t level,
                                                     uint32_t n_meshes, const BBox *__restrict__ ebox, uint2 *__restrict__ flags) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i > nL) return;
  uint2 f = make_uint2(0u, 0u);
  if (i < nL) {
    const BNode n = nodes[lnode[i]];
    if (!build_is_leaf(n, level, n_meshes)) {
      const uint32_t axis = level % 3u;
      const float plane = build_plane(n, axis);
      const BBox e = ebox[lelem[i]];
      float c0mx[3], c1mn[3];
#pragma unroll
      for (uint32_t a = 0; a < 3; a++) {
        c0mx[a] = a == axis ? plane : n.mx[a];
        c1mn[a] = a == axis ? plane : n.mn[a];
      }
      f.x = build_overlaps(n.mn, c0mx, e) ? 1u : 0u;
      f.y = build_overlaps(c1mn, n.mx, e) ? 1u : 0u;
    }
  }
  flags[i] = f;
}

// Per node, from the listing scan S: {children, child listings, leaf references, 0}; thread nF writes the sentinel.
__global__ void __launch_bounds__(256) k_build_counts(const BNode *__restrict__ nodes, uint32_t nF, uint32_t level, uint32_t n_meshes,
                                                      const uint2 *__restrict__ S, uint4 *__restrict__ nc) {
  const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j > nF) return;
  uint4 r = make_uint4(0u, 0u, 0u, 0u);
  if (j < nF) {
    const BNode n = nodes[j];
    if (build_is_leaf(n, level, n_meshes)) {
      r.z = n.cnt;
    } else {
      const uint32_t c0 = S[n.seg + n.cnt].x - S[n.seg].x, c1 = S[n.seg + n.cnt].y - S[n.seg].y;
      r.x = (c0 ? 1u : 0u) + (c1 ? 1u : 0u);
      r.y = c0 + c1;
    }
  }
  nc[j] = r;
}

// Per node: the next level's children (child 0 first, empty children not created), child indices (into the next
// level), and a leaf's reference count and offset into this level's leaf buffer.
__global__ void __launch_bounds__(256) k_build_emit(const BNode *__restrict__ nodes, uint32_t nF, uint32_t level, uint32_t n_meshes,
                                                    const uint2 *__restrict__ S, const uint4 *__restrict__ NS, BNode *__restrict__ next,
                                                    uint32_t *__restrict__ child, uint32_t *__restrict__ leaf_cnt,
                                                    uint32_t *__restrict__ leaf_off) {
  const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= nF) return;
  const BNode n = nodes[j];
  uint32_t ch0 = CRT_INVALID, ch1 = CRT_INVALID;
  if (build_is_leaf(n, level, n_meshes)) {
    leaf_cnt[j] = n.cnt;
    leaf_off[j] = NS[j].z;
  } else {
    const uint32_t axis = level % 3u;
    const float plane = build_plane(n, axis);
    const uint32_t c0 = S[n.seg + n.cnt].x - S[n.seg].x, c1 = S[n.seg + n.cnt].y - S[n.seg].y;
    uint32_t pos = NS[j].x;
    BNode c = n;
    if (c0) {
#pragma unroll
      for (uint32_t a = 0; a < 3; a++) c.mx[a] = a == axis ? plane : n.mx[a];
      c.seg = NS[j].y;
      c.cnt = c0;
      next[pos] = c;
      ch0 = pos++;
    }
    if (c1) {
      c = n;
#pragma unroll
      for (uint32_t a = 0; a < 3; a++) c.mn[a] = a == axis ? plane : n.mn[a];
      c.seg = NS[j].y + c0;
      c.cnt = c1;
      next[pos] = c;
      ch1 = pos;
    }
    leaf_cnt[j] = 0;
    leaf_off[j] = 0;
  }
  child[2 * j] = ch0;
  child[2 * j + 1] = ch1;
}

// Per listing: stable scatter into the next level's listing (or into this level's leaf buffer); the overlap flags are
// the scan's differences.
__global__ void __launch_bounds__(256) k_build_scatter(const BNode *__restrict__ nodes, const uint32_t *__restrict__ lelem,
                                                       const uint32_t *__restrict__ lnode, uint32_t nL, uint32_t level, uint32_t n_meshes,
                                                       const uint2 *__restrict__ S, const uint4 *__restrict__ NS,
                                                       uint32_t *__restrict__ next_elem, uint32_t *__restrict__ next_node,
                                                       uint32_t *__restrict__ leafbuf) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nL) return;
  const uint32_t j = lnode[i], e = lelem[i];
  const BNode n = nodes[j];
  if (build_is_leaf(n, level, n_meshes)) {
    leafbuf[NS[j].z + (i - n.seg)] = e;
    return;
  }
  const uint2 s0 = S[n.seg], si = S[i], si1 = S[i + 1];
  const uint32_t c0 = S[n.seg + n.cnt].x - s0.x;
  if (si1.x != si.x) {
    const uint32_t p = NS[j].y + (si.x - s0.x);
    next_elem[p] = e;
    next_node[p] = NS[j].x;
  }
  if (si1.y != si.y) {
    const uint32_t p = NS[j].y + c0 + (si.y - s0.y);
    next_elem[p] = e;
    next_node[p] = NS[j].x + (c0 ? 1u : 0u);
  }
}

// ---- numbering -----------------------------------------------------------------------------------------------------
// Bottom-up: subtree node and reference counts; and upload_one's nesting rule for the mesh trees (every box has
// min <= max, every child box lies inside its parent's): a failing node clears *nested.
CRT_DI bool build_box_nested(const BNode &p, const BNode &c) {
  for (int k = 0; k < 3; k++)
    if (!(c.mn[k] >= p.mn[k]) || !(c.mx[k] <= p.mx[k]) || !(c.mn[k] <= c.mx[k])) return false;
  return true;
}
__global__ void __launch_bounds__(256) k_build_up(const BNode *__restrict__ nodes, uint32_t nF, uint32_t n_meshes,
                                                  const uint32_t *__restrict__ child, const uint32_t *__restrict__ leaf_cnt,
                                                  uint32_t *__restrict__ size, uint32_t *__restrict__ rsize,
                                                  const BNode *__restrict__ next, const uint32_t *__restrict__ next_size,
                                                  const uint32_t *__restrict__ next_rsize, uint32_t *__restrict__ nested) {
  const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= nF) return;
  const BNode n = nodes[j];
  uint32_t s = 1, r = leaf_cnt[j];
  bool ok = true;
  for (int k = 0; k < 3; k++)
    if (!(n.mn[k] <= n.mx[k])) ok = false;
  for (int side = 0; side < 2; side++) {
    const uint32_t c = child[2 * j + side];
    if (c == CRT_INVALID) continue;
    s += next_size[c];
    r += next_rsize[c];
    if (!build_box_nested(n, next[c])) ok = false;
  }
  size[j] = s;
  rsize[j] = r;
  if (!ok && n.tree < n_meshes) atomicAnd(nested, 0u);
}
// Top-down: the reference's pre-order (child0 = self + 1, child1 = self + 1 + size(child0)), the visiting order
// (child1 = self + 1, child0 = self + 1 + size(child1)) and the first leaf reference of each subtree, within its tree.
__global__ void __launch_bounds__(256) k_build_down(uint32_t nF, const uint32_t *__restrict__ child, const uint32_t *__restrict__ pre,
                                                    const uint32_t *__restrict__ vis, const uint32_t *__restrict__ ref,
                                                    const uint32_t *__restrict__ next_size, const uint32_t *__restrict__ next_rsize,
                                                    uint32_t *__restrict__ next_pre, uint32_t *__restrict__ next_vis,
                                                    uint32_t *__restrict__ next_ref) {
  const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= nF) return;
  const uint32_t c0 = child[2 * j], c1 = child[2 * j + 1];
  const uint32_t s0 = c0 != CRT_INVALID ? next_size[c0] : 0u, s1 = c1 != CRT_INVALID ? next_size[c1] : 0u;
  if (c0 != CRT_INVALID) {
    next_pre[c0] = pre[j] + 1;
    next_vis[c0] = vis[j] + 1 + s1;
    next_ref[c0] = ref[j];
  }
  if (c1 != CRT_INVALID) {
    next_pre[c1] = pre[j] + 1 + s0;
    next_vis[c1] = vis[j] + 1;
    next_ref[c1] = ref[j] + (c0 != CRT_INVALID ? next_rsize[c0] : 0u);
  }
}

// ---- output --------------------------------------------------------------------------------------------------------
// The culling margin's inputs (mesh_cull_margin in crtb200_core.cu), in double, with std::min / std::max as the selects
// they compile to, so that a NaN operand is treated per position as on the host; every per-mesh maximum starts at +0.0
// and only a strictly larger value replaces it, so the maxima are order-free and kept as the bits of non-negative
// doubles.  Slots per mesh: 0 overhang, 1 slop, 2 absmax, 3 "a normal is not its triangle's" (then +inf).
CRT_DI double smin(double a, double b) { return (b < a) ? b : a; }
CRT_DI double smax(double a, double b) { return (a < b) ? b : a; }

// Per node of a level: its record in the visiting-order array and in the reference numbering (kept for the read-back
// when kd != nullptr), its leaf references, and the overhang / absmax terms of mesh-tree nodes.
__global__ void __launch_bounds__(256) k_build_write(const BNode *__restrict__ nodes, uint32_t nF, uint32_t n_meshes, uint32_t n_items,
                                                     const uint32_t *__restrict__ child, const uint32_t *__restrict__ leaf_cnt,
                                                     const uint32_t *__restrict__ leaf_off, const uint32_t *__restrict__ leafbuf,
                                                     const uint32_t *__restrict__ size, const uint32_t *__restrict__ pre,
                                                     const uint32_t *__restrict__ vis, const uint32_t *__restrict__ ref,
                                                     const uint32_t *__restrict__ next_pre, const uint32_t *__restrict__ next_vis,
                                                     const uint32_t *__restrict__ node_base, const uint32_t *__restrict__ ref_base,
                                                     const uint32_t *__restrict__ item_base, const uint32_t *__restrict__ mesh_tri,
                                                     const float4 *__restrict__ geom, float4 *__restrict__ out_nodes,
                                                     uint32_t *__restrict__ out_refs, uint32_t *__restrict__ out_top_refs,
                                                     crtb200_kdnode *__restrict__ kd, uint32_t *__restrict__ kd_refs,
                                                     unsigned long long *__restrict__ slots) {
  const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
  uint32_t key = CRT_INVALID;
  double overhang = 0.0, absmax = 0.0;
  if (j < nF) {
    const BNode n = nodes[j];
    const uint32_t t = n.tree, nb = node_base[t], rb = ref_base[t], cnt = leaf_cnt[j];
    const uint32_t c0 = child[2 * j], c1 = child[2 * j + 1];
    const uint32_t vg = nb + vis[j];
    uint32_t a, b;
    if (cnt) {
      a = CRT_LEAF_FLAG | cnt;
      b = rb + ref[j];
    } else {
      a = vg + size[j];
      b = (c0 != CRT_INVALID && c1 != CRT_INVALID) ? nb + next_vis[c0] : CRT_INVALID;
    }
    out_nodes[2 * (size_t)vg] = make_float4(n.mn[0], n.mn[1], n.mn[2], __uint_as_float(a));
    out_nodes[2 * (size_t)vg + 1] = make_float4(n.mx[0], n.mx[1], n.mx[2], __uint_as_float(b));
    if (kd) {
      crtb200_kdnode k;
      for (int i = 0; i < 3; i++) {
        k.box_min[i] = n.mn[i];
        k.box_max[i] = n.mx[i];
      }
      k.child[0] = c0 != CRT_INVALID ? next_pre[c0] : CRT_INVALID;
      k.child[1] = c1 != CRT_INVALID ? next_pre[c1] : CRT_INVALID;
      k.leaf_start = cnt ? ref[j] : 0u;
      k.leaf_count = cnt;
      kd[nb + pre[j]] = k;
    }
    if (t < n_meshes) {
      key = t;
      for (int i = 0; i < 3; i++) absmax = smax(absmax, smax(fabs((double)n.mn[i]), fabs((double)n.mx[i])));
      for (uint32_t q = 0; q < cnt; q++) {
        const uint32_t local = leafbuf[leaf_off[j] + q] - item_base[t];
        const uint32_t p = rb + ref[j] + q;
        const size_t tri = (size_t)mesh_tri[t] + local;
        out_refs[p] = (uint32_t)tri;
        if (kd_refs) kd_refs[p] = local;
        const float4 v0 = geom[3 * tri], v1 = geom[3 * tri + 1], v2 = geom[3 * tri + 2];
        const double x[3][3] = {{v0.x, v1.x, v2.x}, {v0.y, v1.y, v2.y}, {v0.z, v1.z, v2.z}};
        for (int i = 0; i < 3; i++) {
          const double lo = smin(x[i][0], smin(x[i][1], x[i][2])), hi = smax(x[i][0], smax(x[i][1], x[i][2]));
          overhang = smax(overhang, smax((double)n.mn[i] - lo, hi - (double)n.mx[i]));
        }
      }
    } else {
      for (uint32_t q = 0; q < cnt; q++) out_top_refs[rb + ref[j] + q] = leafbuf[leaf_off[j] + q] - n_items;
    }
  }
  build_warp_max(slots, key, 0, (unsigned long long)__double_as_longlong(overhang));
  build_warp_max(slots, key, 2, (unsigned long long)__double_as_longlong(absmax));
}

// Per mesh-tree item: the triangle's slop term, its vertices' absmax, and whether its uploaded normal fails the
// geometric-normal test (mesh_cull_margin's per-triangle loop, same operations in the same order, built --fmad=false).
__global__ void __launch_bounds__(256) k_build_tri_margin(const float4 *__restrict__ geom, const uint32_t *__restrict__ item_base,
                                                          const uint32_t *__restrict__ mesh_tri, uint32_t n_meshes, uint32_t n_items,
                                                          unsigned long long *__restrict__ slots) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  uint32_t key = CRT_INVALID;
  double slop = 0.0, absmax = 0.0;
  unsigned long long bad = 0;
  if (i < n_items) {
    const uint32_t m = build_item_mesh(item_base, n_meshes, i);
    key = m;
    const size_t t = (size_t)mesh_tri[m] + (i - item_base[m]);
    double p[3][3];
    float nn[3];
    for (int v = 0; v < 3; v++) {
      const float4 g = geom[3 * t + v];
      p[v][0] = g.x;
      p[v][1] = g.y;
      p[v][2] = g.z;
      nn[v] = g.w;
      for (int k = 0; k < 3; k++) absmax = smax(absmax, fabs(p[v][k]));
    }
    double len[3];
    for (int k = 0; k < 3; k++) {
      const double *a = p[k], *b = p[(k + 1) % 3];
      len[k] = sqrt((b[0] - a[0]) * (b[0] - a[0]) + (b[1] - a[1]) * (b[1] - a[1]) + (b[2] - a[2]) * (b[2] - a[2]));
    }
    const double u[3] = {p[1][0] - p[0][0], p[1][1] - p[0][1], p[1][2] - p[0][2]};
    const double w[3] = {p[2][0] - p[0][0], p[2][1] - p[0][1], p[2][2] - p[0][2]};
    const double cr[3] = {u[1] * w[2] - u[2] * w[1], u[2] * w[0] - u[0] * w[2], u[0] * w[1] - u[1] * w[0]};
    const double a2 = sqrt(cr[0] * cr[0] + cr[1] * cr[1] + cr[2] * cr[2]);
    if (!(a2 > 0.0) || !isfinite(a2)) {
      for (int k = 0; k < 3; k++)
        if (isfinite(nn[k]) && nn[k] != 0.0f) bad = 1;
    } else {
      for (int k = 0; k < 3; k++)
        if (!(fabs((double)nn[k] - cr[k] / a2) <= 1e-3)) bad = 1;
      const double emax = smax(len[0], smax(len[1], len[2]));
      slop = smax(slop, (double)CRT_FLT_EPSILON * (1.0 + 8.0 * emax * emax) * (len[0] + len[1] + len[2]) / a2);
    }
  }
  build_warp_max(slots, key, 1, (unsigned long long)__double_as_longlong(slop));
  build_warp_max(slots, key, 2, (unsigned long long)__double_as_longlong(absmax));
  build_warp_max(slots, key, 3, bad);
}

// Per mesh: mu = overhang + 4 * slop + 64 ulp * absmax, +inf when the trees do not nest or a normal failed.
__global__ void __launch_bounds__(256) k_build_margins(uint32_t n_meshes, const unsigned long long *__restrict__ slots,
                                                       const uint32_t *__restrict__ nested, DMesh *__restrict__ meshes) {
  const uint32_t m = blockIdx.x * blockDim.x + threadIdx.x;
  if (m >= n_meshes) return;
  const float inf = __int_as_float(0x7f800000);
  float mu_f = inf;
  if (*nested && !slots[4ull * m + 3]) {
    const double overhang = __longlong_as_double((long long)slots[4ull * m]), slop = __longlong_as_double((long long)slots[4ull * m + 1]),
                 absmax = __longlong_as_double((long long)slots[4ull * m + 2]);
    const double mu = overhang + 4.0 * slop + 64.0 * (double)CRT_FLT_EPSILON * absmax;
    mu_f = (isfinite(mu) && mu < 1e30) ? (float)(mu * (1.0 + 1e-6)) : inf;
  }
  meshes[m].cull_margin = mu_f;
}

// ---- vertex update: crtb200_update_vertices_device (DESIGN.md 3.14) --------------------------------------------------
// Mesh::Mesh (Scene.cpp:5-30; csrc/frontend/crt_scene.cpp): per triangle n = cross(p1 - p0, p2 - p0), normalised; per
// vertex the sum, from +0.0, of the face normals of its corners in (triangle, corner) order, normalised.

// Per triangle: its three records of the build's triangle geometry (position, face normal component k in w), its face
// normal, and its corners (key = vertex id, value = triangle) for the stable sort into the incidence list.
__global__ void __launch_bounds__(256) k_update_tri_records(const float *__restrict__ pos, const uint4 *__restrict__ tri_shade,
                                                            uint32_t n_tris, float4 *__restrict__ geom, float4 *__restrict__ face_n,
                                                            uint32_t *__restrict__ corner_vtx, uint32_t *__restrict__ corner_tri) {
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n_tris) return;
  const uint4 s = tri_shade[t];
  const uint32_t iv[3] = {s.x, s.y, s.z};
  V3 p[3];
#pragma unroll
  for (int k = 0; k < 3; k++) p[k] = mk(pos[3 * (size_t)iv[k]], pos[3 * (size_t)iv[k] + 1], pos[3 * (size_t)iv[k] + 2]);
  const V3 n = vnorm(vcross(vsub(p[1], p[0]), vsub(p[2], p[0])));
  const float nk[3] = {n.x, n.y, n.z};
#pragma unroll
  for (int k = 0; k < 3; k++) {
    geom[3 * (size_t)t + k] = make_float4(p[k].x, p[k].y, p[k].z, nk[k]);
    corner_vtx[3 * (size_t)t + k] = iv[k];
    corner_tri[3 * (size_t)t + k] = t;
  }
  face_n[t] = make_float4(n.x, n.y, n.z, 0.f);
}

// Per vertex: its corners are the run of its id in the sorted keys (found by binary search); their face normals are
// added in order to +0.0 (not started from the first term: +0 + -0 = +0 is what the reference computes), then
// normalised.  A vertex no triangle references keeps (0, 0, 0).
__global__ void __launch_bounds__(256) k_update_vertex_normals(const uint32_t *__restrict__ sorted_vtx, const uint32_t *__restrict__ sorted_tri,
                                                               uint64_t n_corners, uint32_t n_vertices, const float4 *__restrict__ face_n,
                                                               float4 *__restrict__ vtx_normal) {
  const uint32_t v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= n_vertices) return;
  uint64_t lo = 0, hi = n_corners;  // first corner with key >= v
  while (lo < hi) {
    const uint64_t mid = (lo + hi) >> 1;
    if (sorted_vtx[mid] < v) lo = mid + 1; else hi = mid;
  }
  V3 sum = mk(0.0f, 0.0f, 0.0f);
  for (uint64_t i = lo; i < n_corners && sorted_vtx[i] == v; i++) {
    const float4 f = face_n[sorted_tri[i]];
    sum = vadd(sum, mk(f.x, f.y, f.z));
  }
  sum = vnorm(sum);
  vtx_normal[v] = make_float4(sum.x, sum.y, sum.z, 0.f);
}

}  // namespace crtd
