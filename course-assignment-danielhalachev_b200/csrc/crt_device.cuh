// crt_device.cuh -- device-side data layout and the exact-arithmetic building blocks of the wavefront pipeline.
//
// Every floating-point expression on the result path is written with the explicit round-to-nearest intrinsics
// (__fmul_rn / __fadd_rn / __fsub_rn / __fdiv_rn / __fsqrt_rn), which are never contracted into FMAs and are
// IEEE-754 correctly rounded independent of -fmad / -prec-div / -prec-sqrt.  The library is additionally built with
// --fmad=false.  The operand ORDER of each expression follows the reference (SURVEY.md App. A), because the parity
// bar is bit-exact hit ids and bit-identical float RGB.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace crtd {

// ------------------------------------------------------------------------------------------------------------
// HBM layout (all arrays immutable after upload, 16-byte aligned records)
//
//  nodes     2 x float4 per KD node, ALL trees in one array (mesh trees first, then the top-level tree).  Inside a
//            tree the nodes are stored in the reference's VISITING order (child[1] subtree before child[0] subtree,
//            KDTree.cpp:65-72 pushes 0 then 1 on a LIFO stack) so the fixed-order DFS needs no stack at all:
//              lo = {min.x, min.y, min.z, a}   hi = {max.x, max.y, max.z, b}
//              inner node : a = index of the next node when the slab test fails ("skip", end of its subtree)
//              leaf node  : a = 0x80000000 | reference count, b = first reference; next node is always index + 1
//            Passing nodes continue at index + 1.  A 32-byte node is exactly one DRAM/L2 sector.
//  leaf_refs u32 GLOBAL triangle ids of the mesh trees' leaves, in the reference's stored order.
//  top_refs  u32 mesh ids of the top-level tree's leaves.
//  tri_geom  3 x float4 per triangle: {v0, n.x} {v1, n.y} {v2, n.z}  (48 B: everything Ray::intersectWithTriangle reads)
//  tri_shade uint4 per triangle: {i0, i1, i2, mesh}  -- only touched once per ray, at shading time
// ------------------------------------------------------------------------------------------------------------
//
// Conservative culling (traversal mode 0, the default).  DMesh::cull_margin (mu) is computed at upload so that every
// leaf L listing a triangle T satisfies bbox(T) c inflate(L, mu) and every point the reference's triangle test can
// accept for T lies within mu of bbox(T) (DESIGN.md section 3.6 has the derivation and the proof of exactness).
// Consequence: a leaf (or subtree, by box nesting) whose box inflated by mu lies wholly behind the ray origin, or wholly
// beyond a distance limit, contributes no finite candidate with t >= 0 (resp. t <= limit) -- skipping it removes no
// candidate that can change the result.  mu = +inf switches culling off for a mesh (trees that do not nest, triangles
// whose uploaded normal is not their geometric normal).
struct DMesh {
  uint32_t node_begin, node_end;  // [begin, end) in `nodes`
  uint32_t material;
  uint32_t first_triangle;
  float cull_margin;              // mu of this mesh's tree (see above); +inf = never cull
};
struct DMaterial {
  uint32_t type, smooth, texture;
  float ior;
  float albedo[3];
  float pad;
};
struct DTexture {
  uint32_t kind;
  float color_a[3];
  float color_b[3];
  float scalar;
  uint32_t width, height;
  unsigned long long texel_offset;
};
struct DLight {
  float pos[3];
  float intensity;  // static_cast<float>(light.intentsity), exact for the u32 -> f32 conversion of the reference
};

struct DScene {
  const float4 *nodes;
  const uint32_t *leaf_refs;
  const uint32_t *top_refs;
  const float4 *tri_geom;
  const uint4 *tri_shade;
  const float4 *vtx_normal;
  const float2 *vtx_uv;
  const DMesh *meshes;
  const DMaterial *materials;
  const DTexture *textures;
  const float *texels;
  const DLight *lights;
  uint32_t n_lights, n_meshes;
  uint32_t top_begin, top_end;
  uint32_t width, height;
  float bg[3];
  uint32_t dedup_meshes;  // per-ray visited-mesh set: 1 = a 64-bit register (n_meshes <= 64), 2 = dedup_words words per
                          // lane in dynamic shared memory (n_meshes <= 512), 0 = none (more meshes: every listing is walked)
  uint32_t dedup_words;
};

struct DCamera {
  float pos[3];
  float rot[9];
};

// ------------------------------------------------------------------------------------------------------------
// exact float helpers
// ------------------------------------------------------------------------------------------------------------
#define CRT_DI __device__ __forceinline__
#ifndef CRT_TRAV_BLOCK
#define CRT_TRAV_BLOCK 256      // threads per CTA of the persistent traversal kernels
#endif
#ifndef CRT_NODE_PAIR
#define CRT_NODE_PAIR 1  // MODE 2 node phase: test nodes idx and idx + 1 together (trav_fast2)
#endif
#ifndef CRT_PREFETCH_SKIP
#define CRT_PREFETCH_SKIP 0  // tuning: prefetch a node's skip target into L1 as soon as the node arrives
#endif

CRT_DI float fmul(float a, float b) { return __fmul_rn(a, b); }
CRT_DI float fadd(float a, float b) { return __fadd_rn(a, b); }
CRT_DI float fsub(float a, float b) { return __fsub_rn(a, b); }
CRT_DI float fdiv(float a, float b) { return __fdiv_rn(a, b); }
CRT_DI float fsqrt(float a) { return __fsqrt_rn(a); }

struct V3 {
  float x, y, z;
};
CRT_DI V3 mk(float x, float y, float z) {
  V3 r;
  r.x = x;
  r.y = y;
  r.z = z;
  return r;
}
CRT_DI V3 vsub(V3 a, V3 b) { return mk(fsub(a.x, b.x), fsub(a.y, b.y), fsub(a.z, b.z)); }
CRT_DI V3 vadd(V3 a, V3 b) { return mk(fadd(a.x, b.x), fadd(a.y, b.y), fadd(a.z, b.z)); }
// (a0*b0 + a1*b1) + a2*b2                                                         Vector.cpp:57-59
CRT_DI float vdot(V3 a, V3 b) { return fadd(fadd(fmul(a.x, b.x), fmul(a.y, b.y)), fmul(a.z, b.z)); }
// Vector.cpp:61-65
CRT_DI V3 vcross(V3 a, V3 b) {
  return mk(fsub(fmul(a.y, b.z), fmul(a.z, b.y)), fsub(fmul(a.z, b.x), fmul(a.x, b.z)),
            fsub(fmul(a.x, b.y), fmul(a.y, b.x)));
}
CRT_DI V3 vscale(V3 a, float s) { return mk(fmul(a.x, s), fmul(a.y, s), fmul(a.z, s)); }  // Vector * float
CRT_DI V3 sscale(float s, V3 a) { return mk(fmul(s, a.x), fmul(s, a.y), fmul(s, a.z)); }  // float * Vector
CRT_DI float vlen(V3 a) { return fsqrt(fadd(fadd(fmul(a.x, a.x), fmul(a.y, a.y)), fmul(a.z, a.z))); }
// Vector::normalize                                                             Vector.cpp:97-106
CRT_DI V3 vnorm(V3 a) {
  float l = vlen(a);
  if (l == 0.0f) return a;
  l = fdiv(1.0f, l);
  return mk(fmul(a.x, l), fmul(a.y, l), fmul(a.z, l));
}
// Vector::reflect: *this - (2 * dot) * normal                                   Vector.cpp:119-122
CRT_DI V3 vreflect(V3 d, V3 n) { return vsub(d, sscale(fmul(2.0f, vdot(d, n)), n)); }
// std::max(a,b) = (a<b)?b:a, std::min(a,b) = (b<a)?b:a -- written as selects so NaN operands behave like libstdc++
CRT_DI float stdmax(float a, float b) { return (a < b) ? b : a; }
CRT_DI float stdmin(float a, float b) { return (b < a) ? b : a; }

#define CRT_FLT_EPSILON 1.1920928955078125e-7f
#define CRT_FLT_MAX 3.402823466e+38f
#define CRT_INVALID 0xFFFFFFFFu
#define CRT_LEAF_FLAG 0x80000000u

// ------------------------------------------------------------------------------------------------------------
// Read-only loads of the scene with an L1 residency policy per data class (A/B knobs for tools/ builds; 0 = ld.global.nc
// with the default policy, which is what ships -- see profiles/r2_tuning.md section 5 for the measurements):
//   1 = L1::evict_last   2 = L1::no_allocate   3 = L1::evict_first
// CRT_NODE_LD applies to KD nodes, CRT_TRI_LD to leaf references and triangle records.
// ------------------------------------------------------------------------------------------------------------
#ifndef CRT_NODE_LD
#define CRT_NODE_LD 0
#endif
#ifndef CRT_TRI_LD
#define CRT_TRI_LD 0
#endif
template <int POLICY>
CRT_DI float4 ld_policy(const float4 *p) {
  if (POLICY == 0) return __ldg(p);
  float4 v;
  if (POLICY == 1) asm volatile("ld.global.nc.L1::evict_last.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
  if (POLICY == 2) asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
  if (POLICY == 3) asm volatile("ld.global.nc.L1::evict_first.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
  return v;
}
template <int POLICY>
CRT_DI uint32_t ld_policy(const uint32_t *p) {
  if (POLICY == 0) return __ldg(p);
  uint32_t v = 0;
  if (POLICY == 1) asm volatile("ld.global.nc.L1::evict_last.u32 %0, [%1];" : "=r"(v) : "l"(p));
  if (POLICY == 2) asm volatile("ld.global.nc.L1::no_allocate.u32 %0, [%1];" : "=r"(v) : "l"(p));
  if (POLICY == 3) asm volatile("ld.global.nc.L1::evict_first.u32 %0, [%1];" : "=r"(v) : "l"(p));
  return v;
}
CRT_DI float4 ld_node(const float4 *p) { return ld_policy<CRT_NODE_LD>(p); }
CRT_DI float4 ld_tri(const float4 *p) { return ld_policy<CRT_TRI_LD>(p); }
CRT_DI uint32_t ld_ref(const uint32_t *p) { return ld_policy<CRT_TRI_LD>(p); }

// ------------------------------------------------------------------------------------------------------------
// rays
// ------------------------------------------------------------------------------------------------------------
struct Ray {
  V3 o, d;
  V3 inv;         // 1.0f / d per axis (BoundingBox.h:95), hoisted: depends on the ray only
  uint32_t flags; // bit i: |d_i| < FLT_EPSILON (BoundingBox.h:90); bit 3: primary ray (back-face cull, Ray.cpp:13);
                  // bit 4: some component of o / d / inv is NaN or inf (slab test must take the select-exact path)
};

#define CRT_RAY_SLOW_MASK 0x17u  // any axis-parallel flag or the non-finite flag

CRT_DI void ray_prepare(Ray &r, bool primary) {
  r.flags = primary ? 8u : 0u;
  if (fabsf(r.d.x) < CRT_FLT_EPSILON) r.flags |= 1u;
  if (fabsf(r.d.y) < CRT_FLT_EPSILON) r.flags |= 2u;
  if (fabsf(r.d.z) < CRT_FLT_EPSILON) r.flags |= 4u;
  r.inv.x = fdiv(1.0f, r.d.x);
  r.inv.y = fdiv(1.0f, r.d.y);
  r.inv.z = fdiv(1.0f, r.d.z);
  // exponent all-ones <=> NaN or inf.  inv of a flagged (parallel) axis is never used, so it does not count.
  uint32_t e = __float_as_uint(r.o.x) | __float_as_uint(r.o.y) | __float_as_uint(r.o.z);
  const uint32_t nf = 0x7f800000u;
  bool bad = ((__float_as_uint(r.o.x) & nf) == nf) || ((__float_as_uint(r.o.y) & nf) == nf) || ((__float_as_uint(r.o.z) & nf) == nf) ||
             ((__float_as_uint(r.d.x) & nf) == nf) || ((__float_as_uint(r.d.y) & nf) == nf) || ((__float_as_uint(r.d.z) & nf) == nf);
  (void)e;
  if (!(r.flags & 1u)) bad = bad || ((__float_as_uint(r.inv.x) & nf) == nf);
  if (!(r.flags & 2u)) bad = bad || ((__float_as_uint(r.inv.y) & nf) == nf);
  if (!(r.flags & 4u)) bad = bad || ((__float_as_uint(r.inv.z) & nf) == nf);
  if (bad) r.flags |= 16u;
}

// RayTracer::getRay + the second normalisation of shootRay                      RayTracer.cpp:61-80, 420
// x, y = the pixel position: col + 0.5, row + 0.5, or col + jitter, row + jitter (sampling contract, DESIGN.md 3.10)
CRT_DI void primary_ray_at(const DCamera &cam, uint32_t W, uint32_t H, float x, float y, V3 &o, V3 &d) {
  x = fdiv(x, (float)W);
  y = fdiv(y, (float)H);
  x = fsub(fmul(2.0f, x), 1.0f);
  y = fsub(1.0f, fmul(2.0f, y));
  x = fmul(x, fdiv((float)W, (float)H));
  const float z = -1.0f;
  // Vector * Matrix<3>                                                          Matrix.h:137-142
  V3 dr = mk(fadd(fadd(fmul(x, cam.rot[0]), fmul(y, cam.rot[3])), fmul(z, cam.rot[6])),
             fadd(fadd(fmul(x, cam.rot[1]), fmul(y, cam.rot[4])), fmul(z, cam.rot[7])),
             fadd(fadd(fmul(x, cam.rot[2]), fmul(y, cam.rot[5])), fmul(z, cam.rot[8])));
  d = vnorm(vnorm(dr));
  o = mk(cam.pos[0], cam.pos[1], cam.pos[2]);
}
CRT_DI void primary_ray(const DCamera &cam, uint32_t W, uint32_t H, uint32_t row, uint32_t col, V3 &o, V3 &d) {
  primary_ray_at(cam, W, H, fadd((float)col, 0.5f), fadd((float)row, 0.5f), o, d);
}

// BoundingBox::hasIntersection                                                  BoundingBox.h:85-108
// (no t1 >= 0 test: boxes behind the origin pass; NaN bounds never reject -- both as in the reference).
//
// slab_test_exact: the reference's statements as selects (std::max / std::min / swap NaN behaviour included); the early
// returns of the reference only skip work, every reject condition is evaluated on the same running (t0, t1), so OR-ing
// them is exact.  An axis with |d| < FLT_EPSILON leaves (t0, t1) untouched.
CRT_DI bool slab_test_exact(const float4 lo, const float4 hi, const Ray &r, float &t0, float &t1) {
  t0 = -CRT_FLT_MAX;
  t1 = CRT_FLT_MAX;
  bool reject = false;
#define CRT_SLAB_AXIS(bit, O, I, MN, MX)                                  \
  {                                                                       \
    const bool par = (r.flags & bit) != 0u;                               \
    const float a_ = fmul(fsub(MN, O), I);                                \
    const float b_ = fmul(fsub(MX, O), I);                                \
    const bool sw = a_ > b_;                                              \
    const float tn = sw ? b_ : a_;                                        \
    const float tf = sw ? a_ : b_;                                        \
    const float n0 = stdmax(t0, tn);                                      \
    const float n1 = stdmin(t1, tf);                                      \
    t0 = par ? t0 : n0;                                                   \
    t1 = par ? t1 : n1;                                                   \
    reject = reject || (par ? (O < MN || O > MX) : (t0 > t1));            \
  }
  CRT_SLAB_AXIS(1u, r.o.x, r.inv.x, lo.x, hi.x)
  CRT_SLAB_AXIS(2u, r.o.y, r.inv.y, lo.y, hi.y)
  CRT_SLAB_AXIS(4u, r.o.z, r.inv.z, lo.z, hi.z)
#undef CRT_SLAB_AXIS
  return !reject;
}

// Fast path for the overwhelmingly common ray: all of o, d, 1/d finite and no axis-parallel component.  Then every
// (bound - o) * inv is finite (finite boxes), so the swap / std::max / std::min selects see no NaN and equal the hardware
// min / max up to the sign of zero, which no later comparison observes; and because t0 only grows and t1 only
// shrinks, the reference's three "t0 > t1" early returns collapse into one final test.
CRT_DI bool slab_test(const float4 lo, const float4 hi, const Ray &r, float &t0, float &t1) {
  if (r.flags & CRT_RAY_SLOW_MASK) return slab_test_exact(lo, hi, r, t0, t1);
  const float ax = fmul(fsub(lo.x, r.o.x), r.inv.x), bx = fmul(fsub(hi.x, r.o.x), r.inv.x);
  const float ay = fmul(fsub(lo.y, r.o.y), r.inv.y), by = fmul(fsub(hi.y, r.o.y), r.inv.y);
  const float az = fmul(fsub(lo.z, r.o.z), r.inv.z), bz = fmul(fsub(hi.z, r.o.z), r.inv.z);
  t0 = fmaxf(fmaxf(fmaxf(-CRT_FLT_MAX, fminf(ax, bx)), fminf(ay, by)), fminf(az, bz));
  t1 = fminf(fminf(fminf(CRT_FLT_MAX, fmaxf(ax, bx)), fmaxf(ay, by)), fmaxf(az, bz));
  return !(t0 > t1);
}

// Ray::intersectWithTriangle + Triangle::pointIsInTriangle                       Ray.cpp:9-31, Triangle.cpp:37-57
// Returns true for a candidate; t may be NaN / inf exactly like the reference (SURVEY App. B-3).  The early exits are
// structured `if`s (immediate reconvergence), in the reference's order: cull, t < 0, edge 0, edge 1, edge 2.
CRT_DI bool triangle_test(const float4 g0, const float4 g1, const float4 g2, const Ray &r, float &t_out, V3 &p_out) {
  const V3 n = mk(g0.w, g1.w, g2.w);
  const V3 v0 = mk(g0.x, g0.y, g0.z);
  const float nd = vdot(r.d, n);
  const float dist = -vdot(v0, n);
  const float t = fdiv(-fadd(vdot(n, r.o), dist), nd);
  bool hit = !(((r.flags & 8u) && nd >= 0.0f) || (t < 0.0f));
  if (hit) {
    const V3 p = vadd(r.o, vscale(r.d, t));
    const V3 v1 = mk(g1.x, g1.y, g1.z);
    hit = !(vdot(n, vcross(vsub(v1, v0), vsub(p, v0))) < -CRT_FLT_EPSILON);
    if (hit) {
      const V3 v2 = mk(g2.x, g2.y, g2.z);
      hit = !(vdot(n, vcross(vsub(v2, v1), vsub(p, v1))) < -CRT_FLT_EPSILON) &&
            !(vdot(n, vcross(vsub(v0, v2), vsub(p, v2))) < -CRT_FLT_EPSILON);
      t_out = t;
      p_out = p;
    }
  }
  return hit;
}

// ------------------------------------------------------------------------------------------------------------
// Stack-free two-level traversal state (one per lane, registers only).
//   top        cursor in the top-level tree          [top_begin, top_end)
//   mref/mend  cursor in the current top-level leaf's mesh list
//   cur/cend   cursor in the current mesh tree
//   tref/tend  cursor in the current mesh leaf's triangle list
// Order of events = the reference's: KDTree.cpp:127-166 (top level) around KDTree.cpp:48-87 (per mesh).
// ------------------------------------------------------------------------------------------------------------
struct Trav {
  uint32_t cur, cend;     // node cursor and its end: inside a mesh tree, or in the top-level tree
  uint32_t resume;        // top-level cursor to continue from once the current leaf's meshes are done
  uint32_t mref, mend;    // cursor in the current top-level leaf's mesh list
  uint32_t tref, tend;    // cursor in the current mesh leaf's triangle list
  uint32_t below;         // 1 while working below a top-level leaf (mesh list / mesh trees)
  unsigned long long seen;  // meshes already traversed for this ray (scenes with <= 64 meshes)
  uint32_t leaf;          // node index of the pending leaf (trav_fast2): encounter-order key for the long-walk pass
  float mu;               // culling margin of the tree being walked, in space units (+inf: top-level tree / culling off)
};
#define CRT_INF __int_as_float(0x7f800000)
// visited-mesh bitset of scenes with more than 64 meshes: word w of thread t at crt_dyn_smem[w * blockDim.x + t].
// Kept out of line: the common case (<= 64 meshes, a 64-bit register) must not pay registers for it.
extern __shared__ uint32_t crt_dyn_smem[];
static __device__ __noinline__ void dedup_smem_clear(const uint32_t words) {
  for (uint32_t w = 0; w < words; w++) crt_dyn_smem[w * blockDim.x + threadIdx.x] = 0u;
}
static __device__ __noinline__ bool dedup_smem_test_and_set(const uint32_t m) {
  uint32_t *w = crt_dyn_smem + (m >> 5) * blockDim.x + threadIdx.x;
  const uint32_t bit = 1u << (m & 31u), old = *w;
  *w = old | bit;
  return (old & bit) != 0u;
}
// WIDE: the kernel was instantiated for scenes whose visited-mesh set lives in shared memory (65..512 meshes).  The
// one-ray-per-lane traversal kernels exist in both flavours so that the common one carries no code for the other
// (measured: with a run-time switch inside one kernel hw11_room_128 lost 10 %, profiles/r2_tuning.md section 5).
template <bool WIDE>
CRT_DI void trav_begin(Trav &s, const DScene &sc) {
  if (WIDE && sc.dedup_meshes == 2u) dedup_smem_clear(sc.dedup_words);
  s.cur = sc.top_begin;
  s.cend = sc.top_end;
  s.resume = sc.top_end;
  s.mref = s.mend = 0;
  s.tref = s.tend = 0;
  s.below = 0;
  s.seen = 0ull;
  s.leaf = 0;
  s.mu = CRT_INF;
}

// Culling margin for ray r inside a mesh whose upload-time margin is `mesh_mu`: the rounding of the hit point and of
// the slab parameters is bounded by a few ulp of (|o| + mesh extent); mesh_mu already carries the extent part, the
// origin part is added here (64 ulp: an order of magnitude above the bound in DESIGN.md section 3.6).  Rays that take
// the select-exact slab path (axis-parallel / non-finite components) are never culled.
CRT_DI float cull_margin_for(const Ray &r, const float mesh_mu) {
  if (r.flags & CRT_RAY_SLOW_MASK) return CRT_INF;
  return mesh_mu + (64.0f * CRT_FLT_EPSILON) * (fabsf(r.o.x) + fabsf(r.o.y) + fabsf(r.o.z));
}

// The reference's slab test (pass / fail exactly as BoundingBox::hasIntersection) plus, for CULL, the two conservative
// skips.  With tn_i / tf_i the near / far slab parameters of axis i and m_i = mu * |1 / d_i| (mu in t units along that axis):
//   behind : some far plane lies more than mu behind the origin        tf_i < -m_i         (only when `allow_behind`)
//   beyond : some near plane lies more than mu beyond the limit        tn_i - m_i > limit
// Both are "box inflated by mu misses the ray segment [0, limit]" written per axis; NaN / +inf operands never cull.
// `m` = cull_margins(r, mu), the m_i above.
// SLOW = false: the caller knows that r is a fast ray (no CRT_RAY_SLOW_MASK flag), and the test carries neither the flag
// test nor the select-exact path.
CRT_DI V3 cull_margins(const Ray &r, const float mu) { return mk(mu * fabsf(r.inv.x), mu * fabsf(r.inv.y), mu * fabsf(r.inv.z)); }
template <bool CULL, bool SLOW = true>
CRT_DI bool node_test(const float4 lo, const float4 hi, const Ray &r, const V3 m, const float limit, const bool allow_behind) {
  if (SLOW && (r.flags & CRT_RAY_SLOW_MASK)) {
    float t0, t1;
    return slab_test_exact(lo, hi, r, t0, t1);
  }
  const float ax = fmul(fsub(lo.x, r.o.x), r.inv.x), bx = fmul(fsub(hi.x, r.o.x), r.inv.x);
  const float ay = fmul(fsub(lo.y, r.o.y), r.inv.y), by = fmul(fsub(hi.y, r.o.y), r.inv.y);
  const float az = fmul(fsub(lo.z, r.o.z), r.inv.z), bz = fmul(fsub(hi.z, r.o.z), r.inv.z);
  const float nx = fminf(ax, bx), fx = fmaxf(ax, bx);
  const float ny = fminf(ay, by), fy = fmaxf(ay, by);
  const float nz = fminf(az, bz), fz = fmaxf(az, bz);
  const float t0 = fmaxf(fmaxf(fmaxf(-CRT_FLT_MAX, nx), ny), nz);
  const float t1 = fminf(fminf(fminf(CRT_FLT_MAX, fx), fy), fz);
  bool pass = !(t0 > t1);
  if (CULL) {
    const bool behind = allow_behind && ((fx < -m.x) || (fy < -m.y) || (fz < -m.z));
    const bool beyond = fmaxf(fmaxf(nx - m.x, ny - m.y), nz - m.z) > limit;  // fmaxf drops a NaN operand, as || drops its false test
    pass = pass && !behind && !beyond;
  }
  return pass;
}

// One traversal micro-step of the walk (trav_fast / trav_fast2 for an AABB step, trav_slow between trees): the state
// transitions of KDTree.cpp:48-87 / 127-166.  trav_slow returns TRAV_STEP = keep stepping or TRAV_DONE = traversal
// complete.  Top-level and mesh-level AABB tests share one code path so lanes at different levels do not diverge.
//   SKIP_REFRACTIVE  shadow rays ignore refractive meshes (AccelerationStructure.cpp:67-71).
//   DEDUP            a mesh listed in several top-level leaves is traversed once per ray instead of once per listing.
//                    Exact: a repeated traversal (KDTree.cpp:131-155 does repeat it) yields the same candidates again,
//                    which can neither replace the kept one (strict <) nor be the first candidate.  Off when counting
//                    the reference's visit-all work.
//   CULL             conservative culling inside mesh trees (node_test): `limit` = the best finite hit so far / the
//                    light distance, `allow_behind` = a finite candidate exists (closest hit) / always (shadow).
enum { TRAV_STEP = 0, TRAV_LEAF = 1, TRAV_DONE = 2 };
template <bool SKIP_REFRACTIVE, int DEDUP, bool CULL>
CRT_DI int trav_slow(Trav &s, const DScene &sc, const Ray &r);

// The step split in two for the MODE 2 kernels (crt_kernels.cuh), whose tight node loop only wants the AABB step:
//   trav_fast   one AABB test for a lane with cur != cend.  Returns true while the lane can take another fast step;
//               false when a triangle range is pending (tref..tend) or the cursor ran off its tree (trav_slow is due).
//   trav_slow   the bookkeeping between trees for a lane with cur == cend and no pending triangles: next mesh of the
//               current top-level leaf, or back to the top-level tree, or TRAV_DONE.
// Together they perform exactly the state transitions of the reference's walk.
template <bool COUNT, bool CULL, bool SLOW>
CRT_DI bool trav_fast(Trav &s, const DScene &sc, const Ray &r, uint32_t &node_tests, const V3 m, const float limit, const bool allow_behind) {
  const uint32_t idx = s.cur;
  const float4 lo = ld_node(&sc.nodes[2 * (size_t)idx]);
  const float4 hi = ld_node(&sc.nodes[2 * (size_t)idx + 1]);
  const uint32_t a = __float_as_uint(lo.w);
  const bool leaf = (a & CRT_LEAF_FLAG) != 0u;
#if CRT_PREFETCH_SKIP
  // the node after this subtree is visited whatever happens here (visit-all order): start pulling it into L1
  if (!leaf) asm volatile("prefetch.global.L1 [%0];" ::"l"(&sc.nodes[2 * (size_t)a]));
#endif
  if (COUNT) node_tests++;
  const bool pass = node_test<CULL, SLOW>(lo, hi, r, m, limit, allow_behind);
  s.cur = (pass || leaf) ? idx + 1 : a;
  if (pass && leaf) {
    const uint32_t first = __float_as_uint(hi.w), last = first + (a & ~CRT_LEAF_FLAG);
    if (s.below) {
      s.tref = first;
      s.tend = last;
    } else {  // a top-level leaf: remember where to continue, then walk its meshes (trav_slow)
      s.mref = first;
      s.mend = last;
      s.resume = s.cur;
      s.cur = s.cend;
      s.below = 1u;
    }
    s.leaf = idx;
    return false;
  }
  return s.cur < s.cend;
}
// trav_fast for two consecutive nodes at once (CRT_NODE_PAIR).  Node idx + 1 is the next node of the walk whenever
// node idx passes or is a leaf -- about 56 % of the steps on the 1 M-triangle scene -- so its box is loaded and tested
// together with node idx's: two independent load + ALU chains per iteration instead of one, and 1.5x fewer iterations
// of a loop whose iteration time is the latency of the slowest lane's load.  When node idx fails (an inner node) the
// second test is simply discarded; testing a node the reference would not have reached cannot change the walk,
// because only the pass / fail of nodes that ARE reached is acted on.
template <bool COUNT, bool CULL, bool SLOW>
CRT_DI bool trav_fast2(Trav &s, const DScene &sc, const Ray &r, uint32_t &node_tests, const V3 m, const float limit, const bool allow_behind) {
  const uint32_t idx = s.cur;
  const bool has2 = idx + 1u < s.cend;
  const uint32_t jdx = has2 ? idx + 1u : idx;
  const float4 lo0 = ld_node(&sc.nodes[2 * (size_t)idx]), hi0 = ld_node(&sc.nodes[2 * (size_t)idx + 1]);
  const float4 lo1 = ld_node(&sc.nodes[2 * (size_t)jdx]), hi1 = ld_node(&sc.nodes[2 * (size_t)jdx + 1]);
  const bool pass0 = node_test<CULL, SLOW>(lo0, hi0, r, m, limit, allow_behind);
  const bool pass1 = node_test<CULL, SLOW>(lo1, hi1, r, m, limit, allow_behind);
  const uint32_t a0 = __float_as_uint(lo0.w), a1 = __float_as_uint(lo1.w);
  if (COUNT) node_tests++;
  // which of the two nodes decides where the walk goes: the second one iff the first is stepped over (inner + pass, or a
  // failing leaf) and a second one exists.  The leaf flag is the sign bit of a.
  const bool second = has2 && (pass0 != ((int32_t)a0 < 0));
  if (COUNT && second) node_tests++;
  const uint32_t a = second ? a1 : a0, at = second ? jdx : idx;
  // (pass as predicate logic: a ?: between two bools compiles to integer selects and a compare)
  const bool pass = (second && pass1) || (!second && pass0), leaf = (int32_t)a < 0;
  s.cur = (pass || leaf) ? at + 1u : a;
  if (pass && leaf) {
    const uint32_t first = __float_as_uint(second ? hi1.w : hi0.w), last = first + (a & ~CRT_LEAF_FLAG);
    if (s.below) {
      s.tref = first;
      s.tend = last;
    } else {
      s.mref = first;
      s.mend = last;
      s.resume = s.cur;
      s.cur = s.cend;
      s.below = 1u;
    }
    s.leaf = at;
    return false;
  }
  return s.cur < s.cend;
}

// DEDUP: 0 = every listing of a mesh is walked (the reference's work; counting mode), 1 = visited-mesh set in the 64-bit
// register Trav::seen (scenes with <= 64 meshes), 2 = in shared memory (65..512 meshes; kernels instantiated WIDE).
// Scenes with more meshes than that walk
// every listing -- correct (the candidates repeat and a repeat never wins a strict <), only slower.
template <bool SKIP_REFRACTIVE, int DEDUP, bool CULL>
CRT_DI int trav_slow(Trav &s, const DScene &sc, const Ray &r) {
  if (s.mref != s.mend) {
    const uint32_t m = __ldg(&sc.top_refs[s.mref++]);
    const DMesh me = sc.meshes[m];
    bool skip = SKIP_REFRACTIVE && sc.materials[me.material].type == 3u;
    if ((DEDUP & 1) && sc.dedup_meshes == 1u) {
      const unsigned long long bit = 1ull << (m & 63u);
      skip = skip || (s.seen & bit) != 0ull;
      s.seen |= bit;
    } else if ((DEDUP & 2) && sc.dedup_meshes == 2u) {
      if (dedup_smem_test_and_set(m)) skip = true;
    }
    if (!skip) {
      s.cur = me.node_begin;
      s.cend = me.node_end;
      if (CULL) s.mu = cull_margin_for(r, me.cull_margin);
    }
    return TRAV_STEP;
  }
  if (s.below) {
    s.below = 0u;
    s.cur = s.resume;
    s.cend = sc.top_end;
    s.mu = CRT_INF;  // the top-level tree is never culled (its leaves list whole meshes)
    return TRAV_STEP;
  }
  return TRAV_DONE;
}

// Closest-hit bookkeeping = "closest = intersections[0]; min = inf; for c: if (c.t < min) ..." (KDTree.cpp:75-86,
// 156-166) folded into a stream: the first candidate is kept unless a later one has t < min (strict).  Folding the
// per-mesh and the across-mesh scans into one stream is exact (DESIGN.md section 3.2).
struct Closest {
  float min_t, best_t;
  uint32_t best_tri;  // CRT_INVALID = no candidate yet
};
CRT_DI void closest_begin(Closest &c) {
  c.min_t = __int_as_float(0x7f800000);
  c.best_t = 0.0f;
  c.best_tri = CRT_INVALID;
}
CRT_DI void closest_offer(Closest &c, uint32_t tri, float t) {
  if (c.best_tri == CRT_INVALID) {
    c.best_tri = tri;
    c.best_t = t;
  }
  if (t < c.min_t) {
    c.min_t = t;
    c.best_t = t;
    c.best_tri = tri;
  }
}

}  // namespace crtd
