/* crtb200.h -- C ABI of the B200-native renderer core (libcrtb200.so).
 *
 * Drop-in boundary for the per-pixel hot path of the Chaos course ray tracer
 * (reference: SourceCode/src/RayTracer.cpp).  The reference has no FFI; its boundary is the C++ member
 *     std::vector<std::vector<Color>> RayTracer::render(const std::string&, RenderOptions)
 *         (include/tracer/RayTracer.h:100, src/RayTracer.cpp:204-298)
 * constructed by  explicit RayTracer(Scene&)  (RayTracer.h:97, RayTracer.cpp:45-51), camera mutated through
 * Camera& setCamera() (RayTracer.h:99).  Every entry point below names the reference interface it replaces.
 * INTEGRATION.md shows the binding a maintainer adds to RayTracer.cpp.
 *
 * Conventions: plain C, plain pointers + sizes, no torch / C++ types.  Every function returns 0 on success or a
 * negative crtb200_status; crtb200_last_error_ctx(ctx) returns the message of the last failed call on that context
 * (crtb200_last_error() the last one of the calling thread, for calls that have no context yet).
 * Host pointers handed to upload/render are borrowed for the duration of the call only.  One context = one caller
 * thread at a time (the reference's render() is not re-entrant either, RayTracer.cpp:205-206); a context drives one
 * GPU (crtb200_create) or several (crtb200_create_multi: scene replicated, every frame split by tiles).
 * There is NO CPU fallback: every call fails with CRTB200_ERR_CUDA when no sm_100 device is usable.
 */
#ifndef CRTB200_H
#define CRTB200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CRTB200_ABI_VERSION 2u
#define CRTB200_INVALID 0xFFFFFFFFu /* = INVALID_INDEX, include/tree/KDTree.h:11 */

typedef enum crtb200_status {
  CRTB200_OK = 0,
  CRTB200_ERR_ARG = -1,    /* null / inconsistent argument                           */
  CRTB200_ERR_CUDA = -2,   /* CUDA runtime error or no usable device                 */
  CRTB200_ERR_STATE = -3,  /* call order (render before upload, ...)                 */
  CRTB200_ERR_MEMORY = -4, /* the frame does not fit the configured device budget    */
  CRTB200_ERR_SCENE = -5   /* scene arrays fail validation (index out of range, ...) */
} crtb200_status;

/* enum MaterialType { Diffuse, Reflective, Constant, Refractive }  include/tracer/Material.h:7 */
enum { CRTB200_MAT_DIFFUSE = 0, CRTB200_MAT_REFLECTIVE = 1, CRTB200_MAT_CONSTANT = 2, CRTB200_MAT_REFRACTIVE = 3 };
/* texture classes of include/tracer/Texture.h:18-59 */
enum { CRTB200_TEX_ALBEDO = 0, CRTB200_TEX_EDGES = 1, CRTB200_TEX_CHECKER = 2, CRTB200_TEX_BITMAP = 3 };
/* enum RayType { PrimaryRay, ShadowRay, ReflectionRay, RefractionRay, DiffuseRay }  include/tracer/Ray.h:14 */
enum { CRTB200_RAY_PRIMARY = 0, CRTB200_RAY_SHADOW = 1, CRTB200_RAY_REFLECTION = 2, CRTB200_RAY_REFRACTION = 3, CRTB200_RAY_DIFFUSE = 4 };

/* One KD-tree node in the REFERENCE's numbering: KDTree<T>::TreeNode (include/tree/KDTree.h:16-21), nodes appended
 * in DFS pre-order by createNode (KDTree.h:33-38), root = 0 of its tree.  A node is a leaf iff leaf_count > 0
 * (KDTree.cpp:58 tests !indexes.empty()).  child indices are relative to the tree's first node. */
typedef struct crtb200_kdnode {
  float box_min[3];
  float box_max[3];
  uint32_t child[2];   /* CRTB200_INVALID when absent (KDTree.cpp:35,41)                        */
  uint32_t leaf_start; /* into the tree's leaf-reference array, relative to the tree's first ref */
  uint32_t leaf_count;
} crtb200_kdnode;

/* Mesh (include/tracer/Scene.h:25-38) + its TriangleKDTree (include/tree/AccelerationStructure.h:6-13). */
typedef struct crtb200_mesh {
  uint32_t material;       /* index into materials                                              */
  uint32_t first_triangle; /* the mesh's triangles are [first_triangle, first_triangle + n)     */
  uint32_t n_triangles;
  uint32_t first_vertex; /* informational; triangle_vertex holds GLOBAL vertex ids             */
  uint32_t n_vertices;
  uint32_t first_node; /* the mesh tree's nodes are mesh_nodes[first_node .. first_node+n_nodes) */
  uint32_t n_nodes;
  uint32_t first_leaf_ref; /* mesh_leaf_refs[first_leaf_ref ..) hold MESH-LOCAL triangle indices  */
  uint32_t n_leaf_refs;
} crtb200_mesh;

/* Material (include/tracer/Material.h:9-30). texture = CRTB200_INVALID for the non-USE_TEXTURES flavour. */
typedef struct crtb200_material {
  uint32_t type;
  uint32_t smooth_shading;
  uint32_t texture;
  float albedo[3];
  float ior;
} crtb200_material;

/* Texture classes (include/tracer/Texture.h:18-59, src/Texture.cpp:14-72).
 *   ALBEDO : color_a                         EDGES  : color_a = inner, color_b = edge, scalar = width
 *   CHECKER: color_a / color_b, scalar = square size
 *   BITMAP : width x height float RGB texels at texels[3*texel_offset ..] (already /255, Texture.cpp:55-59) */
typedef struct crtb200_texture {
  uint32_t kind;
  float color_a[3];
  float color_b[3];
  float scalar;
  uint32_t width, height;
  uint64_t texel_offset;
} crtb200_texture;

/* struct Light { Vector position; unsigned intentsity; }  include/tracer/Scene.h:20-23 */
typedef struct crtb200_light {
  float position[3];
  uint32_t intensity;
} crtb200_light;

/* Everything the hot path reads: Scene (Scene.h:50-69), the scene AccelerationStructure (RayTracer.h:65) flattened.
 * All arrays are host memory; indices are validated on upload. */
typedef struct crtb200_scene {
  uint32_t abi_version; /* CRTB200_ABI_VERSION */
  uint32_t width, height; /* sceneSettings.image */
  float background[3];    /* sceneSettings.sceneBackgroundColor */

  uint32_t n_vertices;
  const float *vertex_position; /* 3 per vertex: Vertex::position                                         */
  const float *vertex_normal;   /* 3 per vertex: Vertex::normal after Mesh::Mesh (Scene.cpp:5-30)         */
  const float *vertex_uv;       /* 3 per vertex (Vertex::UV) or NULL                                      */

  uint32_t n_triangles;
  const uint32_t *triangle_vertex; /* 3 global vertex ids per triangle, in Mesh::triangles order            */
  const float *triangle_normal;    /* 3 per triangle: Triangle::normal (Triangle.cpp:13-16), as computed by  */
                                   /* the host front end in binary32 without FMA                            */
  uint32_t n_meshes;
  const crtb200_mesh *meshes;
  uint32_t n_materials;
  const crtb200_material *materials;
  uint32_t n_textures;
  const crtb200_texture *textures;
  uint64_t n_texels;
  const float *texels;
  uint32_t n_lights;
  const crtb200_light *lights;

  uint32_t n_mesh_nodes;
  const crtb200_kdnode *mesh_nodes;
  uint32_t n_mesh_leaf_refs;
  const uint32_t *mesh_leaf_refs;
  uint32_t n_top_nodes; /* ObjectKDTree (AccelerationStructure.h:21-33): leaves reference mesh indices */
  const crtb200_kdnode *top_nodes;
  uint32_t n_top_leaf_refs;
  const uint32_t *top_leaf_refs;
} crtb200_scene;

/* Camera state read by getRay (RayTracer.cpp:61-80): position + row-major 3x3 (Camera.h:7-8). */
typedef struct crtb200_camera {
  float position[3];
  float rotation[9];
} crtb200_camera;

/* One rectangle handed to renderRectangle(row, col, w, h)  (RayTracer.cpp:82-85). */
typedef struct crtb200_rect {
  uint32_t row, col, width, height;
} crtb200_rect;

/* RenderOptions (RayTracer.h:25-50) minus the GI members (crtb200_sampling, set per context) + the rectangle list
 * the reference's schedulers would produce (RayTracer.cpp:114-202).  n_rects = 0 renders the whole image. */
typedef struct crtb200_options {
  uint32_t max_depth;    /* MAX_DEPTH, default 5           */
  float shadow_bias;     /* SHADOW_BIAS, default 1e-4f     */
  float reflection_bias; /* REFLECTION_BIAS, default 1e-4f */
  float refraction_bias; /* REFRACTION_BIAS, default 1e-4f */
  uint32_t n_rects;
  const crtb200_rect *rects;
  uint32_t traversal; /* 0 = DEFAULT: the reference's walk (KDTree.cpp:48-87, 127-166) minus the subtrees that provably  */
                      /*     cannot contribute (conservative culling with a per-mesh margin, DESIGN.md 3.6), long    */
                      /*     walks finished by a group of lanes (tail hand-off, DESIGN.md 3.8), shadow rays whose light */
                      /*     term is exactly zero answered without a walk (3.9).  Results are identical to the        */
                      /*     reference's: hit ids, t, float RGB, ray counts.                                          */
                      /* 1 = the reference's literal itinerary: every node whose box passes is visited, nothing is    */
                      /*     skipped or reordered (what count_work = 1 counts; the round-1 default).                  */
  uint32_t count_work; /* 0 = off; 1 = count node / triangle tests under the reference's visit-all rule (shadow  */
                       /* early termination disabled; same pixels) -- the figure the roofline arithmetic uses;  */
                       /* 2 = count the tests the production kernels really perform                             */
  /* tile sharding (multi-GPU): render only tile blocks b with b % shard_count == shard_index; 0/1 = all */
  uint32_t shard_index, shard_count;
  /* crtb200_render_device with shard_count > 1: 0 = write the shard's pixels compactly (a slab, for an NCCL gather +    */
  /* crtb200_assemble_shards); 1 = write them at their place in a FULL frame -- d_rgb_out / d_rgb8_out then usually    */
  /* point at the gathering rank's frame, mapped with crtb200_ipc_open: the store kernel does the transfer (NVLink)   */
  uint32_t shard_full_frame;
} crtb200_options;

/* Primary-ray closest hit, the record the parity gate compares (mesh index, mesh-local triangle index, t). */
typedef struct crtb200_hit {
  int32_t mesh; /* -1 = miss */
  int32_t triangle;
  float t;
} crtb200_hit;

typedef struct crtb200_stats {
  uint64_t rays_primary, rays_shadow, rays_reflection, rays_refraction; /* traced rays, SURVEY 8(d) definition */
  /* AABB / triangle tests per options.count_work, split by kernel: closest-hit (K2) and shadow (K3) */
  uint64_t node_tests_closest, triangle_tests_closest;
  uint64_t node_tests_shadow, triangle_tests_shadow;
  double device_ms;  /* CUDA-event time of the whole frame on the launching stream                          */
  double closest_ms; /* of which: closest-hit traversal launches (K2, all levels)                            */
  double shadow_ms;  /* of which: shadow any-hit + accumulate launches (K3)                                  */
  double total_ms;   /* host wall time of the call, copies included                                          */
  uint32_t kernel_launches;
  uint32_t levels;
  /* tail hand-off (DESIGN.md 3.8): walks finished one warp per ray by k_coop, and the part of closest_ms / shadow_ms  */
  /* spent there                                                                                                      */
  uint64_t handoff_closest, handoff_shadow;
  double coop_closest_ms, coop_shadow_ms;
  /* shadow rays (included in rays_shadow) that were answered without a walk because their light term is exactly zero  */
  /* whatever the visibility: surface turned away from the light, RayTracer.cpp:313-327 (DESIGN.md 3.9)                */
  uint64_t shadow_rays_zero_term;
} crtb200_stats;

typedef struct crtb200_ctx crtb200_ctx;

/* library / device */
uint32_t crtb200_abi_version(void);
const char *crtb200_last_error(void);
int crtb200_device_count(int *count);

const char *crtb200_last_error_ctx(const crtb200_ctx *ctx);

/* replaces: RayTracer::RayTracer(Scene&) resource acquisition (RayTracer.cpp:45-51) */
int crtb200_create(int device, crtb200_ctx **out);
/* The same on n GPUs of one node (SURVEY 8(b) "Proposed exports", 8(e)): replaces the std::thread bucket pool of
 * RayTracer::renderBucketsThreadpool (RayTracer.cpp:141-158) at device scale.  The context behaves like a single-GPU
 * one -- same calls, same results bit for bit -- but crtb200_upload_scene replicates the scene on every GPU and every
 * frame's 8x4-pixel tiles are dealt round-robin over the GPUs; each GPU stores its pixels straight into the frame on
 * device_ids[0] through peer-mapped memory (NVLink), from where the frame is returned.  A device id may repeat (several
 * tile shards on one GPU; used by the single-GPU tests). */
int crtb200_create_multi(const int *device_ids, int n, crtb200_ctx **out);
int crtb200_device_list(const crtb200_ctx *ctx, int *device_ids, int capacity, int *count);
int crtb200_destroy(crtb200_ctx *ctx);
/* device budget in bytes for the per-frame ray queues (default 16 GiB); frames that need more are chunked */
int crtb200_set_queue_budget(crtb200_ctx *ctx, uint64_t bytes);
/* chunks of a frame rendered concurrently on separate streams (default 2; 1 = strictly sequential kernels, which is
 * what the per-kernel timers closest_ms / shadow_ms of crtb200_stats require -- they read 0 otherwise) */
int crtb200_set_concurrency(crtb200_ctx *ctx, uint32_t chunks_in_flight);

/* The GI members of RenderOptions (RayTracer.h:25-50: USE_GI, GI_SAMPLE_SIZE, RAYS_PER_PIXEL, MONTE_CARLO_BIAS) and the
 * GI / supersampling branch of RayTracer::render and shootRay (RayTracer.cpp:90-104, 331-354; Vector.cpp:124-135), under
 * this project's reproducible sampling contract (DESIGN.md 3.10) instead of the reference's clock()-seeded rand():
 * Philox4x32-10 keyed by {seed, frame_index}, counters derived from the global pixel, the sample and the ray's place in
 * the ray tree, so a frame does not depend on chunking, tile shards or GPU count.  With use_gi = 0 every render call
 * renders exactly what it renders without this call (rays_per_pixel only matters with GI on, as in the reference). */
typedef struct crtb200_sampling {
  uint32_t use_gi;         /* USE_GI                                                                       */
  uint32_t gi_samples;     /* GI_SAMPLE_SIZE: diffuse bounce rays per diffuse hit (G), at most 1024         */
  uint32_t rays_per_pixel; /* RAYS_PER_PIXEL: jittered primary rays per pixel, averaged in sample order    */
  float monte_carlo_bias;  /* MONTE_CARLO_BIAS: diffuse ray origin = hit point + normal * bias             */
  uint32_t seed;           /* Philox key word 0                                                            */
  uint32_t frame_index;    /* Philox key word 1 (crtb200_render_frames: frame f uses frame_index + f)      */
} crtb200_sampling;

typedef struct crtb200_sampling_stats {
  uint64_t rays_diffuse; /* DiffuseRay rays traced by the last render (not part of crtb200_stats)          */
  uint32_t samples;      /* samples per pixel of the last render (1 with sampling off)                     */
  uint32_t reserved;
} crtb200_sampling_stats;

/* replaces: RenderOptions::USE_GI / GI_SAMPLE_SIZE / RAYS_PER_PIXEL / MONTE_CARLO_BIAS (RayTracer.h:25-50) as passed to
 * RayTracer::render.  Applies to every later render call of the context (like crtb200_set_concurrency); NULL or
 * use_gi = 0 turns sampling off.  CRTB200_ERR_ARG when rays_per_pixel == 0 with GI on or gi_samples > 1024.  A frame
 * whose ray tree (G^depth children per pixel) does not fit the queue budget fails with CRTB200_ERR_MEMORY. */
int crtb200_set_sampling(crtb200_ctx *ctx, const crtb200_sampling *sampling);
/* replaces: nothing in the reference (it counts no rays); the DiffuseRay count of RayTracer.cpp:331-354 */
int crtb200_last_sampling_stats(crtb200_ctx *ctx, crtb200_sampling_stats *stats);

/* Progressive sessions (DESIGN.md 3.10.1): a GI frame rendered in steps of samples, readable after any step, saved and
 * resumed.  None of these has a counterpart in the reference: RayTracer::render runs all RAYS_PER_PIXEL samples of a
 * pixel in one loop and keeps no running sum (RayTracer.cpp:90-104).  One session per context; it holds a persistent
 * per-pixel accumulator of 40 bytes per pixel on each GPU (that GPU's tile shard).  After steps totalling n samples,
 * crtb200_accum_read returns bit for bit what crtb200_render returns with the same camera and options and
 * rays_per_pixel = n, and the steps' ray counts (and, with count_work = 1, test counts) add up to that frame's.
 * Ordinary renders and crtb200_set_sampling between steps do not affect the session; crtb200_upload_scene,
 * crtb200_upload_geometry, crtb200_update_vertices_device and crtb200_destroy end it.  Every call but begin fails with CRTB200_ERR_STATE without a session. */

/* replaces: the per-pixel sample loop's set-up, RayTracer.cpp:90-104 (no counterpart: see above).  Snapshots camera,
 * options (the rects array is copied) and sampling (rays_per_pixel is ignored) and starts at 0 samples; a session in
 * progress ends.  CRTB200_ERR_ARG when use_gi = 0 or options->shard_count > 1 (several GPUs: crtb200_create_multi);
 * CRTB200_ERR_MEMORY when the accumulator does not fit on a device. */
int crtb200_accum_begin(crtb200_ctx *ctx, const crtb200_camera *camera, const crtb200_options *options,
                        const crtb200_sampling *sampling);
/* replaces: n_samples more iterations of the sample loop of RayTracer.cpp:90-104 (no counterpart: see above).  Renders
 * samples [done, done + n_samples) of every covered pixel exactly as a one-shot frame renders them, accumulating
 * S = S + c and Q = Q + c * c per channel in sample order.  stats (optional) and crtb200_last_stats /
 * crtb200_last_sampling_stats describe this step.  CRTB200_ERR_ARG when n_samples == 0. */
int crtb200_accum_step(crtb200_ctx *ctx, uint32_t n_samples, crtb200_stats *stats);
/* replaces: the division by RAYS_PER_PIXEL and the colorBuffer store after the loop, RayTracer.cpp:90-106 (no
 * counterpart: see above).  S / float(samples) into rgb_out / rgb8_out and sample 0's primary hit into hits_out, each
 * optional and laid out as in crtb200_render; pixels outside the session's rects keep the context's colour buffer, as
 * crtb200_render leaves them.  CRTB200_ERR_STATE at 0 samples.  Adds nothing to the statistics. */
int crtb200_accum_read(crtb200_ctx *ctx, float *rgb_out, uint8_t *rgb8_out, crtb200_hit *hits_out, uint32_t *samples_done);
/* replaces: nothing in the reference (see above).  sum_out / sumsq_out: S and Q, H*W*3 float32 row-major, 0 outside
 * the rects; hit0_out: H*W sample-0 hits (mesh = triangle = -1 for a miss and outside the rects; t bits as traced).
 * Each optional. */
int crtb200_accum_save(crtb200_ctx *ctx, float *sum_out, float *sumsq_out, crtb200_hit *hit0_out, uint32_t *samples_done);
/* replaces: nothing in the reference (see above).  The reverse of crtb200_accum_save, on a session begun with the same
 * camera, options and sampling: later steps continue as if the saved samples had been rendered here.  Pixels outside
 * the rects are not read.  CRTB200_ERR_ARG, and the session ends, when a hit names no triangle of the scene. */
int crtb200_accum_load(crtb200_ctx *ctx, const float *sum, const float *sumsq, const crtb200_hit *hit0,
                       uint32_t samples_done);
/* replaces: nothing in the reference (see above).  Ends the session and frees its accumulators; no-op without one. */
int crtb200_accum_end(crtb200_ctx *ctx);

/* Adaptive sessions (DESIGN.md 3.10.2): a progressive session in which each pixel stops sampling once its noise is
 * below a bound and later passes trace only the pixels still sampling.  After its n-th sample a pixel stops iff
 * n >= max_samples, or n >= min_samples and every channel's standard error of the mean is at most
 * abs_error + rel_error * |mean| (the rule of crt_s_adapt_stop in csrc/crt_sampling.h).  A stopped pixel never starts
 * again, so pixel p of a read is bit for bit crtb200_render's pixel p with rays_per_pixel = n_p, its own count. */
typedef struct crtb200_adaptive {
  uint32_t min_samples; /* >= 2 */
  uint32_t max_samples; /* >= min_samples */
  float abs_error;      /* >= 0 */
  float rel_error;      /* >= 0 */
} crtb200_adaptive;

typedef struct crtb200_progress {
  uint32_t passes;          /* passes run so far (samples of a plain session)                       */
  uint32_t reserved;
  uint64_t covered_pixels;  /* pixels inside the session's rects                                      */
  uint64_t active_pixels;   /* covered pixels still sampling (every covered pixel of a plain session) */
  uint64_t pixel_samples;   /* sum of the per-pixel sample counts (covered x passes when plain)       */
} crtb200_progress;

/* replaces: nothing in the reference.  crtb200_accum_begin with a stop rule, fixed for the session's life.  A step of n
 * runs n passes; pass s renders sample s of every active pixel as a one-shot frame renders it.  CRTB200_ERR_ARG, besides
 * crtb200_accum_begin's cases, when min_samples < 2, max_samples < min_samples or an error bound is negative or NaN. */
int crtb200_accum_begin_adaptive(crtb200_ctx *ctx, const crtb200_camera *camera, const crtb200_options *options,
                                 const crtb200_sampling *sampling, const crtb200_adaptive *adaptive);
/* replaces: nothing in the reference.  Passes, covered and active pixels and pixel-samples of the session (plain or
 * adaptive).  CRTB200_ERR_STATE without a session. */
int crtb200_accum_progress(crtb200_ctx *ctx, crtb200_progress *progress);
/* replaces: nothing in the reference.  counts_out: H*W per-pixel sample counts n_p, 0 outside the rects.
 * CRTB200_ERR_STATE without a session. */
int crtb200_accum_counts(crtb200_ctx *ctx, uint32_t *counts_out);
/* replaces: nothing in the reference.  crtb200_accum_load of an adaptive session with its counts map (H*W, as
 * crtb200_accum_counts writes it; NULL = passes everywhere).  A pixel is active iff n_p == passes and the rule does not
 * stop it at n_p.  CRTB200_ERR_ARG, and the session ends, when a count inside the rects exceeds passes or is 0 while
 * passes > 0; CRTB200_ERR_ARG when the session is plain and counts is not NULL. */
int crtb200_accum_load_counts(crtb200_ctx *ctx, const float *sum, const float *sumsq, const crtb200_hit *hit0,
                              const uint32_t *counts, uint32_t passes);

/* replaces: the data RayTracer keeps in `scene`, `boundingBox`, `accelerationStructure` (RayTracer.h:64-67).
 * Copies + re-lays-out everything to device SoA during the call (host flattener H1). */
int crtb200_upload_scene(crtb200_ctx *ctx, const crtb200_scene *scene);

/* replaces: TriangleKDTree(mesh, 25, 8) per mesh and ObjectKDTree(scene, 25, 4) (AccelerationStructure.h:10-11,
 * AccelerationStructure.cpp:12-50) plus crtb200_upload_scene: the KD trees are built on the device (DESIGN.md 3.11), one
 * replica per GPU of the context, node for node the trees of the host front end (csrc/frontend/crt_kdtree.cpp), and the
 * context is left exactly as crtb200_upload_scene leaves it given those trees.  The scene's n_mesh_nodes,
 * n_mesh_leaf_refs, n_top_nodes and n_top_leaf_refs must be 0 and their pointers NULL (else CRTB200_ERR_ARG); the tree
 * fields of crtb200_mesh are ignored; every other array is validated as by crtb200_upload_scene, with the same codes.
 * Ends a progressive session.  CRTB200_ERR_MEMORY when the build's scratch does not fit; it is freed before returning. */
int crtb200_upload_geometry(crtb200_ctx *ctx, const crtb200_scene *scene);

/* The trees of the last crtb200_upload_geometry, in the reference's numbering and the crtb200_scene layout. */
typedef struct crtb200_trees {
  uint32_t n_meshes, n_mesh_nodes, n_mesh_leaf_refs, n_top_nodes, n_top_leaf_refs;
  uint32_t reserved;
  uint64_t peak_scratch_bytes; /* the build's device scratch at its peak, on the first GPU of the context             */
  double build_ms;             /* CUDA-event time of the build on that GPU, from its first to its last kernel          */
  crtb200_mesh *meshes;        /* n_meshes records as uploaded, with first_node, n_nodes, first_leaf_ref, n_leaf_refs */
  crtb200_kdnode *mesh_nodes;  /* n_mesh_nodes                                                                      */
  uint32_t *mesh_leaf_refs;    /* n_mesh_leaf_refs mesh-local triangle indices                                      */
  crtb200_kdnode *top_nodes;   /* n_top_nodes                                                                       */
  uint32_t *top_leaf_refs;     /* n_top_leaf_refs mesh indices                                                      */
} crtb200_trees;
/* replaces: the AccelerationStructure a RayTracer holds (RayTracer.h:65), read back.  Fills the counts, then every
 * non-NULL array (sized from a call with NULL arrays).  CRTB200_ERR_STATE unless the context's trees were built on the
 * device: by crtb200_upload_geometry or crtb200_update_vertices_device. */
int crtb200_scene_trees(crtb200_ctx *ctx, crtb200_trees *trees);

/* The device scene state of one GPU of the context, as the traversal kernels read it (csrc/crt_device.cuh). */
typedef struct crtb200_scene_layout {
  uint32_t n_nodes, n_leaf_refs, n_top_refs, n_meshes;
  uint32_t top_begin, top_end; /* the top-level tree's node range                                              */
  uint32_t nested_ok;          /* 1 = culling and the tail hand-off are enabled for the scene (DESIGN.md 3.7) */
  uint32_t reserved;
  uint32_t *nodes;     /* 8 words per 32-byte node of the visiting-order array: min.xyz, a, max.xyz, b   */
  uint32_t *leaf_refs; /* global triangle ids                                                           */
  uint32_t *top_refs;  /* mesh ids                                                                      */
  uint32_t *meshes;    /* 5 words per mesh: node_begin, node_end, material, first_triangle, cull_margin bits */
} crtb200_scene_layout;
/* Test hook: copies GPU device_index's (0 = the first of the context) scene state to the host -- counts always, then
 * every non-NULL array -- so tests can compare crtb200_upload_geometry with crtb200_upload_scene bit for bit.
 * CRTB200_ERR_STATE without a scene. */
int crtb200_debug_scene_layout(crtb200_ctx *ctx, int device_index, crtb200_scene_layout *layout);

/* replaces: rebuilding a RayTracer for a scene whose vertices moved -- Mesh::Mesh's face and vertex normals
 * (Scene.cpp:5-30) and TriangleKDTree / ObjectKDTree (AccelerationStructure.cpp:12-50) -- from DEVICE memory
 * (DESIGN.md 3.14).  d_positions holds n_vertices * 3 float32 in device memory of the context's first GPU, 4-byte
 * aligned; n_vertices must be the uploaded scene's vertex count (0 for a scene without vertices: d_positions may then
 * be NULL).  Afterwards every GPU of the context holds exactly what crtb200_upload_geometry leaves for the uploaded
 * scene with these positions, its triangle and vertex normals as Mesh::Mesh computes them from these positions (in
 * binary32 without contraction), and everything else unchanged; crtb200_scene_trees then describes the new trees and
 * this build, whichever upload the scene came from.  The positions are read after the work already enqueued on `stream`
 * (a cudaStream_t, NULL = default), so renders, queries and shades enqueued there before finish first; work of this
 * context on other streams is the caller's to order, as for uploads.  Synchronous: on return every GPU holds the new
 * scene and d_positions may be overwritten.  Ends a progressive session.  Unlike an upload it keeps the colour buffer
 * (pixels outside a later render's rects keep their values, as across camera moves), and it leaves
 * crtb200_last_stats, the sampling stats and crtb200_last_query_stats alone.
 * CRTB200_ERR_STATE without a scene.  CRTB200_ERR_ARG: null positions with n_vertices > 0, positions not device memory
 * of the first GPU or misaligned, a wrong n_vertices.  CRTB200_ERR_MEMORY when the build's scratch does not fit.  A
 * failure after the update began leaves the context without a scene, as a failed crtb200_upload_geometry does. */
int crtb200_update_vertices_device(crtb200_ctx *ctx, const float *d_positions, uint32_t n_vertices, void *stream);
/* Test hook: GPU device_index's triangle records (n_triangles * 12 float32: p0.xyz, n.x, p1.xyz, n.y, p2.xyz, n.z, the
 * tri_geom layout) and vertex normals (n_vertices * 3), each optional.  CRTB200_ERR_STATE without a scene. */
int crtb200_debug_scene_geometry(crtb200_ctx *ctx, int device_index, float *tri_geom_out, float *vertex_normal_out);

/* replaces: RayTracer::render's scheduler switch + renderRectangle pixel loop (RayTracer.cpp:82-112,209-286).
 * rgb_out: H*W*3 float32 row-major, host memory, = the colorBuffer render() returns (RayTracer.cpp:297).  Pixels not
 * covered by options->rects keep the value of the previous render of this context (initially 0), like colorBuffer.
 * rgb8_out (optional): H*W*3 uint8, PPMColor quantisation (Color.cpp:12-16).
 * hits_out (optional): H*W primary-ray closest hits.   stats (optional). */
int crtb200_render(crtb200_ctx *ctx, const crtb200_camera *camera, const crtb200_options *options, float *rgb_out,
                   uint8_t *rgb8_out, crtb200_hit *hits_out, crtb200_stats *stats);

/* replaces: the animation loop body app/animation.cpp:24-38 (setCamera + render per frame), batched.
 * rgb_out / rgb8_out: n_frames consecutive frames. */
int crtb200_render_frames(crtb200_ctx *ctx, const crtb200_camera *cameras, uint32_t n_frames,
                          const crtb200_options *options, float *rgb_out, uint8_t *rgb8_out, crtb200_stats *stats);

/* Device-resident variant for callers that own device memory and a stream (multi-GPU gather, benchmarks):
 * d_rgb_out / d_rgb8_out are DEVICE pointers (either may be NULL), stream is a cudaStream_t (NULL = default).
 * Asynchronous: returns after enqueueing.  With tile sharding the output is the full-frame layout; pixels of
 * other shards are left untouched.  Stats are available through crtb200_last_stats after synchronisation. */
int crtb200_render_device(crtb200_ctx *ctx, const crtb200_camera *camera, const crtb200_options *options,
                          float *d_rgb_out, uint8_t *d_rgb8_out, void *stream);
int crtb200_last_stats(crtb200_ctx *ctx, crtb200_stats *stats);

/* Tile sharding for multi-GPU (one context per GPU, scene replicated; SURVEY 8(e)).  8x4-pixel tiles are dealt
 * round-robin: tile t belongs to shard t % shard_count.  With options->shard_count > 1 crtb200_render_device writes the
 * shard's pixels COMPACTLY into d_rgb_out (crtb200_shard_items(ctx, shard_count) x 3 floats, equal for all shards so the
 * slabs can be all-gathered / gathered with NCCL); d_rgb8_out must be NULL.  crtb200_assemble_shards scatters
 * shard_count consecutive slabs back into a full frame (and/or PPMColor bytes) on the gathering rank. */
int crtb200_shard_items(crtb200_ctx *ctx, uint32_t shard_count, uint32_t *items);
/* One process per GPU without a gather: the gathering rank exports its frame buffer (cudaIpcGetMemHandle, 64 bytes to
 * ship to the other ranks by any means), the others map it and render their shard straight into it with
 * options.shard_full_frame = 1.  Completion still needs a barrier between the ranks' streams (e.g. one tiny NCCL
 * all-reduce).  d_ptr must be the base of a cudaMalloc allocation of the exporting process. */
#define CRTB200_IPC_HANDLE_BYTES 64
int crtb200_ipc_alloc(int device, size_t bytes, void **d_ptr_out); /* a whole cudaMalloc allocation, exportable */
int crtb200_ipc_free(int device, void *d_ptr);
int crtb200_ipc_export(void *d_ptr, uint8_t handle_out[CRTB200_IPC_HANDLE_BYTES]);
int crtb200_ipc_open(int device, const uint8_t handle[CRTB200_IPC_HANDLE_BYTES], void **d_ptr_out);
int crtb200_ipc_close(int device, void *d_ptr);
int crtb200_assemble_shards(crtb200_ctx *ctx, const float *d_slabs, uint32_t shard_count, float *d_rgb_out,
                            uint8_t *d_rgb8_out, void *stream);

/* replaces: RayTracer::getRay + the re-normalisation of shootRay (RayTracer.cpp:61-80,420), exposed so the
 * parity tests can compare primary rays bit for bit.  rays_out: H*W*6 float32 (origin xyz, direction xyz), host;
 * crtb200_generate_rays_device copied back (synchronous). */
int crtb200_generate_rays(crtb200_ctx *ctx, const crtb200_camera *camera, float *rays_out);

/* replaces: RayTracer::getRay + the re-normalisation of shootRay (RayTracer.cpp:61-80,420) for every pixel, into caller
 * DEVICE memory: d_rays_out holds H*W*6 float32 (layout of crtb200_generate_rays) on the context's first GPU, 4-byte
 * aligned (else CRTB200_ERR_ARG; CRTB200_ERR_STATE without a scene).  Asynchronous on `stream` (a cudaStream_t, NULL = default), like
 * crtb200_render_device: a camera-ray batch for crtb200_trace_rays_device without a host round trip. */
int crtb200_generate_rays_device(crtb200_ctx *ctx, const crtb200_camera *camera, float *d_rays_out, void *stream);

/* A batch of caller-supplied rays in DEVICE memory of the context's first GPU (DESIGN.md 3.12). */
typedef struct crtb200_ray_batch {
  uint32_t n;                /* rays; n < 2^31 (CRTB200_ERR_ARG otherwise); 0 = nothing to do                          */
  uint32_t ray_type;         /* CRTB200_RAY_PRIMARY / _REFLECTION / _REFRACTION: closest hit; CRTB200_RAY_SHADOW: any hit */
  uint32_t traversal;        /* as crtb200_options.traversal: 0 = culled walk + tail hand-off, 1 = the literal itinerary */
  uint32_t count_work;       /* as crtb200_options.count_work (0 / 1 / 2)                                               */
  const float *rays;         /* n * 6 float32: origin xyz, direction xyz (the crtb200_trace_rays layout)                */
  const float *max_distance; /* n float32, shadow queries only                                                         */
  crtb200_hit *hits;         /* n records, closest-hit queries only (public numbering; miss: -1, -1, t = 0)            */
  uint8_t *occluded;         /* n bytes, shadow queries only                                                           */
} crtb200_ray_batch;

/* replaces: RayTracer::trace (RayTracer.cpp:453-458) and the non-GI RayTracer::hasIntersection (RayTracer.cpp:507-518)
 * -- KDTree::intersect, public in the reference -- for caller-supplied rays held in device memory.  Closest hit follows
 * RayTracer::trace, with the primary ray's back-face rule for CRTB200_RAY_PRIMARY only; a shadow query skips refractive
 * meshes and answers 1 iff some candidate has |P - o| <= max_distance.  Directions need not be unit length; NaN,
 * axis-parallel and zero directions behave as in the reference.  The answers do not depend on traversal, the GPU list or
 * the stream.  The rays are walked by the production traversal loop, with culling and tail hand-off for traversal 0.
 * On a crtb200_create_multi context the batch is split into contiguous ranges, one per GPU, each reading its rays and
 * writing its answers in the first GPU's memory through the peer mapping.  Asynchronous on `stream` (a cudaStream_t,
 * NULL = default), with the same rule about concurrent use of one context as crtb200_render_device.
 * CRTB200_ERR_ARG: a pointer the ray type needs is not device memory of the context's first GPU, rays / max_distance /
 * hits not 4-byte aligned, CRTB200_RAY_DIFFUSE or an unknown ray type, traversal or count_work, n >= 2^31.
 * CRTB200_ERR_STATE without a scene.  A query never changes crtb200_last_stats, the sampling stats, the colour buffer or
 * a progressive session; it keeps a small scratch per GPU, allocated on first use, until crtb200_destroy. */
int crtb200_trace_rays_device(crtb200_ctx *ctx, const crtb200_ray_batch *batch, void *stream);
/* replaces: nothing in the reference (it counts no rays).  After synchronisation: the last query's n in the rays_* field
 * of its type, node and triangle tests under its count_work, handoff_*, device_ms (its span on the caller's stream)
 * and kernel_launches, summed over the GPUs; every other field 0. */
int crtb200_last_query_stats(crtb200_ctx *ctx, crtb200_stats *stats);

/* replaces: RayTracer::trace (RayTracer.cpp:453-458) / RayTracer::hasIntersection (RayTracer.cpp:507-518) for caller-
 * supplied rays in HOST memory: stages them to the device, runs crtb200_trace_rays_device on the context's stream and
 * copies the answers back (synchronous).  rays: n*6 float32; ray_type: CRTB200_RAY_*; for shadow queries max_distance
 * holds n floats and occluded_out n bytes; for closest-hit queries hits_out holds n records.  traversal as in
 * crtb200_ray_batch (same answers either way). */
int crtb200_trace_rays(crtb200_ctx *ctx, const float *rays, uint32_t n, uint32_t ray_type, uint32_t traversal,
                       const float *max_distance, crtb200_hit *hits_out, uint8_t *occluded_out);

/* A batch of caller-supplied rays to shade, in DEVICE memory of the context's first GPU (DESIGN.md 3.13). */
typedef struct crtb200_shade_batch {
  uint32_t n;            /* rays; n < 2^31 (CRTB200_ERR_ARG otherwise); 0 = nothing to do                              */
  uint32_t ray_type;     /* CRTB200_RAY_PRIMARY (the primary ray's back-face rule) / _REFLECTION / _REFRACTION          */
  uint32_t traversal;    /* as crtb200_options.traversal                                                               */
  uint32_t count_work;   /* as crtb200_options.count_work                                                              */
  uint32_t max_depth;    /* MAX_DEPTH, <= 31                                                                           */
  float shadow_bias, reflection_bias, refraction_bias;
  uint32_t sample;       /* GI only: Philox counter word s of every ray of the batch                                   */
  uint32_t first_index;  /* GI only: ray i is "pixel" p = first_index + i (mod 2^32)                                   */
  const float *rays;     /* n * 6 float32: origin xyz, direction xyz (any length)                                      */
  float *rgb;            /* n * 3 float32, required                                                                    */
  crtb200_hit *hits;     /* n records, optional: the ray's own closest hit (public numbering; miss: -1, -1, t = 0)     */
} crtb200_shade_batch;

/* replaces: RayTracer::shootRay(ray, 0) (RayTracer.cpp:419-451) for a batch of caller-supplied rays: colour i is bit for
 * bit shootRay of ray i, including its normalisation of the direction (:420), under the batch's ray type, max_depth and
 * biases.  shootRay(ray, d) under MAX_DEPTH = M is shootRay(ray, 0) under MAX_DEPTH = M - d, so no depth argument
 * exists.  With the context's sampling on (crtb200_set_sampling) a ray is one GI sample: key {seed, frame_index},
 * pixel p = first_index + i, sample s = `sample`, root path key R(p, s, 0, 0).z -- the jittered camera ray of pixel p's
 * sample s shaded this way is that sample of a GI frame; rays_per_pixel is ignored.  Shading the once-normalised getRay
 * ray of each pixel with sampling off gives crtb200_render's frame.  The answers do not depend on traversal, the tail
 * hand-off, the queue budget, the GPU list, the stream, or how a GI batch is split into calls (given first_index).
 * The rays run through the frame pipeline (level loop, shadow pass, resolve).  On a crtb200_create_multi context the
 * batch is split into contiguous ranges, one per GPU, each writing its colours and hits into the first GPU's memory
 * through the peer mapping.  Asynchronous on `stream` (a cudaStream_t, NULL = default), with the same rule about
 * concurrent use of one context as crtb200_render_device.  After synchronisation crtb200_last_stats and
 * crtb200_last_sampling_stats describe this call: level-0 rays under the batch's type, shadow, secondary and diffuse
 * rays, tests under count_work, hand-offs, device_ms, kernel_launches.  The colour buffer, a progressive session and
 * crtb200_last_query_stats are untouched.
 * CRTB200_ERR_ARG: null batch / rays / rgb; rays, rgb or a non-null hits not device memory of the context's first GPU or
 * not 4-byte aligned; CRTB200_RAY_SHADOW, _DIFFUSE or an unknown ray type; traversal > 1, count_work > 2,
 * max_depth > 31, n >= 2^31.  CRTB200_ERR_STATE without a scene.  CRTB200_ERR_MEMORY when the ray tree does not fit
 * the queue budget, as for frames. */
int crtb200_shade_rays_device(crtb200_ctx *ctx, const crtb200_shade_batch *batch, void *stream);

/* Test hook: evaluates the device's (1 - cos)^5 routine (csrc/crt_powf5.h), the stand-in for glibc's
 * std::powf(x, 5) of RayTracer.cpp:407, on n host floats -- so the parity suite can check it bit for bit against libm. */
int crtb200_debug_powf5(crtb200_ctx *ctx, const float *x, uint32_t n, float *out);

#ifdef __cplusplus
}
#endif
#endif /* CRTB200_H */
