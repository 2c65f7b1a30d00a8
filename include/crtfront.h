/* crtfront.h -- C entry points of the host front end (libcrtfront.so) for non-C++ callers (the Python test and
 * benchmark harness binds these with ctypes).  The front end itself is C++ and mirrors the reference's classes
 * (csrc/frontend/crt_scene.hpp, crt_raytracer.hpp); these wrappers expose exactly that API:
 *   SceneParser::parseScene (SceneParser.cpp:39-66)      -> crtfe_scene_load
 *   AccelerationStructure(scene) (AccelerationStructure.cpp:27-50) + flattening -> crtfe_scene_flatten
 *   flattening without the trees (built on the GPU by crtb200_upload_geometry) -> crtfe_scene_flatten_geometry
 *   RayTracer(scene) / setCamera / render / exportPPM (RayTracer.h:97-101) -> crtfe_tracer_*
 *   Camera::pan/tilt/roll/truck (Camera.cpp:33-70)       -> crtfe_camera_*
 * All functions return 0 on success, negative on error; crtfe_last_error() gives the message. */
#ifndef CRTFRONT_H
#define CRTFRONT_H

#include "crtb200.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct crtfe_scene crtfe_scene;
typedef struct crtfe_tracer crtfe_tracer;

typedef struct crtfe_scene_info {
  uint32_t width, height, bucket_size;
  uint32_t n_meshes, n_materials, n_textures, n_lights;
  uint64_t n_triangles, n_vertices;
  float background[3];
  crtb200_camera camera;
} crtfe_scene_info;

const char *crtfe_last_error(void);

int crtfe_scene_load(const char *path_to_scene, const char *scene_folder, crtfe_scene **out);
int crtfe_scene_free(crtfe_scene *scene);
int crtfe_scene_get_info(const crtfe_scene *scene, crtfe_scene_info *info);
/* builds the KD trees and the flattened arrays (idempotent); *out stays valid until crtfe_scene_free */
int crtfe_scene_flatten(crtfe_scene *scene, uint32_t threads, const crtb200_scene **out, double *build_seconds);
/* the same flattened arrays without the KD build, for crtb200_upload_geometry: tree counts 0, tree arrays NULL, the
 * meshes' tree fields 0 (idempotent; independent of crtfe_scene_flatten's result, which it leaves as it is) */
int crtfe_scene_flatten_geometry(crtfe_scene *scene, const crtb200_scene **out, double *seconds);

/* rectangle grid of the reference's schedulers (RayTracer.cpp:114-158); mode = RenderOptimization value (10 = B200) */
int crtfe_rectangles(uint32_t width, uint32_t height, uint32_t mode, uint32_t bucket_size, uint32_t hw_threads,
                     crtb200_rect *out, uint32_t capacity, uint32_t *count);

int crtfe_camera_pan(crtb200_camera *camera, float degrees);
int crtfe_camera_tilt(crtb200_camera *camera, float degrees);
int crtfe_camera_roll(crtb200_camera *camera, float degrees);
int crtfe_camera_truck(crtb200_camera *camera, const float direction[3]);

int crtfe_write_ppm(const char *path, const float *rgb, uint32_t width, uint32_t height);
/* scene-file writer helpers (synthetic workloads): append n comma-separated numbers to a text file, "%.9g" / decimal */
int crtfe_append_f32(const char *path, const float *values, uint64_t n);
int crtfe_append_u32(const char *path, const uint32_t *values, uint64_t n);

/* RayTracer mirror */
int crtfe_tracer_create(crtfe_scene *scene, int device, crtfe_tracer **out);
int crtfe_tracer_free(crtfe_tracer *tracer);
int crtfe_tracer_set_camera(crtfe_tracer *tracer, const crtb200_camera *camera);
int crtfe_tracer_get_camera(crtfe_tracer *tracer, crtb200_camera *camera);
/* RayTracer::render(pathToImage, RenderOptions{mode, max_depth, false}); rgb_out (optional) receives H*W*3 floats */
int crtfe_tracer_render(crtfe_tracer *tracer, const char *path_to_image, uint32_t mode, uint32_t max_depth,
                        uint32_t literal_walk, float *rgb_out, crtb200_stats *stats);
/* RayTracer::render(pathToImage, RenderOptions{mode, max_depth, use_gi, gi_samples, rays_per_pixel, ...,
 * monte_carlo_bias}) with RenderOptions::SEED = seed: GI and jittered supersampling under the sampling contract of
 * crtb200_set_sampling (frame_index 0) */
int crtfe_tracer_render_sampled(crtfe_tracer *tracer, const char *path_to_image, uint32_t mode, uint32_t max_depth,
                                uint32_t literal_walk, uint32_t use_gi, uint32_t gi_samples, uint32_t rays_per_pixel,
                                float monte_carlo_bias, uint32_t seed, float *rgb_out, crtb200_stats *stats);

#ifdef __cplusplus
}
#endif
#endif /* CRTFRONT_H */
