// extern "C" wrappers of the C++ front end (include/crtfront.h).
#include <cstdio>
#include <cstring>
#include <memory>
#include <string>

#include "../../../include/crtfront.h"
#include "crt_raytracer.hpp"

using namespace crt;

struct crtfe_scene {
  Scene scene;
  FlatScene flat, geometry;  // crtfe_scene_flatten / crtfe_scene_flatten_geometry, each built once
  bool flattened = false, geometry_flattened = false;
};
struct crtfe_tracer {
  std::unique_ptr<RayTracer> tracer;
  crtfe_scene *scene;
};

static thread_local std::string g_error;
static int fail(const std::string &m) {
  g_error = m;
  return -1;
}
#define CRTFE_TRY(body)              \
  try {                              \
    body;                            \
    return 0;                        \
  } catch (const std::exception &e) { \
    return fail(e.what());           \
  } catch (...) {                    \
    return fail("unknown error");    \
  }

static Camera toCamera(const crtb200_camera &c) {
  Camera cam(Vector(c.position[0], c.position[1], c.position[2]));
  for (int i = 0; i < 9; i++) cam.rotationMatrix.m[i / 3][i % 3] = c.rotation[i];
  return cam;
}
static void fromCamera(const Camera &cam, crtb200_camera &c) {
  for (int i = 0; i < 3; i++) c.position[i] = cam.position[i];
  for (int i = 0; i < 9; i++) c.rotation[i] = cam.rotationMatrix.m[i / 3][i % 3];
}

extern "C" {

const char *crtfe_last_error(void) { return g_error.c_str(); }

int crtfe_scene_load(const char *path, const char *folder, crtfe_scene **out) {
  if (!path || !out) return fail("null argument");
  CRTFE_TRY({
    auto s = std::make_unique<crtfe_scene>();
    s->scene = SceneParser::parseScene(path, folder ? folder : "");
    *out = s.release();
  })
}
// Appends n comma-separated numbers to a text file ("%.9g" for binary32 values: shortest text that round-trips through
// the reference's double-parsing GetFloat(), SceneParser.cpp; decimal for u32).  Used by the synthetic-scene writer: a
// 10 M-triangle .crtscene holds 45 M numbers.
static int append_numbers(const char *path, const void *data, uint64_t n, bool is_float) {
  if (!path || (!data && n)) return fail("null argument");
  FILE *f = std::fopen(path, "ab");
  if (!f) return fail(std::string("cannot open ") + path);
  std::string buf;
  buf.reserve(1 << 20);
  char tmp[40];
  for (uint64_t i = 0; i < n; i++) {
    int len;
    if (is_float) {
      len = std::snprintf(tmp, sizeof(tmp), "%.9g", (double)static_cast<const float *>(data)[i]);
    } else {
      uint32_t v = static_cast<const uint32_t *>(data)[i];
      char *e = tmp + sizeof(tmp), *q = e;
      do {
        *--q = (char)('0' + v % 10u);
        v /= 10u;
      } while (v);
      len = (int)(e - q);
      std::memmove(tmp, q, (size_t)len);
    }
    if (i) buf.push_back(',');
    buf.append(tmp, (size_t)len);
    if (buf.size() > (1u << 20) - 64) {
      std::fwrite(buf.data(), 1, buf.size(), f);
      buf.clear();
    }
  }
  std::fwrite(buf.data(), 1, buf.size(), f);
  const bool ok = std::fclose(f) == 0;
  return ok ? 0 : fail("write failed");
}
int crtfe_append_f32(const char *path, const float *values, uint64_t n) { return append_numbers(path, values, n, true); }
int crtfe_append_u32(const char *path, const uint32_t *values, uint64_t n) { return append_numbers(path, values, n, false); }

int crtfe_scene_free(crtfe_scene *s) {
  delete s;
  return 0;
}
int crtfe_scene_get_info(const crtfe_scene *s, crtfe_scene_info *info) {
  if (!s || !info) return fail("null argument");
  std::memset(info, 0, sizeof(*info));
  info->width = s->scene.sceneSettings.image.width;
  info->height = s->scene.sceneSettings.image.height;
  info->bucket_size = s->scene.sceneSettings.bucketSize;
  info->n_meshes = static_cast<uint32_t>(s->scene.objects.size());
  info->n_materials = static_cast<uint32_t>(s->scene.materials.size());
  info->n_textures = static_cast<uint32_t>(s->scene.textures.size());
  info->n_lights = static_cast<uint32_t>(s->scene.lights.size());
  info->n_triangles = s->scene.triangleCount();
  for (auto &o : s->scene.objects) info->n_vertices += o.positions.size();
  for (int i = 0; i < 3; i++) info->background[i] = s->scene.sceneSettings.sceneBackgroundColor[i];
  fromCamera(s->scene.camera, info->camera);
  return 0;
}
int crtfe_scene_flatten(crtfe_scene *s, uint32_t threads, const crtb200_scene **out, double *seconds) {
  if (!s || !out) return fail("null argument");
  CRTFE_TRY({
    if (!s->flattened) {
      buildFlatScene(s->scene, s->flat, threads);
      s->flattened = true;
    }
    *out = &s->flat.abi;
    if (seconds) *seconds = s->flat.buildSeconds;
  })
}
int crtfe_scene_flatten_geometry(crtfe_scene *s, const crtb200_scene **out, double *seconds) {
  if (!s || !out) return fail("null argument");
  CRTFE_TRY({
    if (!s->geometry_flattened) {
      buildFlatScene(s->scene, s->geometry, 1, false);
      s->geometry_flattened = true;
    }
    *out = &s->geometry.abi;
    if (seconds) *seconds = s->geometry.buildSeconds;
  })
}
int crtfe_rectangles(uint32_t w, uint32_t h, uint32_t mode, uint32_t bucket, uint32_t hw, crtb200_rect *out,
                     uint32_t capacity, uint32_t *count) {
  if (!count) return fail("null argument");
  std::vector<crtb200_rect> r;
  if (!computeRectangles(w, h, static_cast<RenderOptimization>(mode), bucket, hw, r)) return fail("empty rectangle grid");
  *count = static_cast<uint32_t>(r.size());
  if (out) {
    if (capacity < r.size()) return fail("rectangle capacity too small");
    std::memcpy(out, r.data(), r.size() * sizeof(crtb200_rect));
  }
  return 0;
}
int crtfe_camera_pan(crtb200_camera *c, float deg) {
  if (!c) return fail("null argument");
  Camera cam = toCamera(*c);
  cam.pan(deg);
  fromCamera(cam, *c);
  return 0;
}
int crtfe_camera_tilt(crtb200_camera *c, float deg) {
  if (!c) return fail("null argument");
  Camera cam = toCamera(*c);
  cam.tilt(deg);
  fromCamera(cam, *c);
  return 0;
}
int crtfe_camera_roll(crtb200_camera *c, float deg) {
  if (!c) return fail("null argument");
  Camera cam = toCamera(*c);
  cam.roll(deg);
  fromCamera(cam, *c);
  return 0;
}
int crtfe_camera_truck(crtb200_camera *c, const float d[3]) {
  if (!c || !d) return fail("null argument");
  Camera cam = toCamera(*c);
  cam.truck(Vector(d[0], d[1], d[2]));
  fromCamera(cam, *c);
  return 0;
}
int crtfe_write_ppm(const char *path, const float *rgb, uint32_t w, uint32_t h) {
  if (!path || !rgb) return fail("null argument");
  CRTFE_TRY(writePPM(path, rgb, w, h))
}
int crtfe_tracer_create(crtfe_scene *s, int device, crtfe_tracer **out) {
  if (!s || !out) return fail("null argument");
  CRTFE_TRY({
    auto t = std::make_unique<crtfe_tracer>();
    t->scene = s;
    t->tracer = std::make_unique<RayTracer>(s->scene, device);
    *out = t.release();
  })
}
int crtfe_tracer_free(crtfe_tracer *t) {
  delete t;
  return 0;
}
int crtfe_tracer_set_camera(crtfe_tracer *t, const crtb200_camera *c) {
  if (!t || !c) return fail("null argument");
  t->tracer->setCamera() = toCamera(*c);
  return 0;
}
int crtfe_tracer_get_camera(crtfe_tracer *t, crtb200_camera *c) {
  if (!t || !c) return fail("null argument");
  fromCamera(t->tracer->getCamera(), *c);
  return 0;
}
int crtfe_tracer_render(crtfe_tracer *t, const char *path, uint32_t mode, uint32_t maxDepth, uint32_t literalWalk,
                        float *rgbOut, crtb200_stats *stats) {
  if (!t) return fail("null argument");
  CRTFE_TRY({
    RenderOptions ro(static_cast<RenderOptimization>(mode), maxDepth, false);
    ro.LITERAL_WALK = literalWalk != 0;
    const std::vector<float> &buf = t->tracer->renderFlat(path ? path : "", ro);
    if (rgbOut) std::memcpy(rgbOut, buf.data(), buf.size() * sizeof(float));
    if (stats) *stats = t->tracer->lastStats();
  })
}
int crtfe_tracer_render_sampled(crtfe_tracer *t, const char *path, uint32_t mode, uint32_t maxDepth, uint32_t literalWalk,
                                uint32_t useGI, uint32_t giSamples, uint32_t raysPerPixel, float monteCarloBias, uint32_t seed,
                                float *rgbOut, crtb200_stats *stats) {
  if (!t) return fail("null argument");
  CRTFE_TRY({
    RenderOptions ro(static_cast<RenderOptimization>(mode), maxDepth, useGI != 0, giSamples, raysPerPixel);
    ro.MONTE_CARLO_BIAS = monteCarloBias;
    ro.LITERAL_WALK = literalWalk != 0;
    ro.SEED = seed;
    const std::vector<float> &buf = t->tracer->renderFlat(path ? path : "", ro);
    if (rgbOut) std::memcpy(rgbOut, buf.data(), buf.size() * sizeof(float));
    if (stats) *stats = t->tracer->lastStats();
  })
}
}
