#include "crt_raytracer.hpp"

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <stdexcept>
#include <thread>

namespace crt {

bool computeRectangles(unsigned width, unsigned height, RenderOptimization mode, unsigned bucketSize,
                       unsigned hardwareThreads, std::vector<crtb200_rect> &out) {
  out.clear();
  unsigned short rectangleCount = 1;  // `unsigned short rectangleCount`, RayTracer.h:75 (truncates bucket_size)
  unsigned short threadCount = 1;
  switch (mode) {  // RayTracer.cpp:209-286
    case NoOptimization:
    case AABB:
    case BVH:
      rectangleCount = 1;
      threadCount = 1;
      break;
    case Regions:
      rectangleCount = static_cast<unsigned short>(hardwareThreads);
      threadCount = static_cast<unsigned short>(hardwareThreads);
      break;
    default:
      rectangleCount = static_cast<unsigned short>(bucketSize);
      threadCount = static_cast<unsigned short>(hardwareThreads);
      break;
  }
  unsigned ny = static_cast<unsigned>(std::sqrt(rectangleCount));  // RayTracer.cpp:115-118,143-146
  if (ny == 0) ny = 1;
  unsigned nx = rectangleCount / ny;
  if (nx == 0) return false;  // the reference divides by zero here
  unsigned w = width / nx, h = height / ny;
  auto push = [&](unsigned row, unsigned col) {
    unsigned rowLimit = std::min(height, row + h), colLimit = std::min(width, col + w);  // RayTracer.cpp:84-85
    if (row < rowLimit && col < colLimit) out.push_back({row, col, colLimit - col, rowLimit - row});
  };
  if (mode == NoOptimization || mode == AABB || mode == BVH || mode == Regions) {
    if (threadCount == 1) {  // RayTracer.cpp:123-126
      push(0, 0);
      return true;
    }
    for (unsigned i = 0; i < threadCount; i++) push((i / nx) * h, (i * w) % width);  // RayTracer.cpp:130-134
    return true;
  }
  for (unsigned i = 0; i < rectangleCount; i++) push((i / nx) * h, (i * w) % width);  // RayTracer.cpp:150-152
  return true;
}

void writePPM(const std::string &path, const float *rgb, unsigned width, unsigned height) {
  FILE *f = std::fopen(path.c_str(), "wb");
  if (!f) throw std::runtime_error("cannot write " + path);
  std::fprintf(f, "P3\n%u %u\n255\n", width, height);
  static char lut[256][4];
  static int lutLen[256];
  static bool init = false;
  if (!init) {
    for (int i = 0; i < 256; i++) lutLen[i] = std::snprintf(lut[i], 4, "%d", i);
    init = true;
  }
  std::vector<char> line(size_t(width) * 12 + 2);
  for (unsigned row = 0; row < height; row++) {
    char *p = line.data();
    for (unsigned col = 0; col < width; col++) {
      const float *px = rgb + (size_t(row) * width + col) * 3;
      for (int k = 0; k < 3; k++) {
        // PPMColor: static_cast<unsigned short>(std::clamp(c, 0.0f, 1.0f) * 255)   Color.cpp:12-16
        float c = px[k];
        c = (c < 0.0f) ? 0.0f : ((1.0f < c) ? 1.0f : c);
        float scaled = c * 255;
        unsigned v = (scaled == scaled) ? static_cast<unsigned short>(scaled) : 0u;  // NaN -> 0 (x86 cvttss2si)
        if (v > 255) v = 255;
        for (int j = 0; j < lutLen[v]; j++) *p++ = lut[v][j];
        *p++ = (k < 2) ? ' ' : '\t';
      }
    }
    *p++ = '\n';
    std::fwrite(line.data(), 1, size_t(p - line.data()), f);
  }
  std::fclose(f);
}

RayTracer::RayTracer(Scene &scene_, int device) : scene(scene_), camera(scene_.camera) {
  buildFlatScene(scene, flat);
  colorBuffer.assign(size_t(scene.sceneSettings.image.width) * scene.sceneSettings.image.height * 3, 0.0f);
  if (device < 0) {
    // every visible GPU: the frame's tiles are dealt over them (crtb200_create_multi), like the reference deals its
    // buckets over hardware_concurrency() threads (RayTracer.cpp:141-158)
    int n = 0;
    if (crtb200_device_count(&n) != CRTB200_OK || n < 1)
      throw std::runtime_error(std::string("crtb200_device_count: ") + crtb200_last_error());
    std::vector<int> ids(static_cast<size_t>(n));
    for (int i = 0; i < n; i++) ids[static_cast<size_t>(i)] = i;
    if (crtb200_create_multi(ids.data(), n, &ctx) != CRTB200_OK)
      throw std::runtime_error(std::string("crtb200_create_multi: ") + crtb200_last_error());
  } else if (crtb200_create(device, &ctx) != CRTB200_OK) {
    throw std::runtime_error(std::string("crtb200_create: ") + crtb200_last_error());
  }
  if (crtb200_upload_scene(ctx, &flat.abi) != CRTB200_OK) {
    std::string msg = std::string("crtb200_upload_scene: ") + crtb200_last_error_ctx(ctx);
    crtb200_destroy(ctx);
    ctx = nullptr;
    throw std::runtime_error(msg);
  }
}

RayTracer::~RayTracer() {
  if (ctx) crtb200_destroy(ctx);
}

const std::vector<float> &RayTracer::renderFlat(const std::string &pathToImage, RenderOptions ro) {
  // The brute-force and single-AABB modes do not go through the KD trees in the reference: they use the linear scan of
  // RayTracer::trace / hasIntersection (RayTracer.cpp:459-505, 521-537), which breaks equal-t ties by scene order and
  // starts from minDistance = FLT_MAX (so NaN / inf candidates never win) -- not the tree modes' rules.  The B200 core
  // implements the tree path only, so those modes are refused rather than rendered with the wrong tie rules.
  switch (ro.optimization) {
    case BVH:
    case BVHBucketsThreadPool:
    case BVHBucketsQueue:
    case B200Wavefront:
      break;
    default:
      throw std::runtime_error("RayTracer::render: only the tree modes (BVH, BVHBucketsThreadPool, BVHBucketsQueue, B200Wavefront) "
                               "are rendered by the B200 core; the brute-force / AABB modes follow RayTracer::trace's linear-scan rules");
  }
  const unsigned W = scene.sceneSettings.image.width, H = scene.sceneSettings.image.height;
  std::vector<crtb200_rect> rects;
  if (!computeRectangles(W, H, ro.optimization, scene.sceneSettings.bucketSize,
                         std::thread::hardware_concurrency(), rects))
    throw std::runtime_error("RayTracer::render: bucket_size yields an empty rectangle grid");
  crtb200_camera cam;
  for (int i = 0; i < 3; i++) cam.position[i] = camera.getPosition()[i];
  for (int i = 0; i < 9; i++) cam.rotation[i] = camera.getRotationMatrix().m[i / 3][i % 3];
  crtb200_options opt{};
  opt.max_depth = ro.MAX_DEPTH;
  opt.shadow_bias = ro.SHADOW_BIAS;
  opt.reflection_bias = ro.REFLECTION_BIAS;
  opt.refraction_bias = ro.REFRACTION_BIAS;
  opt.n_rects = static_cast<uint32_t>(rects.size());
  opt.rects = rects.data();
  opt.traversal = ro.LITERAL_WALK ? 1u : 0u;
  // RenderOptions' GI members apply to this render only: the context's sampling state follows them on every call
  crtb200_sampling smp{};
  smp.use_gi = ro.USE_GI ? 1u : 0u;
  smp.gi_samples = ro.GI_SAMPLE_SIZE;
  smp.rays_per_pixel = ro.RAYS_PER_PIXEL;
  smp.monte_carlo_bias = ro.MONTE_CARLO_BIAS;
  smp.seed = ro.SEED;
  if (crtb200_set_sampling(ctx, &smp) != CRTB200_OK)
    throw std::runtime_error(std::string("crtb200_set_sampling: ") + crtb200_last_error_ctx(ctx));
  if (crtb200_render(ctx, &cam, &opt, colorBuffer.data(), nullptr, nullptr, &stats) != CRTB200_OK)
    throw std::runtime_error(std::string("crtb200_render: ") + crtb200_last_error_ctx(ctx));
  if (!pathToImage.empty()) writePPM(pathToImage, colorBuffer.data(), W, H);
  return colorBuffer;
}

std::vector<std::vector<Color>> RayTracer::render(const std::string &pathToImage, RenderOptions ro) {
  const std::vector<float> &flatBuf = renderFlat(pathToImage, ro);
  const unsigned W = scene.sceneSettings.image.width, H = scene.sceneSettings.image.height;
  std::vector<std::vector<Color>> out(H, std::vector<Color>(W));
  for (unsigned r = 0; r < H; r++)
    for (unsigned c = 0; c < W; c++) {
      const float *p = &flatBuf[(size_t(r) * W + c) * 3];
      out[r][c] = Color(p[0], p[1], p[2]);
    }
  return out;
}

void RayTracer::exportPPM(const std::string &pathToImage, const std::vector<std::vector<Color>> &buffer) {
  const unsigned W = scene.sceneSettings.image.width, H = scene.sceneSettings.image.height;
  std::vector<float> flatBuf(size_t(W) * H * 3, 0.0f);
  for (unsigned r = 0; r < H && r < buffer.size(); r++)
    for (unsigned c = 0; c < W && c < buffer[r].size(); c++) {
      flatBuf[(size_t(r) * W + c) * 3 + 0] = buffer[r][c].x;
      flatBuf[(size_t(r) * W + c) * 3 + 1] = buffer[r][c].y;
      flatBuf[(size_t(r) * W + c) * 3 + 2] = buffer[r][c].z;
    }
  writePPM(pathToImage, flatBuf.data(), W, H);
}

}  // namespace crt
