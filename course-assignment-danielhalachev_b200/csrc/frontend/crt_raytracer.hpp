// RayTracer: the reference's renderer class (include/tracer/RayTracer.h:12-101) as a host-side mirror whose
// render() routes the per-pixel hot path to the B200 core through the C ABI (include/crtb200.h) instead of the
// bucket / thread-pool loop (src/RayTracer.cpp:82-202).  Same names, same argument meaning:
//     RayTracer tracer(scene);  tracer.setCamera().pan(30);  tracer.render("out.ppm", RenderOptions{...});
// There is no CPU rendering path in this class: if the CUDA core cannot run, render() throws.
#pragma once
#include <string>
#include <vector>

#include "crt_kdtree.hpp"
#include "crt_scene.hpp"

namespace crt {

// RayTracer.h:12-23 + the new enumerator.  The B200 core always traverses the KD trees (the reference's `Tree`
// bounding type, modes BVH*).  The brute-force / single-AABB enumerators exist for source compatibility and for
// computeRectangles, but render() refuses them: in the reference they take RayTracer::trace's linear scan
// (RayTracer.cpp:459-505), whose equal-t tie and NaN rules differ from the tree path's (SURVEY App. B-7).
enum RenderOptimization {
  NoOptimization,
  Regions,
  BucketsThreadPool,
  BucketsQueue,
  AABB,
  BucketsThreadPoolAABB,
  BucketsQueueAABB,
  BVH,
  BVHBucketsThreadPool,
  BVHBucketsQueue,
  B200Wavefront  // bucket grid of BVHBucketsThreadPool, rendered by the sm_100a wavefront pipeline
};

struct RenderOptions {  // RayTracer.h:25-50
  RenderOptimization optimization = B200Wavefront;
  bool USE_GI = false;  // GI + jittered supersampling under the reproducible sampling contract (crtb200_set_sampling)
  unsigned MAX_DEPTH = 5;
  unsigned GI_SAMPLE_SIZE = 2;
  unsigned RAYS_PER_PIXEL = 1;
  float SHADOW_BIAS = 1e-4;
  float REFLECTION_BIAS = 1e-4;
  float REFRACTION_BIAS = 1e-4;
  float MONTE_CARLO_BIAS = 1e-4;
  bool LITERAL_WALK = false;  // extension: crtb200_options::traversal = 1, the visit-all itinerary with nothing skipped (same results)
  unsigned SEED = 0;          // extension: Philox key of the GI / supersampling random numbers (crtb200_sampling::seed)
  explicit RenderOptions(RenderOptimization optimization = B200Wavefront, unsigned maxDepth = 5, bool useGI = false,
                         unsigned sampleSize = 2, unsigned raysPerPixel = 1, float shadowBias = 1e-4,
                         float reflectionBias = 1e-4, float refractionBias = 1e-4, float monteCarloBias = 1e-4)
      : optimization(optimization),
        USE_GI(useGI),
        MAX_DEPTH(maxDepth),
        GI_SAMPLE_SIZE(sampleSize),
        RAYS_PER_PIXEL(raysPerPixel),
        SHADOW_BIAS(shadowBias),
        REFLECTION_BIAS(reflectionBias),
        REFRACTION_BIAS(refractionBias),
        MONTE_CARLO_BIAS(monteCarloBias) {}
};

// Rectangle grid the reference's schedulers hand to renderRectangle (RayTracer.cpp:114-158), clipped like
// renderRectangle clips (RayTracer.cpp:84-85).  Returns false when the reference would divide by zero.
bool computeRectangles(unsigned width, unsigned height, RenderOptimization mode, unsigned bucketSize,
                       unsigned hardwareThreads, std::vector<crtb200_rect> &out);

// PPM writer byte-identical to RayTracer::exportPPM + PPMColor (RayTracer.cpp:540-552, Color.cpp:12-21).
void writePPM(const std::string &path, const float *rgb, unsigned width, unsigned height);

class RayTracer {
 public:
  // device >= 0: that GPU; device < 0 (default): every visible GPU, each frame split by tiles (crtb200_create_multi)
  explicit RayTracer(Scene &scene, int device = -1);
  ~RayTracer();
  RayTracer(const RayTracer &) = delete;
  RayTracer &operator=(const RayTracer &) = delete;

  const Camera &getCamera() const { return camera; }
  Camera &setCamera() { return camera; }
  // returns a copy of the colour buffer like the reference (RayTracer.cpp:297)
  std::vector<std::vector<Color>> render(const std::string &pathToImage, RenderOptions renderOptions = RenderOptions());
  // same render, no nested-vector copy: H*W*3 floats, valid until the next render
  const std::vector<float> &renderFlat(const std::string &pathToImage, RenderOptions renderOptions = RenderOptions());
  void exportPPM(const std::string &pathToImage, const std::vector<std::vector<Color>> &colorBuffer);
  const crtb200_stats &lastStats() const { return stats; }
  const FlatScene &flatScene() const { return flat; }
  crtb200_ctx *context() { return ctx; }

 private:
  const Scene &scene;
  Camera camera;
  FlatScene flat;
  crtb200_ctx *ctx = nullptr;
  std::vector<float> colorBuffer;  // persists across render() calls like RayTracer::colorBuffer (RayTracer.h:69)
  crtb200_stats stats{};
};

}  // namespace crt
