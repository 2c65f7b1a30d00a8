/* shade_oracle.c -- TEST INFRASTRUCTURE ONLY.  CPU counterpart of crtb200_shade_rays_device (DESIGN.md 3.13):
 * RayTracer::shootRay(ray, 0) for caller-supplied rays, unsampled (shoot_ray of oracle/crt_oracle.c) and under the
 * sampling contract (shoot_gi of tests/gi_oracle.c), plus the camera rays that turn a frame into such a batch.  It
 * compiles both files in unchanged.  Build (tests/shade_oracle.py): gcc -ffp-contract=off -fopenmp -I <package>/csrc.
 */
#include "gi_oracle.c"

static void oracle_hit(octx *c, const ray_t *r, crtb200_hit *ho) {
  ray_t pr = *r;
  pr.d = vnorm(pr.d); /* RayTracer.cpp:420 */
  octx tmp = *c;      /* (the hit record is not a traced ray: its tests are not counted) */
  hitinfo h = scene_intersect(&tmp, &pr);
  if (h.has) {
    ho->mesh = (int32_t)h.mesh;
    ho->triangle = (int32_t)(h.tri - c->s->meshes[h.mesh].first_triangle);
    ho->t = h.t;
  } else {
    ho->mesh = -1; ho->triangle = -1; ho->t = 0.0f;
  }
}

static ray_t load_ray(const float *rays, uint32_t i, uint32_t ray_type) {
  ray_t r;
  r.o = ld3(rays + 6 * (size_t)i);
  r.d = ld3(rays + 6 * (size_t)i + 3);
  r.type = (int)ray_type;
  return r;
}

#define SHADE_CHUNK 256u /* rays per OpenMP work item */

/* rgb[i] = shoot_ray(ray i of type ray_type, 0) under opt's max_depth and biases; hits[i] (optional) = the closest hit
 * of ray i with its direction normalised.  stats are ACCUMULATED into *stats. */
int crt_oracle_shade_rays(const crtb200_scene *s, const float *rays, uint32_t n, uint32_t ray_type,
                          const crtb200_options *opt, float *rgb, crtb200_hit *hits, crt_oracle_stats *stats, int threads) {
  if (!s || (n && (!rays || !rgb)) || !opt) return -1;
  uint64_t tot_rays[4] = {0, 0, 0, 0}, tot_nodes[2] = {0, 0}, tot_tris[2] = {0, 0};
  if (threads <= 0) threads = 1;
#pragma omp parallel for schedule(dynamic, 1) num_threads(threads) reduction(+ : tot_nodes[:2], tot_tris[:2], tot_rays[:4])
  for (uint32_t i0 = 0; i0 < n; i0 += SHADE_CHUNK) {
    octx c;
    memset(&c, 0, sizeof(c));
    c.s = s;
    c.max_depth = opt->max_depth;
    c.shadow_bias = opt->shadow_bias;
    c.reflection_bias = opt->reflection_bias;
    c.refraction_bias = opt->refraction_bias;
    for (uint32_t i = i0; i < n && i < i0 + SHADE_CHUNK; i++) {
      ray_t r = load_ray(rays, i, ray_type);
      if (hits) oracle_hit(&c, &r, &hits[i]);
      v3 col = shoot_ray(&c, &r, 0);
      rgb[3 * (size_t)i + 0] = col.x; rgb[3 * (size_t)i + 1] = col.y; rgb[3 * (size_t)i + 2] = col.z;
    }
    for (int k = 0; k < 2; k++) {
      tot_nodes[k] += c.node_tests[k];
      tot_tris[k] += c.tri_tests[k];
    }
    for (int k = 0; k < 4; k++) tot_rays[k] += c.rays[k];
  }
  if (stats) {
    stats->rays_primary += tot_rays[CRTB200_RAY_PRIMARY];
    stats->rays_shadow += tot_rays[CRTB200_RAY_SHADOW];
    stats->rays_reflection += tot_rays[CRTB200_RAY_REFLECTION];
    stats->rays_refraction += tot_rays[CRTB200_RAY_REFRACTION];
    stats->node_tests_closest += tot_nodes[0];
    stats->triangle_tests_closest += tot_tris[0];
    stats->node_tests_shadow += tot_nodes[1];
    stats->triangle_tests_shadow += tot_tris[1];
  }
  return 0;
}

/* shoot_gi per ray: pixel p = first_index + i (mod 2^32), sample s = `sample`, root path key R(p, s, 0, 0).z.  stats
 * and *rays_diffuse are ACCUMULATED. */
int crt_oracle_shade_rays_sampled(const crtb200_scene *s, const float *rays, uint32_t n, uint32_t ray_type,
                                  const crtb200_options *opt, const crtb200_sampling *smp, uint32_t sample,
                                  uint32_t first_index, float *rgb, crtb200_hit *hits, crt_oracle_stats *stats,
                                  uint64_t *rays_diffuse, int threads) {
  if (!s || (n && (!rays || !rgb)) || !opt || !smp) return -1;
  uint64_t tot_rays[4] = {0, 0, 0, 0}, tot_nodes[2] = {0, 0}, tot_tris[2] = {0, 0}, tot_diff = 0;
  if (threads <= 0) threads = 1;
#pragma omp parallel for schedule(dynamic, 1) num_threads(threads) reduction(+ : tot_nodes[:2], tot_tris[:2], tot_rays[:4], tot_diff)
  for (uint32_t i0 = 0; i0 < n; i0 += SHADE_CHUNK) {
    gctx g;
    memset(&g, 0, sizeof(g));
    g.c.s = s;
    g.c.max_depth = opt->max_depth;
    g.c.shadow_bias = opt->shadow_bias;
    g.c.reflection_bias = opt->reflection_bias;
    g.c.refraction_bias = opt->refraction_bias;
    g.seed = smp->seed;
    g.frame = smp->frame_index;
    g.gi_samples = smp->gi_samples;
    g.mc_bias = smp->monte_carlo_bias;
    g.s = sample;
    for (uint32_t i = i0; i < n && i < i0 + SHADE_CHUNK; i++) {
      g.p = first_index + i;
      ray_t r = load_ray(rays, i, ray_type);
      if (hits) oracle_hit(&g.c, &r, &hits[i]);
      const crt_s_u4 q = crt_s_philox(g.p, sample, 0u, 0u, g.seed, g.frame);
      v3 col = shoot_gi(&g, &r, 0, q.z);
      rgb[3 * (size_t)i + 0] = col.x; rgb[3 * (size_t)i + 1] = col.y; rgb[3 * (size_t)i + 2] = col.z;
    }
    for (int k = 0; k < 2; k++) {
      tot_nodes[k] += g.c.node_tests[k];
      tot_tris[k] += g.c.tri_tests[k];
    }
    for (int k = 0; k < 4; k++) tot_rays[k] += g.c.rays[k];
    tot_diff += g.rays_diffuse;
  }
  if (stats) {
    stats->rays_primary += tot_rays[CRTB200_RAY_PRIMARY];
    stats->rays_shadow += tot_rays[CRTB200_RAY_SHADOW];
    stats->rays_reflection += tot_rays[CRTB200_RAY_REFLECTION];
    stats->rays_refraction += tot_rays[CRTB200_RAY_REFRACTION];
    stats->node_tests_closest += tot_nodes[0];
    stats->triangle_tests_closest += tot_tris[0];
    stats->node_tests_shadow += tot_nodes[1];
    stats->triangle_tests_shadow += tot_tris[1];
  }
  if (rays_diffuse) *rays_diffuse += tot_diff;
  return 0;
}

static void store_ray(float *out, const ray_t *r) {
  out[0] = r->o.x; out[1] = r->o.y; out[2] = r->o.z; out[3] = r->d.x; out[4] = r->d.y; out[5] = r->d.z;
}

/* RayTracer::getRay of every pixel, row-major H*W*6: getRay's own normalisation only (shootRay adds the second) */
int crt_oracle_camera_rays(const crtb200_scene *s, const crtb200_camera *cam, float *rays_out) {
  if (!s || !cam || !rays_out) return -1;
  for (uint32_t row = 0; row < s->height; row++)
    for (uint32_t col = 0; col < s->width; col++) {
      const ray_t r = get_ray(s, cam, row, col);
      store_ray(rays_out + ((size_t)row * s->width + col) * 6, &r);
    }
  return 0;
}

/* the jittered getRay ray of sample `sample` of every pixel (crt_oracle_render_sampled's), row-major H*W*6 */
int crt_oracle_camera_rays_sampled(const crtb200_scene *s, const crtb200_camera *cam, const crtb200_sampling *smp,
                                   uint32_t sample, float *rays_out) {
  if (!s || !cam || !smp || !rays_out) return -1;
  for (uint32_t row = 0; row < s->height; row++)
    for (uint32_t col = 0; col < s->width; col++) {
      const crt_s_u4 q = crt_s_philox(row * s->width + col, sample, 0u, 0u, smp->seed, smp->frame_index);
      const ray_t r = get_ray_at(s, cam, (float)col + crt_s_unit(q.x), (float)row + crt_s_unit(q.y));
      store_ray(rays_out + ((size_t)row * s->width + col) * 6, &r);
    }
  return 0;
}
