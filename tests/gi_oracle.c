/* gi_oracle.c -- TEST INFRASTRUCTURE ONLY.  CPU restatement of the sampling contract (DESIGN.md section 3.10): global
 * illumination and jittered supersampling, rendered recursively the way the reference's shootRay recursion does
 * (RayTracer.cpp:90-104, 331-354), with the random numbers of csrc/crt_sampling.h threaded through the recursion by
 * path key.  It is a straight extension of the restated reference in oracle/crt_oracle.c, which it compiles in
 * unchanged: the tree walks, triangle tests, texture lookups and the unsampled branches are that file's functions.
 * Build (tests/gi_oracle.py): gcc -ffp-contract=off -fopenmp -I <package>/csrc, like the oracle itself.
 */
#include "../oracle/crt_oracle.c"
#include "crt_sampling.h"

/* ObjectKDTree::checkForIntersection with useGI = true: refractive meshes are NOT skipped (AccelerationStructure.cpp:
 * 67-71 skips them only when !useGI).  scene_occluded skips them for CRTB200_RAY_SHADOW only; this type walks every
 * mesh and is still counted as a shadow ray. */
#define GI_SHADOW_RAY 5

typedef struct {
  octx c;
  uint32_t seed, frame, gi_samples, p, s;
  float mc_bias;
  uint64_t rays_diffuse;
} gctx;

static v3 shoot_gi(gctx *g, ray_t *r, unsigned depth, uint32_t key);

static uint32_t child_key(const gctx *g, uint32_t key, uint32_t slot) {
  return crt_s_child_key(g->seed, g->frame, g->p, g->s, key, slot);
}

/* RayTracer::calculateDiffusion with GI: D = the in-order light sum, then G diffuse bounces */
static v3 shade_diffuse_gi(gctx *g, const hitinfo *h, unsigned depth, uint32_t key) {
  octx *c = &g->c;
  const crtb200_scene *s = c->s;
  const crtb200_material *mat = &s->materials[s->meshes[h->mesh].material];
  const float PI = (float)M_PI;
  const v3 base = (mat->texture != CRTB200_INVALID)
                      ? texture_color(s, &s->textures[mat->texture], h->tri, h->u, h->v, 1.0f - h->u - h->v)
                      : ld3(mat->albedo);
  v3 D = V(0, 0, 0);
  for (uint32_t li = 0; li < s->n_lights; li++) {
    const crtb200_light *l = &s->lights[li];
    v3 ld = vsub(ld3(l->position), h->p);
    float dist = vlen(ld);
    float radius = vlen(ld);
    float area = 4 * radius * radius * PI;
    ld = vnorm(ld);
    float angle = stdmax(0.0f, vdot(ld, h->n));
    ray_t sr;
    sr.o = vadd(h->p, vscale(h->n, c->shadow_bias));
    sr.d = ld;
    sr.type = GI_SHADOW_RAY;
    if (!scene_occluded(c, &sr, dist)) {
      float direct = ((float)l->intensity / area * angle);
      D = vadd(D, sscale(direct, base));
    }
  }
  v3 S = V(0, 0, 0);
  const float n[3] = {h->n.x, h->n.y, h->n.z};
  for (uint32_t j = 0; j < g->gi_samples; j++) {
    float d[3];
    crt_s_diffuse_dir(g->seed, g->frame, g->p, g->s, key, j, n, d);
    ray_t cr;
    cr.o = vadd(h->p, vscale(h->n, g->mc_bias));
    cr.d = V(d[0], d[1], d[2]);
    cr.type = CRTB200_RAY_DIFFUSE;
    S = vadd(S, shoot_gi(g, &cr, depth + 1, child_key(g, key, j)));
  }
  const float g1 = (float)(g->gi_samples + 1u);
  return V((D.x + base.x * S.x) / g1, (D.y + base.y * S.y) / g1, (D.z + base.z * S.z) / g1);
}

/* shade_reflect / shade_refract of crt_oracle.c with the children's path keys (reflection slot 0, refraction slot 1) */
static v3 shade_reflect_gi(gctx *g, const ray_t *r, unsigned depth, const hitinfo *h, uint32_t key) {
  octx *c = &g->c;
  const crtb200_material *mat = &c->s->materials[c->s->meshes[h->mesh].material];
  ray_t rr;
  rr.o = vadd(h->p, vscale(h->n, c->reflection_bias));
  rr.d = vnorm(vreflect(r->d, h->n));
  rr.type = CRTB200_RAY_REFLECTION;
  v3 col = shoot_gi(g, &rr, depth + 1, child_key(g, key, 0));
  return vadd(V(0, 0, 0), V(mat->albedo[0] * col.x, mat->albedo[1] * col.y, mat->albedo[2] * col.z));
}

static v3 shade_refract_gi(gctx *g, const ray_t *r, unsigned depth, const hitinfo *h, uint32_t key) {
  octx *c = &g->c;
  const crtb200_material *mat = &c->s->materials[c->s->meshes[h->mesh].material];
  float eta1 = 1.0f, eta2 = mat->ior;
  v3 normal = h->n;
  float idn = vdot(r->d, normal);
  if (idn > 0) {
    float t = eta1; eta1 = eta2; eta2 = t;
    normal = sscale(-1, normal);
    idn = -idn;
  }
  float cos_a = -idn;
  float sin_a = sqrtf(stdmax(0.0f, 1 - cos_a * cos_a));
  ray_t rr;
  rr.o = vadd(h->p, vscale(normal, c->reflection_bias));
  rr.d = vnorm(vreflect(r->d, normal));
  rr.type = CRTB200_RAY_REFLECTION;
  v3 refl = shoot_gi(g, &rr, depth + 1, child_key(g, key, 0));
  float eta = eta1 / eta2;
  float sin_b = eta * sin_a;
  if (sin_b < 1.0f) {
    float r0 = powf((eta1 - eta2) / (eta1 + eta2), 2);
    float fresnel = r0 + (1 - r0) * powf(1.0f - cos_a, 5);
    float cos_b = sqrtf(stdmax(0.0f, 1 - sin_b * sin_b));
    v3 dir = vsub(sscale(eta, vadd(r->d, sscale(cos_a, normal))), sscale(cos_b, normal));
    ray_t tr;
    tr.o = vsub(h->p, vscale(normal, c->refraction_bias));
    tr.d = vnorm(dir);
    tr.type = CRTB200_RAY_REFRACTION;
    v3 refr = shoot_gi(g, &tr, depth + 1, child_key(g, key, 1));
    return vadd(sscale(fresnel, refl), sscale(1 - fresnel, refr));
  }
  return refl;
}

/* shoot_ray with the path key; diffuse directions already carry shootRay's second normalisation (crt_sampling.h) */
static v3 shoot_gi(gctx *g, ray_t *r, unsigned depth, uint32_t key) {
  octx *c = &g->c;
  v3 bg = ld3(c->s->background);
  if (r->type != CRTB200_RAY_DIFFUSE) r->d = vnorm(r->d);
  if (depth > c->max_depth) return bg;
  if (r->type == CRTB200_RAY_DIFFUSE) g->rays_diffuse++;
  hitinfo h = scene_intersect(c, r);
  if (!h.has) return bg;
  switch (c->s->materials[c->s->meshes[h.mesh].material].type) {
    case CRTB200_MAT_DIFFUSE: return shade_diffuse_gi(g, &h, depth, key);
    case CRTB200_MAT_REFLECTIVE: return shade_reflect_gi(g, r, depth, &h, key);
    case CRTB200_MAT_REFRACTIVE: return shade_refract_gi(g, r, depth, &h, key);
    default: return bg;
  }
}

/* RayTracer::getRay at pixel position (x, y) = (col + jitter, row + jitter) */
static ray_t get_ray_at(const crtb200_scene *s, const crtb200_camera *cam, float x, float y) {
  x = x / (float)s->width;
  y = y / (float)s->height;
  x = (2.0f * x) - 1.0f;
  y = 1.0f - (2.0f * y);
  x = x * ((float)s->width / (float)s->height);
  v3 d = V(x, y, -1.0);
  const float *m = cam->rotation;
  v3 dr = V(d.x * m[0] + d.y * m[3] + d.z * m[6], d.x * m[1] + d.y * m[4] + d.z * m[7],
            d.x * m[2] + d.y * m[5] + d.z * m[8]);
  ray_t r;
  r.o = ld3(cam->position);
  r.d = vnorm(dr);
  r.type = CRTB200_RAY_PRIMARY;
  return r;
}

/* The sampled frame over options->rects: pixel = (((0 + c_0) + c_1) + ...) / float(spp); hits = sample 0's primary
 * hit.  stats are ACCUMULATED into *stats and *rays_diffuse. */
int crt_oracle_render_sampled(const crtb200_scene *s, const crtb200_camera *cam, const crtb200_options *opt,
                              const crtb200_sampling *smp, float *rgb, crtb200_hit *hits, crt_oracle_stats *stats,
                              uint64_t *rays_diffuse, int threads) {
  if (!s || !cam || !opt || !smp || !rgb || smp->rays_per_pixel == 0) return -1;
  crtb200_rect full = {0, 0, s->width, s->height};
  const crtb200_rect *rects = opt->n_rects ? opt->rects : &full;
  uint32_t n_rects = opt->n_rects ? opt->n_rects : 1;
  uint64_t tot_rays[4] = {0, 0, 0, 0}, tot_nodes[2] = {0, 0}, tot_tris[2] = {0, 0}, tot_diff = 0;
  if (threads <= 0) threads = 1;
  for (uint32_t ri = 0; ri < n_rects; ri++) {
    const crtb200_rect rc = rects[ri];
    uint32_t row_limit = rc.row + rc.height < s->height ? rc.row + rc.height : s->height;
    uint32_t col_limit = rc.col + rc.width < s->width ? rc.col + rc.width : s->width;
#pragma omp parallel for schedule(dynamic, 1) num_threads(threads) reduction(+ : tot_nodes[:2], tot_tris[:2], tot_rays[:4], tot_diff)
    for (uint32_t row = rc.row; row < row_limit; row++) {
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
      for (uint32_t col = rc.col; col < col_limit; col++) {
        g.p = row * s->width + col;
        v3 acc = V(0, 0, 0);
        for (uint32_t sm = 0; sm < smp->rays_per_pixel; sm++) {
          g.s = sm;
          const crt_s_u4 q = crt_s_philox(g.p, sm, 0u, 0u, g.seed, g.frame);
          ray_t r = get_ray_at(s, cam, (float)col + crt_s_unit(q.x), (float)row + crt_s_unit(q.y));
          if (hits && sm == 0) {
            ray_t pr = r;
            pr.d = vnorm(pr.d);
            octx tmp = g.c;
            hitinfo h = scene_intersect(&tmp, &pr);
            crtb200_hit *ho = &hits[(size_t)row * s->width + col];
            if (h.has) {
              ho->mesh = (int32_t)h.mesh;
              ho->triangle = (int32_t)(h.tri - s->meshes[h.mesh].first_triangle);
              ho->t = h.t;
            } else {
              ho->mesh = -1; ho->triangle = -1; ho->t = 0.0f;
            }
          }
          acc = vadd(acc, shoot_gi(&g, &r, 0, q.z));
        }
        const float n = (float)smp->rays_per_pixel;
        float *px = rgb + ((size_t)row * s->width + col) * 3;
        px[0] = acc.x / n; px[1] = acc.y / n; px[2] = acc.z / n;
      }
      for (int k = 0; k < 2; k++) {
        tot_nodes[k] += g.c.node_tests[k];
        tot_tris[k] += g.c.tri_tests[k];
      }
      for (int k = 0; k < 4; k++) tot_rays[k] += g.c.rays[k];
      tot_diff += g.rays_diffuse;
    }
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

/* test hooks: the shared header's Philox, tangent frame and diffuse direction */
void crt_oracle_philox(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]) {
  const crt_s_u4 r = crt_s_philox(ctr[0], ctr[1], ctr[2], ctr[3], key[0], key[1]);
  out[0] = r.x; out[1] = r.y; out[2] = r.z; out[3] = r.w;
}
float crt_oracle_unit(uint32_t u) { return crt_s_unit(u); }
void crt_oracle_tangent_frame(const float n[3], float t[3], float b[3]) { crt_s_frame(n, t, b); }
/* n_dirs directions of diffuse slot k for keys key0, key0 + 1, ... (pixel p, sample s) */
void crt_oracle_diffuse_dirs(uint32_t seed, uint32_t frame, uint32_t p, uint32_t s, uint32_t key0, uint32_t k,
                             const float n[3], uint32_t n_dirs, float *out) {
  for (uint32_t i = 0; i < n_dirs; i++) crt_s_diffuse_dir(seed, frame, p, s, key0 + i, k, n, out + 3 * (size_t)i);
}
