/* adaptive_oracle.c -- TEST INFRASTRUCTURE ONLY.  CPU restatement of an adaptive progressive session (DESIGN.md
 * section 3.10.2) on top of the GI restatement of tests/gi_oracle.c, which it compiles in unchanged: per-sample colours
 * are that file's shoot_gi, and the stop rule is crt_s_adapt_stop of crt_sampling.h, as the kernels compile it.
 * Build (tests/adaptive_oracle.py): gcc -ffp-contract=off -fopenmp -I <package>/csrc, like gi_oracle.c.
 */
#include "gi_oracle.c"

/* The accumulator after `passes` passes of an adaptive session over options->rects: each pixel takes samples 0, 1, ...
 * while the rule keeps it active, so sum / sumsq are ((0 + c_0) + c_1) + ... over its counts[p] samples.  Pixels outside
 * the rects are left as they are.  stats and *rays_diffuse are ACCUMULATED, over the samples taken. */
int crt_oracle_render_adaptive(const crtb200_scene *s, const crtb200_camera *cam, const crtb200_options *opt,
                               const crtb200_sampling *smp, const crtb200_adaptive *ad, uint32_t passes, float *sum,
                               float *sumsq, uint32_t *counts, crt_oracle_stats *stats, uint64_t *rays_diffuse,
                               int threads) {
  if (!s || !cam || !opt || !smp || !ad || !sum || !sumsq || !counts) return -1;
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
        float S[3] = {0, 0, 0}, Q[3] = {0, 0, 0};
        uint32_t n = 0;
        while (n < passes) {
          g.s = n;
          const crt_s_u4 q = crt_s_philox(g.p, n, 0u, 0u, g.seed, g.frame);
          ray_t r = get_ray_at(s, cam, (float)col + crt_s_unit(q.x), (float)row + crt_s_unit(q.y));
          const v3 c = shoot_gi(&g, &r, 0, q.z);
          S[0] = S[0] + c.x; S[1] = S[1] + c.y; S[2] = S[2] + c.z;
          Q[0] = Q[0] + c.x * c.x; Q[1] = Q[1] + c.y * c.y; Q[2] = Q[2] + c.z * c.z;
          n++;
          if (crt_s_adapt_stop(n, S, Q, ad->min_samples, ad->max_samples, ad->abs_error, ad->rel_error)) break;
        }
        const size_t px = (size_t)row * s->width + col;
        for (int k = 0; k < 3; k++) {
          sum[3 * px + k] = S[k];
          sumsq[3 * px + k] = Q[k];
        }
        counts[px] = n;
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

/* crt_s_adapt_stop for the known-answer tests */
int crt_oracle_adapt_stop(uint32_t n, const float *S, const float *Q, const crtb200_adaptive *ad) {
  return crt_s_adapt_stop(n, S, Q, ad->min_samples, ad->max_samples, ad->abs_error, ad->rel_error);
}
