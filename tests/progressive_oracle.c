/* progressive_oracle.c -- TEST INFRASTRUCTURE ONLY.  CPU restatement of a progressive session's accumulator
 * (DESIGN.md section 3.10.1) on top of the GI restatement of tests/gi_oracle.c, which it compiles in unchanged: the
 * per-sample colours are that file's shoot_gi, formed exactly as crt_oracle_render_sampled forms them.
 * Build (tests/progressive_oracle.py): gcc -ffp-contract=off -fopenmp -I <package>/csrc, like gi_oracle.c.
 */
#include "gi_oracle.c"

/* The accumulator after smp->rays_per_pixel samples, over options->rects: sum = ((0 + c_0) + c_1) + ...,
 * sumsq = ((0 + c_0 * c_0) + c_1 * c_1) + ... per channel; pixels outside are left as they are. */
int crt_oracle_render_sums(const crtb200_scene *s, const crtb200_camera *cam, const crtb200_options *opt,
                           const crtb200_sampling *smp, float *sum, float *sumsq, int threads) {
  if (!s || !cam || !opt || !smp || !sum || !sumsq) return -1;
  crtb200_rect full = {0, 0, s->width, s->height};
  const crtb200_rect *rects = opt->n_rects ? opt->rects : &full;
  uint32_t n_rects = opt->n_rects ? opt->n_rects : 1;
  if (threads <= 0) threads = 1;
  for (uint32_t ri = 0; ri < n_rects; ri++) {
    const crtb200_rect rc = rects[ri];
    uint32_t row_limit = rc.row + rc.height < s->height ? rc.row + rc.height : s->height;
    uint32_t col_limit = rc.col + rc.width < s->width ? rc.col + rc.width : s->width;
#pragma omp parallel for schedule(dynamic, 1) num_threads(threads)
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
        v3 acc = V(0, 0, 0), acc2 = V(0, 0, 0);
        for (uint32_t sm = 0; sm < smp->rays_per_pixel; sm++) {
          g.s = sm;
          const crt_s_u4 q = crt_s_philox(g.p, sm, 0u, 0u, g.seed, g.frame);
          ray_t r = get_ray_at(s, cam, (float)col + crt_s_unit(q.x), (float)row + crt_s_unit(q.y));
          const v3 c = shoot_gi(&g, &r, 0, q.z);
          acc = vadd(acc, c);
          acc2 = vadd(acc2, V(c.x * c.x, c.y * c.y, c.z * c.z));
        }
        const size_t px = ((size_t)row * s->width + col) * 3;
        sum[px] = acc.x; sum[px + 1] = acc.y; sum[px + 2] = acc.z;
        sumsq[px] = acc2.x; sumsq[px + 1] = acc2.y; sumsq[px + 2] = acc2.z;
      }
    }
  }
  return 0;
}
