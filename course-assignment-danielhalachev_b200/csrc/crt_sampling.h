/* crt_sampling.h -- the sampling contract of global illumination and jittered supersampling (DESIGN.md section 3.10),
 * shared by the CUDA core and the CPU oracle so that both form every sampled value with the same operations in the
 * same order.  This header IS the specification of the operation order.
 *
 *   R(p, s, K, w)   Philox4x32-10 (Salmon et al., "Parallel random numbers: as easy as 1, 2, 3", SC 2011) with
 *                   counter {p, s, K, w} and key {seed, frame_index}: p = global pixel index row * W + col, s = sample
 *                   index, K = ray-tree path key, w = slot / try word
 *   unit(u)         (float)(u >> 8) * 2^-24: exact, in [0, 1)
 *   crt_s_diffuse_dir  cosine-weighted hemisphere direction around N (Malley's method: a uniform point of the unit disk
 *                   by rejection, lifted to the hemisphere) in the tangent frame of Duff et al. 2017, "Building an
 *                   orthonormal basis, revisited" -- built from + - * / sqrt copysign only, so host and device agree
 *                   bit for bit without a shared trig polynomial
 *
 * Device: the round-to-nearest intrinsics, never contracted.  Host: plain binary32 arithmetic; the including
 * translation unit must be compiled with -ffp-contract=off (the oracle's Makefile and the test build do).
 */
#ifndef CRT_SAMPLING_H
#define CRT_SAMPLING_H
#include <stdint.h>

#ifdef __CUDA_ARCH__
#define CRT_S_HD __device__ __forceinline__
#define CRT_S_MUL(a, b) __fmul_rn((a), (b))
#define CRT_S_ADD(a, b) __fadd_rn((a), (b))
#define CRT_S_SUB(a, b) __fsub_rn((a), (b))
#define CRT_S_DIV(a, b) __fdiv_rn((a), (b))
#define CRT_S_SQRT(a) __fsqrt_rn(a)
#define CRT_S_MULHI(a, b) __umulhi((a), (b))
#else
#include <math.h>
#define CRT_S_HD static inline
#define CRT_S_MUL(a, b) ((a) * (b))
#define CRT_S_ADD(a, b) ((a) + (b))
#define CRT_S_SUB(a, b) ((a) - (b))
#define CRT_S_DIV(a, b) ((a) / (b))
#define CRT_S_SQRT(a) sqrtf(a)
#define CRT_S_MULHI(a, b) ((uint32_t)(((uint64_t)(a) * (uint64_t)(b)) >> 32))
#endif

/* tries of the disk rejection loop; (k + 1) + (t << 24) keeps the slot in the low 24 bits of the word */
#define CRT_S_DISK_TRIES 256u

typedef struct crt_s_u4 {
  uint32_t x, y, z, w;
} crt_s_u4;

/* Philox4x32-10: ten rounds, the key bumped by the Weyl constants between rounds */
CRT_S_HD crt_s_u4 crt_s_philox(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1) {
  for (int i = 0; i < 10; i++) {
    if (i) {
      k0 += 0x9E3779B9u;
      k1 += 0xBB67AE85u;
    }
    const uint32_t hi0 = CRT_S_MULHI(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    const uint32_t hi1 = CRT_S_MULHI(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    c0 = hi1 ^ c1 ^ k0;
    c1 = lo1;
    c2 = hi0 ^ c3 ^ k1;
    c3 = lo0;
  }
  crt_s_u4 r;
  r.x = c0;
  r.y = c1;
  r.z = c2;
  r.w = c3;
  return r;
}

CRT_S_HD float crt_s_unit(uint32_t u) { return CRT_S_MUL((float)(u >> 8), 0x1p-24f); }

/* key of child slot k of the ray-tree node with key K (reflection 0, refraction 1, diffuse sample j = j) */
CRT_S_HD uint32_t crt_s_child_key(uint32_t seed, uint32_t frame, uint32_t p, uint32_t s, uint32_t K, uint32_t k) {
  return crt_s_philox(p, s, K, k + 1u, seed, frame).x;
}

/* Vector::normalize (Vector.cpp:97-106): (x*x + y*y) + z*z, sqrt, 1 / l, scale; a zero vector is returned as is */
CRT_S_HD void crt_s_normalize(float *x, float *y, float *z) {
  float l = CRT_S_SQRT(CRT_S_ADD(CRT_S_ADD(CRT_S_MUL(*x, *x), CRT_S_MUL(*y, *y)), CRT_S_MUL(*z, *z)));
  if (l == 0.0f) return;
  l = CRT_S_DIV(1.0f, l);
  *x = CRT_S_MUL(*x, l);
  *y = CRT_S_MUL(*y, l);
  *z = CRT_S_MUL(*z, l);
}

/* Duff et al. 2017, listing 3: T, B with {T, B, N} orthonormal for unit N (N.z = -0.0 takes the negative branch) */
CRT_S_HD void crt_s_frame(const float n[3], float t[3], float b[3]) {
  const float sign = copysignf(1.0f, n[2]);
  const float a = CRT_S_DIV(-1.0f, CRT_S_ADD(sign, n[2]));
  const float bb = CRT_S_MUL(CRT_S_MUL(n[0], n[1]), a);
  t[0] = CRT_S_ADD(1.0f, CRT_S_MUL(CRT_S_MUL(CRT_S_MUL(sign, n[0]), n[0]), a));
  t[1] = CRT_S_MUL(sign, bb);
  t[2] = CRT_S_MUL(-sign, n[0]);
  b[0] = bb;
  b[1] = CRT_S_ADD(sign, CRT_S_MUL(CRT_S_MUL(n[1], n[1]), a));
  b[2] = -n[1];
}

/* The point (a, b) of the unit disk for diffuse slot k of node K: the first try t with a*a + b*b < 1, else (0, 0) */
CRT_S_HD void crt_s_disk(uint32_t seed, uint32_t frame, uint32_t p, uint32_t s, uint32_t K, uint32_t k, float *a_out,
                         float *b_out) {
  float a = 0.0f, b = 0.0f;
  for (uint32_t t = 0; t < CRT_S_DISK_TRIES; t++) {
    const crt_s_u4 r = crt_s_philox(p, s, K, (k + 1u) + (t << 24), seed, frame);
    const float ta = CRT_S_SUB(CRT_S_MUL(2.0f, crt_s_unit(r.y)), 1.0f);
    const float tb = CRT_S_SUB(CRT_S_MUL(2.0f, crt_s_unit(r.z)), 1.0f);
    if (CRT_S_ADD(CRT_S_MUL(ta, ta), CRT_S_MUL(tb, tb)) < 1.0f) {
      a = ta;
      b = tb;
      break;
    }
  }
  *a_out = a;
  *b_out = b;
}

/* Direction of diffuse slot k of node K at a hit with (unflipped) shading normal n:
 *   z = sqrt(1 - (a*a + b*b)),  d = normalize(normalize((a*T + b*B) + z*N))  (the second normalisation is shootRay's)
 * A NaN normal gives a NaN direction. */
CRT_S_HD void crt_s_diffuse_dir(uint32_t seed, uint32_t frame, uint32_t p, uint32_t s, uint32_t K, uint32_t k,
                                const float n[3], float d[3]) {
  float a, b, t[3], bt[3];
  crt_s_disk(seed, frame, p, s, K, k, &a, &b);
  const float z = CRT_S_SQRT(CRT_S_SUB(1.0f, CRT_S_ADD(CRT_S_MUL(a, a), CRT_S_MUL(b, b))));
  crt_s_frame(n, t, bt);
  for (int i = 0; i < 3; i++) d[i] = CRT_S_ADD(CRT_S_ADD(CRT_S_MUL(a, t[i]), CRT_S_MUL(b, bt[i])), CRT_S_MUL(z, n[i]));
  crt_s_normalize(&d[0], &d[1], &d[2]);
  crt_s_normalize(&d[0], &d[1], &d[2]);
}

/* Stop rule of adaptive sessions (DESIGN.md section 3.10.2), evaluated after a pixel's n-th sample with its running
 * sums S, Q (per channel, in sample order), in this order:
 *   nf = (float)n ; m_c = S_c / nf ; v_c = (Q_c - S_c * m_c) / (nf - 1) ; v_c = (v_c > 0) ? v_c : 0
 *   e_c = sqrt(v_c / nf) ; tol_c = abs_error + rel_error * fabsf(m_c)
 *   stop  iff  n >= max_samples  ||  (n >= min_samples && e_0 <= tol_0 && e_1 <= tol_1 && e_2 <= tol_2)
 * min_samples >= 2, so nf - 1 >= 1.  A NaN mean makes tol_c NaN and every comparison false: a pixel with a NaN sample
 * never stops early and samples up to max_samples. */
CRT_S_HD int crt_s_adapt_stop(uint32_t n, const float S[3], const float Q[3], uint32_t min_samples, uint32_t max_samples,
                              float abs_error, float rel_error) {
  if (n >= max_samples) return 1;
  if (n < min_samples) return 0;
  const float nf = (float)n;
  for (int c = 0; c < 3; c++) {
    const float m = CRT_S_DIV(S[c], nf);
    float v = CRT_S_DIV(CRT_S_SUB(Q[c], CRT_S_MUL(S[c], m)), CRT_S_SUB(nf, 1.0f));
    v = (v > 0.0f) ? v : 0.0f;
    const float e = CRT_S_SQRT(CRT_S_DIV(v, nf));
    const float tol = CRT_S_ADD(abs_error, CRT_S_MUL(rel_error, fabsf(m)));
    if (!(e <= tol)) return 0;
  }
  return 1;
}
#endif /* CRT_SAMPLING_H */
