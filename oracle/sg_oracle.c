/*
 * oracle/sg_oracle.c — CPU restatement of the spherical-Gaussian specular shade
 * (reference extensions/sgutils/sg.cu:27-76 forward, :78-175 backward).
 *
 * TEST INFRASTRUCTURE ONLY (see oracle/README.md).  Pinned on the GPU against recorded outputs of the
 * reference's own kernels rebuilt into oracle/_ref/sgutilslib (tests/golden/ref_kernels_sg.npz);
 * the reference ships no CPU kernel and no test vectors for this op (SURVEY.md §4).
 *
 * Per (batch n, Gaussian d):  integral[n,d,:] = sum_{l < n_lights[n]} light_values[n,l,:] * w
 *   ldir = normalize(light_pts[n,l] - prim_pts[n,d]) ; cos = dot(ldir, lobe_dir)
 *   w_type 0: exp(-.5 (acos(clamp cos)/s)^2) / (s * 3.03352966508)     sg.cu:57-59
 *   w_type 1: exp(-.5 (acos(clamp cos)/s)^2)                           sg.cu:60-62
 *   w_type 2: exp((clamp cos - 1)/s) / (s * 2pi)                       sg.cu:63-65
 *   w_type 3: exp((clamp cos - 1)/s)                                   sg.cu:66-68
 * Backward quirks kept (SURVEY.md Appendix B): derivative of acos uses the UNclamped cosine for the
 * in-range test and substitutes -20 at |cos|>=1 (sg.cu:129,139); no gradient to prim_pts/light_pts.
 * grad_light_values (optional, may be NULL) is accumulated (+=) like the reference's atomicAdd.
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>

#define ORC_API __attribute__((visibility("default")))

static const float TWOPI = 6.28318530718f;
static const float INV2PI = 0.15915494309f;
static const float SQRT2PI23 = 3.03352966508f;
static const float INVSQRT2PI23 = 0.32964899322f;

static inline float sq(float v) { return v * v; }
static inline float clampf(float v, float lo, float hi) { return fminf(fmaxf(v, lo), hi); }

ORC_API void orc_sg_fwd(int N, int D, int L, const float* lobe_dirs, const float* lobe_sigmas,
                        const float* light_values, const float* light_pts, const float* prim_pts,
                        const int32_t* n_lights, float* integral, int w_type) {
#pragma omp parallel for collapse(2) schedule(static)
  for (int n = 0; n < N; ++n)
    for (int d = 0; d < D; ++d) {
      const size_t o = (size_t)n * D + d;
      const float dx = lobe_dirs[3 * o], dy = lobe_dirs[3 * o + 1], dz = lobe_dirs[3 * o + 2];
      const float sigma = lobe_sigmas[o];
      const float ppx = prim_pts[3 * o], ppy = prim_pts[3 * o + 1], ppz = prim_pts[3 * o + 2];
      float s0 = 0.f, s1 = 0.f, s2 = 0.f;
      const int nL = n_lights[n];
      for (int l = 0; l < nL; ++l) {
        const size_t lo = (size_t)n * L + l;
        float lx = light_pts[3 * lo] - ppx, ly = light_pts[3 * lo + 1] - ppy, lz = light_pts[3 * lo + 2] - ppz;
        const float len = sqrtf(lx * lx + ly * ly + lz * lz);
        lx /= len; ly /= len; lz /= len;
        const float cos_dot = clampf(lx * dx + ly * dy + lz * dz, -1.f, 1.f);
        const float angle = acosf(cos_dot);
        float w = 0.f;
        switch (w_type) {
          case 0: w = expf(-0.5f * sq(angle / sigma)) / (sigma * SQRT2PI23); break;
          case 1: w = expf(-0.5f * sq(angle / sigma)); break;
          case 2: w = expf((cos_dot - 1.f) / sigma) / (sigma * TWOPI); break;
          case 3: w = expf((cos_dot - 1.f) / sigma); break;
        }
        s0 += light_values[3 * lo] * w; s1 += light_values[3 * lo + 1] * w; s2 += light_values[3 * lo + 2] * w;
      }
      integral[3 * o] = s0; integral[3 * o + 1] = s1; integral[3 * o + 2] = s2;
    }
}

ORC_API void orc_sg_bwd(int N, int D, int L, const float* lobe_dirs, const float* lobe_sigmas,
                        const float* light_values, const float* light_pts, const float* prim_pts,
                        const int32_t* n_lights, const float* grad_integral, float* grad_dirs,
                        float* grad_sigmas, float* grad_light_values, int w_type) {
  double* glv = NULL;
  if (grad_light_values) glv = (double*)calloc((size_t)N * L * 3, sizeof(double));
#pragma omp parallel for collapse(2) schedule(static)
  for (int n = 0; n < N; ++n)
    for (int d = 0; d < D; ++d) {
      const size_t o = (size_t)n * D + d;
      const float gi0 = grad_integral[3 * o], gi1 = grad_integral[3 * o + 1], gi2 = grad_integral[3 * o + 2];
      const float dx = lobe_dirs[3 * o], dy = lobe_dirs[3 * o + 1], dz = lobe_dirs[3 * o + 2];
      const float sigma = lobe_sigmas[o];
      const float ppx = prim_pts[3 * o], ppy = prim_pts[3 * o + 1], ppz = prim_pts[3 * o + 2];
      float gd0 = 0.f, gd1 = 0.f, gd2 = 0.f, gs = 0.f;
      const int nL = n_lights[n];
      for (int l = 0; l < nL; ++l) {
        const size_t lo = (size_t)n * L + l;
        const float e0 = light_values[3 * lo], e1 = light_values[3 * lo + 1], e2 = light_values[3 * lo + 2];
        float lx = light_pts[3 * lo] - ppx, ly = light_pts[3 * lo + 1] - ppy, lz = light_pts[3 * lo + 2] - ppz;
        const float len = sqrtf(lx * lx + ly * ly + lz * lz);
        lx /= len; ly /= len; lz /= len;
        const float cos_dot = lx * dx + ly * dy + lz * dz;
        const float cc = clampf(cos_dot, -1.f, 1.f);
        const float angle = acosf(cc);
        float weight = 0.f, dL_cos = 0.f, dL_angle = 0.f, dL_w = 0.f, ev = 0.f;
        const int inrange = (cos_dot > -1.f && cos_dot < 1.f);
        switch (w_type) {
          case 0:
            ev = expf(-0.5f * sq(angle / sigma));
            weight = ev / (sigma * SQRT2PI23);
            dL_w = gi0 * e0 + gi1 * e1 + gi2 * e2;
            gs += dL_w * ((ev * INVSQRT2PI23 * (sq(angle) - sq(sigma))) / (sq(sigma) * sq(sigma)));
            dL_angle = dL_w * -((INVSQRT2PI23 * angle * ev) / (sq(sigma) * sigma));
            dL_cos = dL_angle * (inrange ? (-1.f / sqrtf(1.f - sq(cos_dot))) : -20.f);
            break;
          case 1:
            ev = expf(-0.5f * sq(angle / sigma));
            weight = ev;
            dL_w = gi0 * e0 + gi1 * e1 + gi2 * e2;
            gs += dL_w * ((ev * sq(angle)) / (sigma * sq(sigma)));
            dL_angle = dL_w * -((angle * ev) / sq(sigma));
            dL_cos = dL_angle * (inrange ? (-1.f / sqrtf(1.f - sq(cos_dot))) : -20.f);
            break;
          case 2:
            ev = expf((cc - 1.f) / sigma);
            weight = ev / (sigma * TWOPI);
            dL_w = gi0 * e0 + gi1 * e1 + gi2 * e2;
            gs += dL_w * ((ev * INV2PI * ((1.f - cc) - sigma)) / (sigma * sq(sigma)));
            dL_cos = dL_w * INV2PI * ev / sq(sigma);
            break;
          case 3:
            ev = expf((cc - 1.f) / sigma);
            weight = ev;
            dL_w = gi0 * e0 + gi1 * e1 + gi2 * e2;
            gs += dL_w * ((ev * (1.f - cc) / sq(sigma)));
            dL_cos = dL_w * ev / sigma;
            break;
        }
        gd0 += dL_cos * lx; gd1 += dL_cos * ly; gd2 += dL_cos * lz;
        if (glv) {
#pragma omp atomic
          glv[3 * lo] += (double)(gi0 * weight);
#pragma omp atomic
          glv[3 * lo + 1] += (double)(gi1 * weight);
#pragma omp atomic
          glv[3 * lo + 2] += (double)(gi2 * weight);
        }
      }
      grad_sigmas[o] = gs;
      grad_dirs[3 * o] = gd0; grad_dirs[3 * o + 1] = gd1; grad_dirs[3 * o + 2] = gd2;
    }
  if (glv) {
    for (size_t i = 0; i < (size_t)N * L * 3; ++i) grad_light_values[i] += (float)glv[i];
    free(glv);
  }
}
