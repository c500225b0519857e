/* pdae_oracle_emd.c -- CPU oracle of the approximate Earth Mover's Distance (csrc/emd.cu): the same fp32 operations in
 * the same order as include/pointdae_b200.h defines them, built with -ffp-contract=off so that every fma is an explicit
 * fmaf.  Two operations differ from the kernels: the pair term uses libm exp2f (flushing subnormal results to zero
 * like ex2.approx.ftz) in place of ex2.approx, and the gradient uses 1 / sqrtf in place of rsqrtf; GPU results are
 * therefore compared with this oracle within a tolerance.  The cost reduction needs no approximation: given the same
 * match it is bit-exact.  Checker only, never a product path. */
#include <float.h>
#include <math.h>
#include <stddef.h>

#define LEVELS 10

static float scale(int j) {
  const float level = j < 9 ? -ldexpf(1.f, 2 * (7 - j)) : 0.f;
  return level * 1.44269504f;
}

static float dist(const float *a, const float *b) {
  const float dx = b[0] - a[0], dy = b[1] - a[1], dz = b[2] - a[2];
  return fmaf(dz, dz, fmaf(dy, dy, dx * dx));
}

static float pair_term(float c, float d) {
  const float e = exp2f(c * d);
  return e < FLT_MIN ? 0.f : e;
}

/* ratios (b,10,n), (b,10,m); match (b,m,n) accumulated in pass 3 like the published kernel (may be NULL);
 * remain: scratch of n + m floats */
void pdae_oracle_emd_match(const float *xyz1, const float *xyz2, int b, int n, int m, float *ratio_l, float *ratio_r,
                           float *match, float *remain) {
  float *reml = remain, *remr = remain + n;
  for (int bi = 0; bi < b; ++bi) {
    const float *x1 = xyz1 + (size_t)bi * n * 3, *x2 = xyz2 + (size_t)bi * m * 3;
    float *rl = ratio_l + (size_t)bi * LEVELS * n, *rr = ratio_r + (size_t)bi * LEVELS * m;
    float *mt = match ? match + (size_t)bi * m * n : NULL;
    const float multl = n >= m ? 1.f : (float)(m / n), multr = n >= m ? (float)(n / m) : 1.f;
    for (int k = 0; k < n; ++k) reml[k] = multl;
    for (int l = 0; l < m; ++l) remr[l] = multr;
    if (mt)
      for (size_t i = 0; i < (size_t)m * n; ++i) mt[i] = 0.f;
    for (int j = 0; j < LEVELS; ++j) {
      const float c = scale(j);
      float *rlj = rl + (size_t)j * n, *rrj = rr + (size_t)j * m;
      for (int k = 0; k < n; ++k) {
        float s = 1e-9f;
        for (int l = 0; l < m; ++l) s = fmaf(pair_term(c, dist(x1 + 3 * k, x2 + 3 * l)), remr[l], s);
        rlj[k] = reml[k] / s;
      }
      for (int l = 0; l < m; ++l) {
        float t = 0.f;
        for (int k = 0; k < n; ++k) t = fmaf(pair_term(c, dist(x1 + 3 * k, x2 + 3 * l)), rlj[k], t);
        const float r = remr[l], sumr = t * r;
        rrj[l] = fminf(r / (sumr + 1e-9f), 1.f) * r;
        remr[l] = fmaxf(0.f, r - sumr);
      }
      for (int k = 0; k < n; ++k) {
        float u = 0.f;
        for (int l = 0; l < m; ++l) {
          const float w = (pair_term(c, dist(x1 + 3 * k, x2 + 3 * l)) * rlj[k]) * rrj[l];
          if (mt) mt[(size_t)l * n + k] += w;
          u += w;
        }
        reml[k] = fmaxf(0.f, reml[k] - u);
      }
    }
  }
}

/* match (b,m,n) rebuilt from the ratios: sum over levels of (e * ratioL) * ratioR from +0 */
void pdae_oracle_emd_rebuild(const float *xyz1, const float *xyz2, int b, int n, int m, const float *ratio_l,
                             const float *ratio_r, float *match) {
  for (int bi = 0; bi < b; ++bi) {
    const float *x1 = xyz1 + (size_t)bi * n * 3, *x2 = xyz2 + (size_t)bi * m * 3;
    const float *rl = ratio_l + (size_t)bi * LEVELS * n, *rr = ratio_r + (size_t)bi * LEVELS * m;
    for (int l = 0; l < m; ++l)
      for (int k = 0; k < n; ++k) {
        const float d = dist(x1 + 3 * k, x2 + 3 * l);
        float acc = 0.f;
        for (int j = 0; j < LEVELS; ++j) acc += (pair_term(scale(j), d) * rl[(size_t)j * n + k]) * rr[(size_t)j * m + l];
        match[((size_t)bi * m + l) * n + k] = acc;
      }
  }
}

void pdae_oracle_emd_cost(const float *xyz1, const float *xyz2, int b, int n, int m, const float *match, float *cost) {
  for (int bi = 0; bi < b; ++bi) {
    const float *x1 = xyz1 + (size_t)bi * n * 3, *x2 = xyz2 + (size_t)bi * m * 3;
    float p[256];
    for (int t = 0; t < 256; ++t) p[t] = 0.f;
    for (int l = 0; l < m; ++l) {
      float acc = 0.f;
      for (int k = 0; k < n; ++k) acc = fmaf(sqrtf(dist(x1 + 3 * k, x2 + 3 * l)), match[((size_t)bi * m + l) * n + k], acc);
      p[l % 256] += acc;
    }
    for (int s = 128; s > 0; s >>= 1)
      for (int t = 0; t < s; ++t) p[t] += p[t + s];
    cost[bi] = p[0];
  }
}

void pdae_oracle_emd_grad(const float *gcost, const float *xyz1, const float *xyz2, int b, int n, int m,
                          const float *match, float *grad1, float *grad2) {
  for (int bi = 0; bi < b; ++bi) {
    const float *x1 = xyz1 + (size_t)bi * n * 3, *x2 = xyz2 + (size_t)bi * m * 3;
    const float *mt = match + (size_t)bi * m * n;
    const float g = gcost[bi];
    for (int k = 0; k < n; ++k) {
      float a[3] = {0.f, 0.f, 0.f};
      for (int l = 0; l < m; ++l) {
        const float *p = x1 + 3 * k, *q = x2 + 3 * l;
        const float coef = mt[(size_t)l * n + k] * (1.f / sqrtf(fmaxf(dist(p, q), 1e-20f)));
        for (int e = 0; e < 3; ++e) a[e] = fmaf(coef, p[e] - q[e], a[e]);
      }
      for (int e = 0; e < 3; ++e) grad1[((size_t)bi * n + k) * 3 + e] = g * a[e];
    }
    for (int l = 0; l < m; ++l) {
      float a[3] = {0.f, 0.f, 0.f};
      for (int k = 0; k < n; ++k) {
        const float *p = x2 + 3 * l, *q = x1 + 3 * k;
        const float coef = mt[(size_t)l * n + k] * (1.f / sqrtf(fmaxf(dist(q, p), 1e-20f)));
        for (int e = 0; e < 3; ++e) a[e] = fmaf(coef, p[e] - q[e], a[e]);
      }
      for (int e = 0; e < 3; ++e) grad2[((size_t)bi * m + l) * 3 + e] = g * a[e];
    }
  }
}
