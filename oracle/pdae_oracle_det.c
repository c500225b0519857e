/* pdae_oracle_det.c -- CPU oracle of the deterministic gradients (the *_det entry points of include/pointdae_b200.h).
 *
 * Every gradient element starts from its own term (+0.0f where the op has none) and adds the scattered contributions
 * in ascending order of the source slot within the cloud, in fp32 with the same expressions as the CUDA kernels.
 * Walking the sources once in ascending order and adding each into its target gives exactly that order per target.
 * Built with -ffp-contract=off like pdae_oracle.c, so no product is fused into an add; the results are compared with
 * the GPU bit for bit.  Targets outside [0, t) are skipped, as the reverse index leaves them out.
 */
#include <stddef.h>
#include <stdint.h>
#include <string.h>

int pdae_oracle_det_version(void) { return 1; }

/* cloud 1 then cloud 2, own terms first: v = (gd * 2) * (a - b[idx]); the matched point receives -v */
static void chamfer_own(const float *A, const float *B, const int *idx, const float *gd, int n, float *g) {
  for (int i = 0; i < n; ++i) {
    const float s = gd[i] * 2.0f;
    for (int c = 0; c < 3; ++c) g[3 * i + c] = s * (A[3 * i + c] - B[3 * idx[i] + c]);
  }
}
static void chamfer_scatter(const float *A, const float *B, const int *idx, const float *gd, int n, int m, float *gb) {
  for (int j = 0; j < n; ++j) {
    const int t = idx[j];
    if (t < 0 || t >= m) continue;
    const float s = gd[j] * 2.0f;
    for (int c = 0; c < 3; ++c) gb[3 * t + c] = gb[3 * t + c] + -(s * (A[3 * j + c] - B[3 * t + c]));
  }
}

void pdae_oracle_chamfer_bwd_ordered(const float *xyz1, const float *xyz2, const int *idx1, const int *idx2,
                                     const float *gd1, const float *gd2, int b, int n, int m, float *gx1, float *gx2) {
  for (int i = 0; i < b; ++i) {
    const float *A = xyz1 + (size_t)i * n * 3, *B = xyz2 + (size_t)i * m * 3;
    const int *i1 = idx1 + (size_t)i * n, *i2 = idx2 + (size_t)i * m;
    const float *g1 = gd1 + (size_t)i * n, *g2 = gd2 + (size_t)i * m;
    float *o1 = gx1 + (size_t)i * n * 3, *o2 = gx2 + (size_t)i * m * 3;
    chamfer_own(A, B, i1, g1, n, o1);
    chamfer_own(B, A, i2, g2, m, o2);
    chamfer_scatter(B, A, i2, g2, m, n, o1);
    chamfer_scatter(A, B, i1, g1, n, m, o2);
  }
}

/* gout (b, c, s / div) with source slot j reading element j / div, optional weight (b, s) -> g (b, c, t) */
static void channel_major(const float *gout, const int *idx, const float *weight, int b, int c, int s, int t, int div,
                          float *g) {
  const int gs = s / div;
  for (int bi = 0; bi < b; ++bi)
    for (int l = 0; l < c; ++l) {
      float *o = g + ((size_t)bi * c + l) * t;
      const float *go = gout + ((size_t)bi * c + l) * gs;
      for (int p = 0; p < t; ++p) o[p] = 0.0f;
      for (int j = 0; j < s; ++j) {
        const int p = idx[(size_t)bi * s + j];
        if (p < 0 || p >= t) continue;
        float v = go[j / div];
        if (weight) v = v * weight[(size_t)bi * s + j];
        o[p] = o[p] + v;
      }
    }
}

void pdae_oracle_gather_grad_ordered(const float *gout, const int *idx, int b, int c, int n, int m, float *gfeat) {
  channel_major(gout, idx, NULL, b, c, m, n, 1, gfeat);
}

void pdae_oracle_group_points_grad_ordered(const float *gout, const int *idx, int b, int c, int n, int npoints, int nsample,
                                           float *gpoints) {
  channel_major(gout, idx, NULL, b, c, npoints * nsample, n, 1, gpoints);
}

void pdae_oracle_three_interpolate_grad_ordered(const float *gout, const int *idx, const float *weight, int b, int c, int n,
                                                int m, float *gpoints) {
  channel_major(gout, idx, weight, b, c, 3 * n, m, 3, gpoints);
}

/* gout physical (b, n, k, 2c) -> gx (b, c, n): centre term of row j (p ascending), then G[i][p][0:c] for every edge
 * i -> idx[i][p] == j, slot i * k + p ascending */
void pdae_oracle_graph_feature_grad_ordered(const float *gout, const int64_t *idx, int b, int c, int n, int k, float *gx) {
  for (int bi = 0; bi < b; ++bi) {
    float *o = gx + (size_t)bi * c * n;
    for (int j = 0; j < n; ++j)
      for (int ch = 0; ch < c; ++ch) {
        float s = 0.0f;
        for (int p = 0; p < k; ++p) {
          const float *G = gout + (((size_t)bi * n + j) * k + p) * 2 * c;
          s = s + (G[c + ch] - G[ch]);
        }
        o[(size_t)ch * n + j] = s;
      }
    for (int i = 0; i < n; ++i)
      for (int p = 0; p < k; ++p) {
        const int64_t j = idx[((size_t)bi * n + i) * k + p];
        if (j < 0 || j >= n) continue;
        const float *G = gout + (((size_t)bi * n + i) * k + p) * 2 * c;
        for (int ch = 0; ch < c; ++ch) o[(size_t)ch * n + j] = o[(size_t)ch * n + j] + G[ch];
      }
  }
}
