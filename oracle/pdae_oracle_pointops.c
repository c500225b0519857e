/* pdae_oracle_pointops.c -- CPU oracle of the segment FPS and segment kNN (csrc/pointops.cu) in the kernels' fp32
 * operations and tie rules (include/pointdae_b200.h).  Build: gcc -O2 -ffp-contract=off (oracle/cpu_pointops.py).
 * The search is plain: every candidate is compared with the current best by (value, tie rank) for FPS and kept in a
 * sorted list by (d^2, index) for kNN; no blocking, no threads. */
#include <math.h>
#include <stdint.h>
#include <string.h>

static void seg_bounds(const int *off, int s, int total, int *lo, int *hi) {
  int a = s ? off[s - 1] : 0, e = off[s];
  if (a < 0) a = 0;
  if (a > total) a = total;
  if (e < a) e = a;
  if (e > total) e = total;
  *lo = a;
  *hi = e;
}

static float dist_yxz(float dx, float dy, float dz) { return fmaf(dz, dz, fmaf(dx, dx, dy * dy)); }
static float dist_seq3(float dx, float dy, float dz) { return fmaf(dz, dz, fmaf(dy, dy, dx * dx)); }

/* opt_n_threads of the reference's pointops, capped at 1024 */
int pdae_oracle_seg_fps_block_size(int n) {
  if (n <= 0) return 1;
  const int pow_2 = (int)(log((double)n) / log(2.0));
  int t = 1 << pow_2;
  if (t > 1024) t = 1024;
  if (t < 1) t = 1;
  return t;
}

static uint32_t brev_lg(uint32_t v, int lg) {
  uint32_t r = 0;
  for (int i = 0; i < lg; ++i) r |= ((v >> i) & 1u) << (lg - 1 - i);
  return r;
}

/* tmp: (n_total) running minima, updated in place (null: a private copy starting from 1e10; scratch (n_total)) */
void pdae_oracle_seg_fps(const float *xyz, int n_total, const int *offset, const int *new_offset, int b, int n,
                         int m_total, float *tmp, int *idx, float *scratch) {
  const int bs = pdae_oracle_seg_fps_block_size(n);
  int lg = 0;
  while ((1 << (lg + 1)) <= bs) ++lg;
  float *run = tmp;
  if (!run) {
    run = scratch;
    for (int k = 0; k < n_total; ++k) run[k] = 1e10f;
  }
  for (int s = 0; s < b; ++s) {
    int sn, en, sm, em;
    seg_bounds(offset, s, n_total, &sn, &en);
    seg_bounds(new_offset, s, m_total, &sm, &em);
    const int cnt = en - sn;
    if (em == sm) continue;
    if (cnt == 0) {
      for (int j = sm; j < em; ++j) idx[j] = sn;
      continue;
    }
    idx[sm] = sn;
    int old = sn;
    for (int j = sm + 1; j < em; ++j) {
      const float ox = xyz[3 * old], oy = xyz[3 * old + 1], oz = xyz[3 * old + 2];
      float best = 0.0f;
      uint64_t best_rank = 0;
      int have = 0, besti = sn;  /* no point taken: the segment start */
      for (int k = sn; k < en; ++k) {
        const float d = dist_yxz(xyz[3 * k] - ox, xyz[3 * k + 1] - oy, xyz[3 * k + 2] - oz);
        const float d2 = fminf(d, run[k]);
        run[k] = d2;
        if (!(d2 > -1.0f)) continue;  /* never taken by the reference's `d2 > best` from best = -1 */
        /* tie rank: (bit-reversed slot, k / bs), slot and k relative to the segment start; -0 == +0 ties */
        const uint32_t rel = (uint32_t)(k - sn);
        const uint64_t rank = ((uint64_t)brev_lg(rel & (uint32_t)(bs - 1), lg) << 32) | (rel >> lg);
        if (!have || d2 > best || (d2 == best && rank < best_rank)) {
          have = 1;
          best = d2;
          best_rank = rank;
          besti = k;
        }
      }
      old = besti;
      idx[j] = old;
    }
  }
}

/* idx / dist2: (m, nsample); the reference's segment of a query is the first s with p < new_offset[s] */
void pdae_oracle_seg_knn(const float *xyz, int n_total, const float *new_xyz, int m, const int *offset,
                         const int *new_offset, int b, int nsample, int *idx, float *dist2) {
  int qlo = 0;
  for (int s = 0; s < b; ++s) {
    int qhi = new_offset[s];
    if (qhi < 0) qhi = 0;
    if (qhi > m) qhi = m;
    if (qhi < qlo) qhi = qlo;
    int sn, en;
    seg_bounds(offset, s, n_total, &sn, &en);
    for (int p = qlo; p < qhi; ++p) {
      const float qx = new_xyz[3 * p], qy = new_xyz[3 * p + 1], qz = new_xyz[3 * p + 2];
      float *dd = dist2 + (size_t)p * nsample;
      int *ii = idx + (size_t)p * nsample;
      int filled = 0;
      for (int k = sn; k < en; ++k) {
        const float d = dist_seq3(xyz[3 * k] - qx, xyz[3 * k + 1] - qy, xyz[3 * k + 2] - qz);
        if (!(d < 1e10f)) continue;
        if (filled == nsample && !(d < dd[nsample - 1])) continue;  /* k ascending: an equal distance loses */
        int pos = filled < nsample ? filled++ : nsample - 1;
        while (pos > 0 && d < dd[pos - 1]) {
          dd[pos] = dd[pos - 1];
          ii[pos] = ii[pos - 1];
          --pos;
        }
        dd[pos] = d;
        ii[pos] = k;
      }
      for (int i = filled; i < nsample; ++i) {
        dd[i] = 1e10f;
        ii[i] = sn;
      }
    }
    qlo = qhi;
  }
  for (int p = qlo; p < m; ++p)
    for (int i = 0; i < nsample; ++i) {
      idx[(size_t)p * nsample + i] = -1;
      dist2[(size_t)p * nsample + i] = 1e10f;
    }
}
