// emd_core.cuh -- the approximate-EMD bodies shared by the equal-size entry points (emd.cu) and the segment entry points
// (segemd.cu): approxmatch over one cloud on a cluster of CTAs, the row / column sums over the match rebuilt from the
// per-level ratios, and the per-cloud cost reduction.  Semantics: include/pointdae_b200.h; design: emd.cu.
#pragma once
#include <cooperative_groups.h>

#include "common.cuh"

namespace pdae {

namespace cg = cooperative_groups;

constexpr int EMD_LEVELS = 10;
constexpr int EMD_THREADS = 128;
constexpr int EMD_CHUNK = EMD_THREADS * 2;  // owned points per CTA per sweep: one f32x2 pack per thread
constexpr int EMD_TILE = 512;               // streamed points per shared-memory tile
constexpr int EMD_MAX_POINTS = 65536;
constexpr int EMD_MAX_CLUSTER = 8;

__device__ __forceinline__ float2 add2(float2 a, float2 b) {
  uint64_t r;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(f2_as_u64(a)), "l"(f2_as_u64(b)));
  return u64_as_f2(r);
}
__device__ __forceinline__ float ex2a(float x) {
  float r;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
__device__ __forceinline__ float2 ex2a2(float2 x) { return make_float2(ex2a(x.x), ex2a(x.y)); }
__device__ __forceinline__ float2 bc2(float v) { return make_float2(v, v); }

// level j = 0..9 is -4^(7-j) (j < 9) or 0; the exponent scale is rn(level * log2(e)) (exact: level is a power of 4)
__device__ __forceinline__ float emd_scale(int j) {
  const float level = j < 9 ? -__int_as_float((127 + 2 * (7 - j)) << 23) : 0.f;
  return __fmul_rn(level, 1.44269504f);
}

// squared distance of the pack: (x2 - x1)^2 with fma(dz,dz, fma(dy,dy, rn(dx*dx))); the sign of the difference does
// not change the bits, so callers pass whichever difference they also need
__device__ __forceinline__ float2 emd_dist2(float2 dx, float2 dy, float2 dz) { return fma2(dz, dz, fma2(dy, dy, mul2(dx, dx))); }

struct Pack3 {
  float2 x, y, z;
};

__device__ __forceinline__ Pack3 load_pack(const float *__restrict__ pts, int i0, int cnt) {
  const int a = min(i0, cnt - 1), b = min(i0 + 1, cnt - 1);  // lanes past the cloud repeat its last point (discarded)
  Pack3 p;
  p.x = make_float2(__ldg(pts + 3 * a), __ldg(pts + 3 * b));
  p.y = make_float2(__ldg(pts + 3 * a + 1), __ldg(pts + 3 * b + 1));
  p.z = make_float2(__ldg(pts + 3 * a + 2), __ldg(pts + 3 * b + 2));
  return p;
}

// One sweep of the CTA's owned pack over the whole other cloud (`cnt` points, tile values `s`), ascending.  OWN2: the
// owned points are cloud 2 (columns).  MODE 0: acc = fma(e, s, acc).  MODE 1: acc = acc + rn(rn(e * rl) * s).
// Every thread of the CTA calls it (it synchronises the CTA).  `s` may have been written by other CTAs of the
// cluster in this launch, so it is read through L2 (ld.global.cg).
template <bool OWN2, int MODE>
__device__ __forceinline__ float2 emd_sweep(const Pack3 &own, float2 rl, float2 acc, float c, const float *__restrict__ oth,
                                            const float *s, int cnt, float4 *tile) {
  const float2 c2 = bc2(c);
  for (int base = 0; base < cnt; base += EMD_TILE) {
    const int tn = min(EMD_TILE, cnt - base);
    __syncthreads();
    for (int i = threadIdx.x; i < tn; i += EMD_THREADS) {
      const float *q = oth + 3 * static_cast<size_t>(base + i);
      tile[i] = make_float4(__ldg(q), __ldg(q + 1), __ldg(q + 2), __ldcg(s + base + i));
    }
    __syncthreads();
#pragma unroll 4
    for (int t = 0; t < tn; ++t) {
      const float4 p = tile[t];
      const float2 dx = OWN2 ? sub2(own.x, bc2(p.x)) : sub2(bc2(p.x), own.x);
      const float2 dy = OWN2 ? sub2(own.y, bc2(p.y)) : sub2(bc2(p.y), own.y);
      const float2 dz = OWN2 ? sub2(own.z, bc2(p.z)) : sub2(bc2(p.z), own.z);
      const float2 e = ex2a2(mul2(emd_dist2(dx, dy, dz), c2));
      if (MODE == 0) acc = fma2(e, bc2(p.w), acc);
      else acc = add2(acc, mul2(mul2(e, rl), bc2(p.w)));
    }
  }
  return acc;
}

__device__ __forceinline__ void emd_cluster_sync(int cs) {
  if (cs == 1) {
    __syncthreads();
  } else {
    __threadfence();
    cg::this_cluster().sync();
  }
}

// The tables of the segment kernels (segemd.cu): ranges[s] = (lo1, hi1, lo2, hi2) of segment s; for the sums, the
// CTA's unit units[blockIdx.x] = (segment, first owned point relative to the segment start) of the owned side, which
// has *count units.  Kept out of the argument structs so that the equal-size kernels keep their parameter layout.
struct EmdSegTables {
  const int4 *ranges;
  const int2 *units;
  const int *count;
};

// Arguments of approxmatch.  Equal-size layout: cloud b is xyz1 (b,n,3) against xyz2 (b,m,3), ratios (b,10,n) and
// (b,10,m).  SEG: n, m are the packed totals and the ratios (10,n) / (10,m).
struct EmdMatchArgs {
  const float *xyz1, *xyz2;
  int n, m, cs;
  float *ratio_l, *ratio_r;  // (B,10,n), (B,10,m)
  float *remain_l, *remain_r;  // workspace (B,n), (B,m)
};

// approxmatch of cloud (or segment) blockIdx.x / cs on the `cs` CTAs of a cluster; owned chunks of EMD_CHUNK points go
// round-robin to the ranks.  SEG: a segment with an empty side returns at once on every CTA of its cluster (they all
// read the same range), before the first cluster barrier.  The SEG terms are compile-time constants otherwise, so the
// equal-size kernel is this code alone.
template <bool SEG>
__device__ __forceinline__ void emd_approxmatch_body(const EmdMatchArgs &a, const EmdSegTables &sg, float4 *tile) {
  const int4 r = SEG ? __ldg(sg.ranges + blockIdx.x / a.cs) : make_int4(0, 0, 0, 0);
  const int cs = a.cs, n = SEG ? r.y - r.x : a.n, m = SEG ? r.w - r.z : a.m;
  const int b = blockIdx.x / cs, rank = blockIdx.x % cs, tid = threadIdx.x;
  if (SEG && (n <= 0 || m <= 0)) return;
  const float *x1 = a.xyz1 + (SEG ? 3 * static_cast<size_t>(r.x) : static_cast<size_t>(b) * n * 3);
  const float *x2 = a.xyz2 + (SEG ? 3 * static_cast<size_t>(r.z) : static_cast<size_t>(b) * m * 3);
  float *rl = a.ratio_l + (SEG ? static_cast<size_t>(r.x) : static_cast<size_t>(b) * EMD_LEVELS * n);
  float *rr = a.ratio_r + (SEG ? static_cast<size_t>(r.z) : static_cast<size_t>(b) * EMD_LEVELS * m);
  float *reml = a.remain_l + (SEG ? static_cast<size_t>(r.x) : static_cast<size_t>(b) * n);
  float *remr = a.remain_r + (SEG ? static_cast<size_t>(r.z) : static_cast<size_t>(b) * m);
  const int sl = SEG ? a.n : n, sr = SEG ? a.m : m;  // level strides of the ratios
  const float multl = n >= m ? 1.f : static_cast<float>(m / n), multr = n >= m ? static_cast<float>(n / m) : 1.f;
  const int nch_n = (n + EMD_CHUNK - 1) / EMD_CHUNK, nch_m = (m + EMD_CHUNK - 1) / EMD_CHUNK;
  for (int i = rank * EMD_THREADS + tid; i < n; i += cs * EMD_THREADS) reml[i] = multl;
  for (int i = rank * EMD_THREADS + tid; i < m; i += cs * EMD_THREADS) remr[i] = multr;
  emd_cluster_sync(cs);
  for (int j = 0; j < EMD_LEVELS; ++j) {
    const float c = emd_scale(j);
    float *rlj = rl + static_cast<size_t>(j) * sl, *rrj = rr + static_cast<size_t>(j) * sr;
    // pass 1, rows: ratioL = remainL / (1e-9 + sum_l e * remainR)
    for (int q = rank; q < nch_n; q += cs) {
      const int k = q * EMD_CHUNK + 2 * tid;
      const float2 acc = emd_sweep<false, 0>(load_pack(x1, k, n), bc2(0.f), bc2(1e-9f), c, x2, remr, m, tile);
      if (k < n) rlj[k] = __fdiv_rn(reml[k], acc.x);
      if (k + 1 < n) rlj[k + 1] = __fdiv_rn(reml[k + 1], acc.y);
    }
    emd_cluster_sync(cs);
    // pass 2, columns: sumr = remainR * sum_k e * ratioL; ratioR, remainR
    for (int q = rank; q < nch_m; q += cs) {
      const int l = q * EMD_CHUNK + 2 * tid;
      const float2 acc = emd_sweep<true, 0>(load_pack(x2, l, m), bc2(0.f), bc2(0.f), c, x1, rlj, n, tile);
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        if (l + h < m) {
          const float r = remr[l + h], sumr = __fmul_rn(h ? acc.y : acc.x, r);
          rrj[l + h] = __fmul_rn(fminf(__fdiv_rn(r, __fadd_rn(sumr, 1e-9f)), 1.f), r);
          remr[l + h] = fmaxf(0.f, __fsub_rn(r, sumr));
        }
      }
    }
    emd_cluster_sync(cs);
    // pass 3, rows: remainL -= sum_l w
    for (int q = rank; q < nch_n; q += cs) {
      const int k = q * EMD_CHUNK + 2 * tid;
      const float2 own_rl = make_float2(k < n ? __ldcg(rlj + k) : 0.f, k + 1 < n ? __ldcg(rlj + k + 1) : 0.f);
      const float2 acc = emd_sweep<false, 1>(load_pack(x1, k, n), own_rl, bc2(0.f), c, x2, rrj, m, tile);
      if (k < n) reml[k] = fmaxf(0.f, __fsub_rn(reml[k], acc.x));
      if (k + 1 < n) reml[k + 1] = fmaxf(0.f, __fsub_rn(reml[k + 1], acc.y));
    }
    // the next pass 1 reads remainR (stable since the barrier above) and this thread's own remainL
  }
}

// ---- consumers of the match: materialisation, cost, gradient ---------------------------------------------------------
// A streamed point: coordinates and its 10 ratios (the other side's), 16 floats so the tile reads as float4s.
struct EmdPt {
  float x, y, z, pad;
  float r[12];
};

// the match element of the pack from the owned ratios `ro` and the streamed point's ratios, in level order from +0:
// acc + rn(rn(e * ratioL) * ratioR) whichever side is owned
template <bool OWN2>
__device__ __forceinline__ float2 emd_rebuild(float2 d, const float2 *ro, const EmdPt &p) {
  float2 acc = bc2(0.f);
#pragma unroll
  for (int j = 0; j < EMD_LEVELS; ++j) {
    const float2 e = ex2a2(mul2(d, bc2(emd_scale(j))));
    acc = add2(acc, OWN2 ? mul2(mul2(e, bc2(p.r[j])), ro[j]) : mul2(mul2(e, ro[j]), bc2(p.r[j])));
  }
  return acc;
}

// Arguments of the sums.  Equal-size layout: (B,n,3) / (B,m,3), ratios (B,10,n) / (B,10,m).  SEG: n, m are the
// packed totals and the ratios (10,n) / (10,m).
struct EmdSumArgs {
  const float *xyz1, *xyz2;
  int n, m;
  const float *match;              // (B,m,n) or null: rebuilt from the ratios
  const float *ratio_l, *ratio_r;  // (B,10,n), (B,10,m)
};

// The owned pack's sums over the whole other cloud, ascending.  Rows (OWN2 = false) or columns (OWN2 = true), one
// CTA per EMD_CHUNK owned points (grid.x) and cloud (grid.y); SEG: one CTA per unit, CTAs past *count return.
//   WHAT 0 (columns): rowcost[l] = sum_k fma(sqrtf(d), match[l][k], .)
//   WHAT 1: grad[p] = g_b * sum fma(rn(match * rsqrtf(fmaxf(d, 1e-20))), p - other, .) per coordinate
//   WHAT 2 (rows, no match given): match[l][k] written from the ratios
// SEG rebuilds the match from the ratios, writes rowcost and grad at global rows and takes g of the unit's segment.
template <bool OWN2, int WHAT, bool SEG = false>
__global__ void __launch_bounds__(EMD_THREADS) emd_sum_kernel(const EmdSumArgs a, const float *__restrict__ gcost,
                                                              float *__restrict__ out, const EmdSegTables sg) {
  __shared__ float4 tile[EMD_TILE / 4 * 4];  // EMD_TILE / 4 points of 4 float4s
  if (SEG && blockIdx.x >= static_cast<unsigned>(__ldg(sg.count))) return;  // uniform for the CTA
  const int2 u = SEG ? __ldg(sg.units + blockIdx.x) : make_int2(0, 0);
  const int4 r = SEG ? __ldg(sg.ranges + u.x) : make_int4(0, 0, 0, 0);
  EmdPt *pts = reinterpret_cast<EmdPt *>(tile);
  constexpr int TP = EMD_TILE / 4;
  const int b = SEG ? u.x : blockIdx.y, tid = threadIdx.x;
  const int n = SEG ? r.y - r.x : a.n, m = SEG ? r.w - r.z : a.m, nown = OWN2 ? m : n, noth = OWN2 ? n : m;
  const int lo_own = OWN2 ? r.z : r.x, lo_oth = OWN2 ? r.x : r.z;  // SEG only
  const int so = SEG ? (OWN2 ? a.m : a.n) : nown, ss = SEG ? (OWN2 ? a.n : a.m) : noth;  // level strides of the ratios
  const float *xo = (OWN2 ? a.xyz2 : a.xyz1) + (SEG ? 3 * static_cast<size_t>(lo_own) : static_cast<size_t>(b) * nown * 3);
  const float *xs = (OWN2 ? a.xyz1 : a.xyz2) + (SEG ? 3 * static_cast<size_t>(lo_oth) : static_cast<size_t>(b) * noth * 3);
  const float *ro_g = (OWN2 ? a.ratio_r : a.ratio_l) + (SEG ? static_cast<size_t>(lo_own) : static_cast<size_t>(b) * EMD_LEVELS * nown);
  const float *rs_g = (OWN2 ? a.ratio_l : a.ratio_r) + (SEG ? static_cast<size_t>(lo_oth) : static_cast<size_t>(b) * EMD_LEVELS * noth);
  const bool rebuild = SEG || a.match == nullptr;
  const float *mat = rebuild ? nullptr : a.match + static_cast<size_t>(b) * m * n;
  const int i = SEG ? u.y + 2 * tid : blockIdx.x * EMD_CHUNK + 2 * tid;
  static_assert(!SEG || WHAT != 2, "the segment sums never write the match");
  const Pack3 own = load_pack(xo, i, nown);
  float2 ro[EMD_LEVELS];
#pragma unroll
  for (int j = 0; j < EMD_LEVELS; ++j) ro[j] = bc2(0.f);
  if (rebuild) {
    const int i0 = min(i, nown - 1), i1 = min(i + 1, nown - 1);
#pragma unroll
    for (int j = 0; j < EMD_LEVELS; ++j) ro[j] = make_float2(__ldg(ro_g + j * so + i0), __ldg(ro_g + j * so + i1));
  }
  float2 gx = bc2(0.f), gy = bc2(0.f), gz = bc2(0.f);
  for (int base = 0; base < noth; base += TP) {
    const int tn = min(TP, noth - base);
    __syncthreads();
    for (int t = threadIdx.x; t < tn; t += EMD_THREADS) {
      EmdPt &p = pts[t];
      const float *q = xs + 3 * static_cast<size_t>(base + t);
      p.x = __ldg(q), p.y = __ldg(q + 1), p.z = __ldg(q + 2);
      if (rebuild) {
#pragma unroll
        for (int j = 0; j < EMD_LEVELS; ++j) p.r[j] = __ldg(rs_g + j * ss + base + t);
      }
    }
    __syncthreads();
#pragma unroll 2
    for (int t = 0; t < tn; ++t) {
      const EmdPt &p = pts[t];
      // own - other: x1 - x2 for rows, x2 - x1 for columns (the gradient's direction); squares do not see the sign
      const float2 dx = sub2(own.x, bc2(p.x)), dy = sub2(own.y, bc2(p.y)), dz = sub2(own.z, bc2(p.z));
      const float2 d = emd_dist2(dx, dy, dz);
      float2 mt;
      if (rebuild) {
        mt = emd_rebuild<OWN2>(d, ro, p);
      } else {
        const int o = base + t;
        const size_t e0 = OWN2 ? static_cast<size_t>(min(i, m - 1)) * n + o : static_cast<size_t>(o) * n + min(i, n - 1);
        const size_t e1 = OWN2 ? static_cast<size_t>(min(i + 1, m - 1)) * n + o : static_cast<size_t>(o) * n + min(i + 1, n - 1);
        mt = make_float2(__ldg(mat + e0), __ldg(mat + e1));
      }
      if (WHAT == 0) {
        gx = fma2(make_float2(sqrtf(d.x), sqrtf(d.y)), mt, gx);
      } else if (WHAT == 1) {
        const float2 coef = mul2(mt, make_float2(rsqrtf(fmaxf(d.x, 1e-20f)), rsqrtf(fmaxf(d.y, 1e-20f))));
        gx = fma2(coef, dx, gx), gy = fma2(coef, dy, gy), gz = fma2(coef, dz, gz);
      } else {
        float *row = out + (static_cast<size_t>(b) * m + base + t) * n;
        if (i < n) row[i] = mt.x;
        if (i + 1 < n) row[i + 1] = mt.y;
      }
    }
  }
  if (WHAT == 0) {
    float *rc = out + (SEG ? static_cast<size_t>(lo_own) : static_cast<size_t>(b) * m);
    if (i < m) rc[i] = gx.x;
    if (i + 1 < m) rc[i + 1] = gx.y;
  } else if (WHAT == 1) {
    const float g = __ldg(gcost + b);
    float *go = out + (SEG ? 3 * static_cast<size_t>(lo_own) : static_cast<size_t>(b) * nown * 3);
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      if (i + h < nown) {
        go[3 * (i + h)] = __fmul_rn(g, h ? gx.y : gx.x);
        go[3 * (i + h) + 1] = __fmul_rn(g, h ? gy.y : gy.x);
        go[3 * (i + h) + 2] = __fmul_rn(g, h ? gz.y : gz.x);
      }
    }
  }
}

// The cost of one cloud from its rowcost (m), on one 256-thread CTA: thread t sums rowcost[t + 256 i] for ascending i
// from +0, then a fixed pairwise tree p[t] += p[t + s], s = 128, 64, ..., 1.  Every thread of the CTA calls it; the
// result is p[0], read by thread 0 after the call.
__device__ __forceinline__ void emd_cost_reduce_body(const float *__restrict__ rc, int m, float *p /*[256]*/) {
  const int t = threadIdx.x;
  float s = 0.f;
  for (int l = t; l < m; l += 256) s = __fadd_rn(s, rc[l]);
  p[t] = s;
  __syncthreads();
  for (int w = 128; w > 0; w >>= 1) {
    if (t < w) p[t] = __fadd_rn(p[t], p[t + w]);
    __syncthreads();
  }
}

// grid of `clusters` clusters of `cs` CTAs (cs == 1: no cluster attribute), EMD_THREADS threads each
template <typename... P, typename... A>
static cudaError_t emd_launch_clusters(void (*kernel)(P...), long long clusters, int cs, cudaStream_t st, A &&...args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(static_cast<unsigned>(clusters * cs), 1, 1);
  cfg.blockDim = dim3(EMD_THREADS, 1, 1);
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = cs;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = cs > 1 ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<A &&>(args)...);
}

// CTAs per cloud: double while the grid is under two CTAs per SM and every CTA still owns a chunk of the larger cloud
static int emd_cluster_size(int b, int n, int m) {
  const int sms = sm_count(), big = n > m ? n : m;
  int cs = 1;
  while (cs < EMD_MAX_CLUSTER && static_cast<long long>(b) * cs < 2LL * sms && cs * 2 * EMD_CHUNK <= big) cs *= 2;
  return cs;
}

}  // namespace pdae
