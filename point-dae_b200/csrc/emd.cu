// emd.cu -- approximate Earth Mover's Distance (Fan et al. 2017 `approxmatch` / `matchcost` / `matchcostgrad`, the
// reference's extensions/emd, module `emd_cuda`) without the (B, m, n) match matrix.
//
// approxmatch runs 10 levels of three passes each (include/pointdae_b200.h gives the arithmetic).  Per level the match
// only accumulates w(k,l) = (e_j(k,l) * ratioL_j[k]) * ratioR_j[l], so the kernel stores the per-level ratios
// (B,10,n) and (B,10,m) -- 80 bytes per point -- and every consumer of the match rebuilds it from them with the same
// expression in the same order.  Every row and column sum is one thread's sequential chain over the whole other
// cloud, so the bits do not depend on how clouds are split over CTAs: a cloud gets one CTA when the batch fills the
// GPU and a cluster of up to 8 CTAs otherwise, chosen from B and the SM count.  The CTAs of a cluster exchange
// remainR / ratioL / ratioR through the global (L2) arrays, read with ld.global.cg after one cluster barrier per pass.
// The other cloud streams through shared-memory tiles; the distance and the sums use packed f32x2 operations.
#include <cooperative_groups.h>

#include "common.cuh"

namespace cg = cooperative_groups;

namespace pdae {

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

struct EmdMatchArgs {
  const float *xyz1, *xyz2;
  int n, m, cs;
  float *ratio_l, *ratio_r;  // (B,10,n), (B,10,m)
  float *remain_l, *remain_r;  // workspace (B,n), (B,m)
};

// grid: B * cs CTAs, clusters of cs (cs == 1: no cluster).  Owned chunks of EMD_CHUNK points go round-robin to ranks.
__global__ void __launch_bounds__(EMD_THREADS) emd_approxmatch_kernel(const EmdMatchArgs a) {
  __shared__ float4 tile[EMD_TILE];
  const int cs = a.cs, n = a.n, m = a.m;
  const int b = blockIdx.x / cs, rank = blockIdx.x % cs, tid = threadIdx.x;
  const float *x1 = a.xyz1 + static_cast<size_t>(b) * n * 3, *x2 = a.xyz2 + static_cast<size_t>(b) * m * 3;
  float *rl = a.ratio_l + static_cast<size_t>(b) * EMD_LEVELS * n, *rr = a.ratio_r + static_cast<size_t>(b) * EMD_LEVELS * m;
  float *reml = a.remain_l + static_cast<size_t>(b) * n, *remr = a.remain_r + static_cast<size_t>(b) * m;
  const float multl = n >= m ? 1.f : static_cast<float>(m / n), multr = n >= m ? static_cast<float>(n / m) : 1.f;
  const int nch_n = (n + EMD_CHUNK - 1) / EMD_CHUNK, nch_m = (m + EMD_CHUNK - 1) / EMD_CHUNK;
  for (int i = rank * EMD_THREADS + tid; i < n; i += cs * EMD_THREADS) reml[i] = multl;
  for (int i = rank * EMD_THREADS + tid; i < m; i += cs * EMD_THREADS) remr[i] = multr;
  emd_cluster_sync(cs);
  for (int j = 0; j < EMD_LEVELS; ++j) {
    const float c = emd_scale(j);
    float *rlj = rl + static_cast<size_t>(j) * n, *rrj = rr + static_cast<size_t>(j) * m;
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

struct EmdSumArgs {
  const float *xyz1, *xyz2;
  int n, m;
  const float *match;              // (B,m,n) or null: rebuilt from the ratios
  const float *ratio_l, *ratio_r;  // (B,10,n), (B,10,m)
};

// The owned pack's sums over the whole other cloud, ascending.  Rows (OWN2 = false) or columns (OWN2 = true), one
// CTA per EMD_CHUNK owned points (grid.x) and cloud (grid.y).
//   WHAT 0 (columns): rowcost[l] = sum_k fma(sqrtf(d), match[l][k], .)
//   WHAT 1: grad[p] = g_b * sum fma(rn(match * rsqrtf(fmaxf(d, 1e-20))), p - other, .) per coordinate
//   WHAT 2 (rows, no match given): match[l][k] written from the ratios
template <bool OWN2, int WHAT>
__global__ void __launch_bounds__(EMD_THREADS) emd_sum_kernel(const EmdSumArgs a, const float *__restrict__ gcost,
                                                              float *__restrict__ out) {
  __shared__ float4 tile[EMD_TILE / 4 * 4];  // EMD_TILE / 4 points of 4 float4s
  EmdPt *pts = reinterpret_cast<EmdPt *>(tile);
  constexpr int TP = EMD_TILE / 4;
  const int b = blockIdx.y, tid = threadIdx.x;
  const int n = a.n, m = a.m, nown = OWN2 ? m : n, noth = OWN2 ? n : m;
  const float *xo = (OWN2 ? a.xyz2 : a.xyz1) + static_cast<size_t>(b) * nown * 3;
  const float *xs = (OWN2 ? a.xyz1 : a.xyz2) + static_cast<size_t>(b) * noth * 3;
  const float *ro_g = (OWN2 ? a.ratio_r : a.ratio_l) + static_cast<size_t>(b) * EMD_LEVELS * nown;
  const float *rs_g = (OWN2 ? a.ratio_l : a.ratio_r) + static_cast<size_t>(b) * EMD_LEVELS * noth;
  const bool rebuild = a.match == nullptr;
  const float *mat = rebuild ? nullptr : a.match + static_cast<size_t>(b) * m * n;
  const int i = blockIdx.x * EMD_CHUNK + 2 * tid;
  const Pack3 own = load_pack(xo, i, nown);
  float2 ro[EMD_LEVELS];
#pragma unroll
  for (int j = 0; j < EMD_LEVELS; ++j) ro[j] = bc2(0.f);
  if (rebuild) {
    const int i0 = min(i, nown - 1), i1 = min(i + 1, nown - 1);
#pragma unroll
    for (int j = 0; j < EMD_LEVELS; ++j) ro[j] = make_float2(__ldg(ro_g + j * nown + i0), __ldg(ro_g + j * nown + i1));
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
        for (int j = 0; j < EMD_LEVELS; ++j) p.r[j] = __ldg(rs_g + j * noth + base + t);
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
    float *rc = out + static_cast<size_t>(b) * m;
    if (i < m) rc[i] = gx.x;
    if (i + 1 < m) rc[i + 1] = gx.y;
  } else if (WHAT == 1) {
    const float g = __ldg(gcost + b);
    float *go = out + static_cast<size_t>(b) * nown * 3;
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

// cost[b]: thread t sums rowcost[t + 256 i] for ascending i from +0, then a fixed pairwise tree p[t] += p[t + s],
// s = 128, 64, ..., 1
__global__ void __launch_bounds__(256) emd_cost_reduce_kernel(const float *__restrict__ rowcost, int m, float *__restrict__ cost) {
  __shared__ float p[256];
  const int b = blockIdx.x, t = threadIdx.x;
  const float *rc = rowcost + static_cast<size_t>(b) * m;
  float s = 0.f;
  for (int l = t; l < m; l += 256) s = __fadd_rn(s, rc[l]);
  p[t] = s;
  __syncthreads();
  for (int w = 128; w > 0; w >>= 1) {
    if (t < w) p[t] = __fadd_rn(p[t], p[t + w]);
    __syncthreads();
  }
  if (t == 0) cost[b] = p[0];
}

static size_t emd_ws_bytes(int b, int n, int m) {
  return align256(static_cast<size_t>(b) * n * sizeof(float)) + align256(static_cast<size_t>(b) * m * sizeof(float));
}

// CTAs per cloud: double while the grid is under two CTAs per SM and every CTA still owns a chunk of the larger cloud
static int emd_cluster_size(int b, int n, int m) {
  const int sms = sm_count(), big = n > m ? n : m;
  int cs = 1;
  while (cs < EMD_MAX_CLUSTER && static_cast<long long>(b) * cs < 2LL * sms && cs * 2 * EMD_CHUNK <= big) cs *= 2;
  return cs;
}

static int emd_check(const float *xyz1, const float *xyz2, int b, int n, int m) {
  if (b < 0 || n <= 0 || m <= 0) return PDAE_E_INVALID;
  if (n > EMD_MAX_POINTS || m > EMD_MAX_POINTS || b > 65535) return PDAE_E_UNSUPPORTED;
  if (b && (!xyz1 || !xyz2)) return PDAE_E_INVALID;
  return 0;
}

}  // namespace pdae

using namespace pdae;

extern "C" size_t pdae_emd_workspace_bytes(int b, int n, int m) {
  if (b <= 0 || n <= 0 || m <= 0) return 0;
  return emd_ws_bytes(b, n, m);
}

extern "C" int pdae_emd_match_f32(const float *xyz1, const float *xyz2, int b, int n, int m, float *ratio_l, float *ratio_r,
                                  float *match, void *workspace, size_t workspace_bytes, pdae_stream_t stream) {
  const int rc = emd_check(xyz1, xyz2, b, n, m);
  if (rc || b == 0) return rc;
  if (!ratio_l || !ratio_r) return PDAE_E_INVALID;
  if (!workspace || workspace_bytes < emd_ws_bytes(b, n, m)) return PDAE_E_WORKSPACE;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  float *reml = static_cast<float *>(workspace);
  float *remr = reinterpret_cast<float *>(static_cast<unsigned char *>(workspace) + align256(static_cast<size_t>(b) * n * 4));
  const int cs = emd_cluster_size(b, n, m);
  const EmdMatchArgs args{xyz1, xyz2, n, m, cs, ratio_l, ratio_r, reml, remr};
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(static_cast<unsigned>(b) * cs, 1, 1);
  cfg.blockDim = dim3(EMD_THREADS, 1, 1);
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = cs;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = cs > 1 ? 1 : 0;
  PDAE_CUDA_TRY(cudaLaunchKernelEx(&cfg, emd_approxmatch_kernel, args));
  if (match) {
    const EmdSumArgs s{xyz1, xyz2, n, m, nullptr, ratio_l, ratio_r};
    emd_sum_kernel<false, 2><<<dim3(ceil_div(n, EMD_CHUNK), b), EMD_THREADS, 0, st>>>(s, nullptr, match);
    PDAE_RETURN_IF_LAUNCH_FAILED();
  }
  return 0;
}

extern "C" int pdae_emd_cost_f32(const float *xyz1, const float *xyz2, int b, int n, int m, const float *match,
                                 const float *ratio_l, const float *ratio_r, float *cost, void *workspace,
                                 size_t workspace_bytes, pdae_stream_t stream) {
  const int rc = emd_check(xyz1, xyz2, b, n, m);
  if (rc || b == 0) return rc;
  if (!cost || (!match && (!ratio_l || !ratio_r))) return PDAE_E_INVALID;
  if (!workspace || workspace_bytes < emd_ws_bytes(b, n, m)) return PDAE_E_WORKSPACE;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  float *rowcost = static_cast<float *>(workspace);
  const EmdSumArgs s{xyz1, xyz2, n, m, match, ratio_l, ratio_r};
  emd_sum_kernel<true, 0><<<dim3(ceil_div(m, EMD_CHUNK), b), EMD_THREADS, 0, st>>>(s, nullptr, rowcost);
  PDAE_RETURN_IF_LAUNCH_FAILED();
  emd_cost_reduce_kernel<<<b, 256, 0, st>>>(rowcost, m, cost);
  PDAE_RETURN_IF_LAUNCH_FAILED();
  return 0;
}

extern "C" int pdae_emd_cost_grad_f32(const float *grad_cost, const float *xyz1, const float *xyz2, int b, int n, int m,
                                      const float *match, const float *ratio_l, const float *ratio_r, float *grad1,
                                      float *grad2, pdae_stream_t stream) {
  const int rc = emd_check(xyz1, xyz2, b, n, m);
  if (rc || b == 0) return rc;
  if (!grad_cost || !grad1 || !grad2 || (!match && (!ratio_l || !ratio_r))) return PDAE_E_INVALID;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const EmdSumArgs s{xyz1, xyz2, n, m, match, ratio_l, ratio_r};
  emd_sum_kernel<false, 1><<<dim3(ceil_div(n, EMD_CHUNK), b), EMD_THREADS, 0, st>>>(s, grad_cost, grad1);
  PDAE_RETURN_IF_LAUNCH_FAILED();
  emd_sum_kernel<true, 1><<<dim3(ceil_div(m, EMD_CHUNK), b), EMD_THREADS, 0, st>>>(s, grad_cost, grad2);
  PDAE_RETURN_IF_LAUNCH_FAILED();
  return 0;
}
