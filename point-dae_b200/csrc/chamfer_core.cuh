// chamfer_core.cuh -- the Chamfer scan body and the Chamfer backward, shared by the equal-size entry points
// (chamfer.cu) and the segment entry points (segchamfer.cu).  Semantics and design: see chamfer.cu.
#pragma once
#include "common.cuh"
#include "reverse.cuh"

namespace pdae {

constexpr int CH_GROUP = 16;    // argmin bookkeeping granularity: four LDS.128 steps = 16 reference points
constexpr int CH_THREADS = 128; // threads of a scan CTA: one 4-warp CTA already saturates an SM's FMA issue
constexpr int CH_TILE = 512;    // reference points per shared-memory tile
constexpr int CH_STEP = 8;      // reference points per inner step: QT*CH_STEP distances are live at once
static_assert(3 * CH_TILE % CH_THREADS == 0, "tile must split evenly over the CTA");
static_assert(CH_TILE % CH_GROUP == 0, "tile must hold whole bookkeeping groups");
static_assert(CH_STEP == 8, "the running-minimum update of chamfer_min_body takes eight distances per query");

// SYM: the squared distance is symmetric bit for bit (the operands of every product only change
// sign), so one evaluation of pair (a_i, b_j) serves both directions: besides the per-query running
// minimum the kernel reduces, for every reference point, the minimum over the warp's 32*QT queries
// (FMNMX3 across the thread's queries, one REDUX.MIN across the lanes) and posts
// (min bits << 32 | query-group id) with a 64-bit RED.MIN per CTA; the column recovery of chamfer.cu then
// finds the lowest query index inside the winning group.  Halves the FMA-pipe work of the forward.
// One pass of a CTA: rows [row_base, row_base + QT*CH_THREADS) of cloud `Q` (clamped to nq) against all nr points of
// `R`.  A warp names itself in the column keys by the id of its 32*QT-row group, row_base / (32*QT) + warp.
// The shared-memory buffers belong to the caller.
// SEG (segment forward, segchamfer.cu): `R` is a segment of a packed cloud and may start at any row, so the index
// recovery takes float4 loads only when R itself is 16-byte aligned; idx is written as ref_offset + local index.
template <int QT, bool SYM, bool SEG = false>
__device__ __forceinline__ void chamfer_min_body(const float *__restrict__ Q, const float *__restrict__ R, int nq, int nr,
                                                 int row_base, size_t cloud, float *dist, int *idx, uint64_t *keys,
                                                 int ref_offset, uint64_t *colkeys, float (*tile)[3][CH_TILE],
                                                 unsigned (*colmin)[CH_THREADS / 32][SYM ? CH_TILE : 4], int tile_begin = 0,
                                                 int tile_end = 0x7fffffff, bool merge = false) {
  constexpr int QPW = 32 * QT;                  // queries per warp
  constexpr int W = CH_THREADS / 32;
  constexpr int LD = 3 * CH_TILE / CH_THREADS;  // floats staged per thread per tile

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int qbase = row_base + warp * QPW;

  float2 qx[QT], qy[QT], qz[QT];
  float best[QT];
  int bgrp[QT];
#pragma unroll
  for (int s = 0; s < QT; ++s) {
    int q = qbase + s * 32 + lane;
    q = q < nq ? q : nq - 1;
    const float x = __ldg(Q + 3 * q), y = __ldg(Q + 3 * q + 1), z = __ldg(Q + 3 * q + 2);
    qx[s] = make_float2(x, x);
    qy[s] = make_float2(y, y);
    qz[s] = make_float2(z, z);
    best[s] = __int_as_float(0x7f800000);
    bgrp[s] = 0;
  }

  float pre[LD];
  const int nr3 = nr * 3;
  auto fetch = [&](int tile_base) {
#pragma unroll
    for (int i = 0; i < LD; ++i) {
      const int f = tid + i * CH_THREADS;
      const int g = tile_base * 3 + f;
      // padding: x = +inf makes the padded distance +inf, which never lowers a minimum
      pre[i] = g < nr3 ? __ldg(R + g) : ((f % 3 == 0) ? __int_as_float(0x7f800000) : 0.0f);
    }
  };
  auto stash = [&](int buf) {
#pragma unroll
    for (int i = 0; i < LD; ++i) {
      const int f = tid + i * CH_THREADS;
      const int p = f / 3, c = f - 3 * p;
      tile[buf][c][p] = pre[i];
    }
  };

  // SYM: post the per-warp column minima of tile `tp` (complete since the last barrier)
  auto flush_cols = [&](int tp) {
    if (!SYM) return;
    uint64_t *ck = colkeys + cloud * nr;
    const int tb = tp * CH_TILE;
    for (int j = tid; j < CH_TILE && tb + j < nr; j += CH_THREADS) {
      unsigned v = colmin[tp & 1][0][j];
      int wm = 0;
#pragma unroll
      for (int w = 1; w < W; ++w) {
        const unsigned u = colmin[tp & 1][w][j];
        wm = u < v ? w : wm;
        v = u < v ? u : v;
      }
      const unsigned who = static_cast<unsigned>(row_base / QPW + wm);
      atomicMin(reinterpret_cast<unsigned long long *>(ck + tb + j), (static_cast<unsigned long long>(v) << 32) | who);
    }
  };

  // a CTA streams tiles [tile_begin, ntiles) of the reference cloud: all of them, or one column chunk of a split unit
  const int ntiles_all = (nr + CH_TILE - 1) / CH_TILE;
  const int ntiles = tile_end < ntiles_all ? tile_end : ntiles_all;
  fetch(tile_begin * CH_TILE);
  stash(tile_begin & 1);
  __syncthreads();
  for (int tl = tile_begin; tl < ntiles; ++tl) {
    const bool more = tl + 1 < ntiles;
    if (more) fetch((tl + 1) * CH_TILE);
    if (tl > tile_begin) flush_cols(tl - 1);
    const float *sx = tile[tl & 1][0], *sy = tile[tl & 1][1], *sz = tile[tl & 1][2];
    unsigned pend[CH_STEP];
#pragma unroll
    for (int r = 0; r < CH_STEP; ++r) pend[r] = 0u;
    int pend_off = -1;
    auto store_pend = [&]() {  // lane 0 parks the warp's column minima of one step
      uint4 *dst = reinterpret_cast<uint4 *>(&colmin[tl & 1][warp][pend_off]);
#pragma unroll
      for (int r = 0; r < CH_STEP; r += 4) dst[r >> 2] = make_uint4(pend[r], pend[r + 1], pend[r + 2], pend[r + 3]);
    };
    const int left = nr - tl * CH_TILE;
    const int ngroups = ((left < CH_TILE ? left : CH_TILE) + CH_GROUP - 1) / CH_GROUP;
    const int group_base = tl * (CH_TILE / CH_GROUP);
#pragma unroll 2
    for (int g = 0; g < ngroups; ++g) {
      const int gid = group_base + g;
      float cur[QT];
#pragma unroll
      for (int s = 0; s < QT; ++s) cur[s] = best[s];
#pragma unroll
      for (int h = 0; h < CH_GROUP; h += CH_STEP) {
        float4 X[CH_STEP / 4], Y[CH_STEP / 4], Z[CH_STEP / 4];
#pragma unroll
        for (int v = 0; v < CH_STEP / 4; ++v) {
          X[v] = *reinterpret_cast<const float4 *>(sx + g * CH_GROUP + h + 4 * v);
          Y[v] = *reinterpret_cast<const float4 *>(sy + g * CH_GROUP + h + 4 * v);
          Z[v] = *reinterpret_cast<const float4 *>(sz + g * CH_GROUP + h + 4 * v);
        }
        float2 dd[QT][CH_STEP / 2];
#pragma unroll
        for (int s = 0; s < QT; ++s) {
#pragma unroll
          for (int v = 0; v < CH_STEP / 4; ++v) {
            dd[s][2 * v] = dist_yxz2(sub2(make_float2(X[v].x, X[v].y), qx[s]), sub2(make_float2(Y[v].x, Y[v].y), qy[s]),
                                     sub2(make_float2(Z[v].x, Z[v].y), qz[s]));
            dd[s][2 * v + 1] = dist_yxz2(sub2(make_float2(X[v].z, X[v].w), qx[s]), sub2(make_float2(Y[v].z, Y[v].w), qy[s]),
                                         sub2(make_float2(Z[v].z, Z[v].w), qz[s]));
          }
          const float t0 = min3(dd[s][0].x, dd[s][0].y, dd[s][1].x);
          const float t1 = min3(dd[s][1].y, dd[s][2].x, dd[s][2].y);
          const float t2 = min3(dd[s][3].x, dd[s][3].y, t0);
          cur[s] = min3(cur[s], t1, t2);
        }
        if (SYM) {  // column minima over this warp's 32*QT queries for the CH_STEP reference points of the step
          // the REDUX results of the previous step are stored only now, a full step of FMA work later, so
          // their latency never stalls the warp
          if (pend_off >= 0 && lane == 0) store_pend();
#pragma unroll
          for (int r = 0; r < CH_STEP; ++r) {
            float c = (r & 1) ? dd[0][r >> 1].y : dd[0][r >> 1].x;
#pragma unroll
            for (int s = 1; s + 1 < QT; s += 2)
              c = min3(c, (r & 1) ? dd[s][r >> 1].y : dd[s][r >> 1].x, (r & 1) ? dd[s + 1][r >> 1].y : dd[s + 1][r >> 1].x);
            if ((QT & 1) == 0) c = fminf(c, (r & 1) ? dd[QT - 1][r >> 1].y : dd[QT - 1][r >> 1].x);
            pend[r] = __reduce_min_sync(0xffffffffu, __float_as_uint(c));
          }
          pend_off = g * CH_GROUP + h;
        }
      }
#pragma unroll
      for (int s = 0; s < QT; ++s) {
        bgrp[s] = cur[s] < best[s] ? gid : bgrp[s];
        best[s] = cur[s];
      }
    }
    if (SYM && pend_off >= 0 && lane == 0) store_pend();
    if (more) stash((tl + 1) & 1);
    __syncthreads();
  }
  flush_cols(ntiles - 1);

  // ---- index recovery: each thread rescans the one 16-point group recorded per query ----------
  // (scanned back to front so the lowest matching index is the one kept)
  int myidx[QT];
  // equal-size clouds: every cloud then starts 16-byte aligned.  A segment: R + 3*base is aligned exactly when R is
  const bool vec_ok = SEG ? (reinterpret_cast<uintptr_t>(R) & 15u) == 0 : (nr & 3) == 0;
#pragma unroll
  for (int s = 0; s < QT; ++s) {
    const int base = bgrp[s] * CH_GROUP;
    int found = 0;
    if (vec_ok && base + CH_GROUP <= nr) {
      const float4 *p4 = reinterpret_cast<const float4 *>(R + 3 * static_cast<size_t>(base));
      float v[3 * CH_GROUP];
#pragma unroll
      for (int t = 0; t < 3 * CH_GROUP / 4; ++t) {
        const float4 w = __ldg(p4 + t);
        v[4 * t] = w.x; v[4 * t + 1] = w.y; v[4 * t + 2] = w.z; v[4 * t + 3] = w.w;
      }
#pragma unroll
      for (int t = CH_GROUP - 1; t >= 0; --t) {
        const float d = dist_yxz(__fsub_rn(v[3 * t], qx[s].x), __fsub_rn(v[3 * t + 1], qy[s].x), __fsub_rn(v[3 * t + 2], qz[s].x));
        found = (d == best[s]) ? base + t : found;
      }
    } else {
#pragma unroll
      for (int t = CH_GROUP - 1; t >= 0; --t) {
        const int j = base + t;
        if (j < nr) {
          const float bx = __ldg(R + 3 * j), by = __ldg(R + 3 * j + 1), bz = __ldg(R + 3 * j + 2);
          const float d = dist_yxz(__fsub_rn(bx, qx[s].x), __fsub_rn(by, qy[s].x), __fsub_rn(bz, qz[s].x));
          found = (d == best[s]) ? j : found;
        }
      }
    }
    myidx[s] = found;
  }

#pragma unroll
  for (int s = 0; s < QT; ++s) {
    const int q = qbase + s * 32 + lane;
    if (q < nq) {
      const size_t o = cloud * nq + q;
      if (keys) {
        const uint64_t key = pack_key(best[s], static_cast<uint32_t>(myidx[s] + ref_offset));
        // column-split unit: the (distance, index) order of the key is the reference's tie rule
        if (merge) atomicMin(reinterpret_cast<unsigned long long *>(keys + o), key);
        else keys[o] = key;
      } else {
        dist[o] = best[s];
        idx[o] = SEG ? myidx[s] + ref_offset : myidx[s];
      }
    }
  }
}

// ---- backward: one thread per point of either cloud, scatter through the saved argmin ---------
// reference: chamfer.cu:173-201 runs (1,16)x256 = 4096 threads over the whole batch and adds BOTH terms of every
// pair with atomics into zero-filled buffers.  Every point receives exactly one "own" term (g * (a_j - b_idx[j]),
// written by its own thread) plus the scattered terms of the points that chose it, so the work is split in two
// launches over all b*(n+m) points: OWN stores the own term with a plain store (which also initialises the
// buffer: no memset), SCATTER then adds -v to the matched point with RED.ADD.F32.  Half the atomics of the
// reference scheme, accumulation order free as in the reference.
//
// GradSrc supplies d(loss)/d(dist) per point: the arrays handed to chamfer.backward, or -- for the fused mean
// losses (ChamferDistanceL2 / L1) -- the upstream scalar times a constant, with the sqrt derivative for L1.
struct GradArrays {
  const float *gd1, *gd2;
  __device__ __forceinline__ float at(bool second, size_t o) const { return __ldg((second ? gd2 : gd1) + o); }
};
struct GradMean {
  const float *gloss;          // upstream gradient of the scalar loss (device)
  const float *dist1, *dist2;  // squared distances of the forward (L1 only)
  float w1, w2;                // d(loss)/d(mean term) / count
  int l1;
  __device__ __forceinline__ float at(bool second, size_t o) const {
    const float g = __fmul_rn(__ldg(gloss), second ? w2 : w1);
    if (!l1) return g;
    // d sqrt(x) = g / (2 sqrt(x)); x == 0 gives inf like torch's SqrtBackward (and NaN after the multiply by 0)
    return __fdiv_rn(g, __fmul_rn(2.0f, __fsqrt_rn(__ldg((second ? dist2 : dist1) + o))));
  }
};

// SEG (segment entry points only): idx < 0 marks a point without a match (its opposite segment is empty); it gets no
// own term and scatters nothing.  The equal-size instantiations (SEG = false) carry no such test.
template <bool SCATTER, typename GradSrc, bool SEG = false>
__global__ void __launch_bounds__(256) chamfer_bwd_kernel(const float *__restrict__ xyz1, const float *__restrict__ xyz2,
                                                          const int *__restrict__ idx1, const int *__restrict__ idx2,
                                                          const GradSrc gs, int n, int m, int blocks_per_cloud,
                                                          float *__restrict__ gx1, float *__restrict__ gx2) {
  const unsigned cloud_u = blockIdx.x / blocks_per_cloud;  // 1-D grid: no 65535-cloud limit (the fine loss has thousands)
  int i = (blockIdx.x - cloud_u * blocks_per_cloud) * blockDim.x + threadIdx.x;  // point of cloud 1 (i < n) or 2 (i - n < m)
  const size_t cloud = cloud_u;
  const bool second = i >= n;
  const float *A, *Bp;
  const int *idx;
  float *ga, *gb;
  size_t o;
  if (!second) {
    A = xyz1 + cloud * n * 3; Bp = xyz2 + cloud * m * 3; idx = idx1 + cloud * n; o = cloud * n + i;
    ga = gx1 + cloud * n * 3; gb = gx2 + cloud * m * 3;
  } else {
    i -= n;
    if (i >= m) return;
    A = xyz2 + cloud * m * 3; Bp = xyz1 + cloud * n * 3; idx = idx2 + cloud * m; o = cloud * m + i;
    ga = gx2 + cloud * m * 3; gb = gx1 + cloud * n * 3;
  }
  const int j2 = __ldg(idx + i);
  if (SEG && j2 < 0) {
    if (!SCATTER) ga[3 * i] = ga[3 * i + 1] = ga[3 * i + 2] = 0.0f;
    return;
  }
  const float g = __fmul_rn(gs.at(second, o), 2.0f);
  float v[3];
#pragma unroll
  for (int c = 0; c < 3; ++c) v[c] = __fmul_rn(g, __fsub_rn(__ldg(A + 3 * i + c), __ldg(Bp + 3 * j2 + c)));
  if (!SCATTER) {
#pragma unroll
    for (int c = 0; c < 3; ++c) ga[3 * i + c] = v[c];
  } else {
    // two reductions per point instead of three: a point's 12 bytes always hold one 8-byte aligned pair (x,y for an even
    // point of an 8-byte aligned cloud, y,z for an odd one) -> one RED.ADD.v2.f32 + one scalar RED.ADD.F32
    float *t = gb + 3 * j2;
    if ((reinterpret_cast<uintptr_t>(t) & 7u) == 0) {
      atomicAdd(reinterpret_cast<float2 *>(t), make_float2(-v[0], -v[1]));
      atomicAdd(t + 2, -v[2]);
    } else if ((reinterpret_cast<uintptr_t>(t + 1) & 7u) == 0) {
      atomicAdd(t, -v[0]);
      atomicAdd(reinterpret_cast<float2 *>(t + 1), make_float2(-v[1], -v[2]));
    } else {
#pragma unroll
      for (int c = 0; c < 3; ++c) atomicAdd(t + c, -v[c]);
    }
  }
}

template <typename GradSrc, bool SEG = false>
static int launch_chamfer_bwd(const float *xyz1, const float *xyz2, const int *idx1, const int *idx2, const GradSrc &gs,
                              int b, int n, int m, float *gx1, float *gx2, cudaStream_t st) {
  const long long bpc = (static_cast<long long>(n) + m + 255) / 256;
  if (bpc * b > 0x7fffffffLL) return PDAE_E_UNSUPPORTED;
  const unsigned grid = static_cast<unsigned>(bpc * b);
  chamfer_bwd_kernel<false, GradSrc, SEG><<<grid, 256, 0, st>>>(xyz1, xyz2, idx1, idx2, gs, n, m, static_cast<int>(bpc), gx1, gx2);
  PDAE_RETURN_IF_LAUNCH_FAILED();
  chamfer_bwd_kernel<true, GradSrc, SEG><<<grid, 256, 0, st>>>(xyz1, xyz2, idx1, idx2, gs, n, m, static_cast<int>(bpc), gx1, gx2);
  PDAE_RETURN_IF_LAUNCH_FAILED();
  return 0;
}

// ---- deterministic backward: the same terms gathered per point in a defined order, no float atomics ------------------
// Point i of cloud 1 gets its own term g_i (a_i - b_idx1[i]), then -v_j for every point j of cloud 2 with idx2[j] == i,
// j ascending, with rounded fp32 adds (cloud 2 symmetric).  rev1 lists, per point of cloud 1, the points of cloud 2
// that chose it (the ordered reverse map of idx2), rev2 the converse.
template <typename GradSrc, bool SEG = false>
__global__ void __launch_bounds__(256) chamfer_bwd_det_kernel(const float *__restrict__ xyz1, const float *__restrict__ xyz2,
                                                              const int *__restrict__ idx1, const int *__restrict__ idx2,
                                                              const GradSrc gs, int n, int m, int blocks_per_cloud, RevMap rev1,
                                                              RevMap rev2, float *__restrict__ gx1, float *__restrict__ gx2) {
  const unsigned cloud_u = blockIdx.x / blocks_per_cloud;
  int i = (blockIdx.x - cloud_u * blocks_per_cloud) * blockDim.x + threadIdx.x;
  const size_t cloud = cloud_u;
  const bool second = i >= n;
  const float *A, *Bp;
  const int *idx, *rp, *rs;
  float *ga;
  size_t o, so;
  if (!second) {
    A = xyz1 + cloud * n * 3; Bp = xyz2 + cloud * m * 3; idx = idx1 + cloud * n; o = cloud * n + i;
    ga = gx1 + cloud * n * 3; so = cloud * m;
    rp = rev1.ptr + cloud * (n + 1); rs = rev1.slot + cloud * m;
  } else {
    i -= n;
    if (i >= m) return;
    A = xyz2 + cloud * m * 3; Bp = xyz1 + cloud * n * 3; idx = idx2 + cloud * m; o = cloud * m + i;
    ga = gx2 + cloud * m * 3; so = cloud * n;
    rp = rev2.ptr + cloud * (m + 1); rs = rev2.slot + cloud * n;
  }
  const int j2 = __ldg(idx + i);
  const bool own = !SEG || j2 >= 0;  // SEG: a point without a match has no own term
  const float g = own ? __fmul_rn(gs.at(second, o), 2.0f) : 0.0f;
  float a[3], acc[3];
#pragma unroll
  for (int c = 0; c < 3; ++c) a[c] = __ldg(A + 3 * i + c);
#pragma unroll
  for (int c = 0; c < 3; ++c) acc[c] = own ? __fmul_rn(g, __fsub_rn(a[c], __ldg(Bp + 3 * j2 + c))) : 0.0f;
  // the sources live in the other cloud: their own points are Bp, their match (this point) is a
  // buckets longer than REV_SHORT (up to a whole cloud for a collapsed prediction) are written by the warp walk below
  const int lo = __ldg(rp + i), hi = __ldg(rp + i + 1);
  if (hi - lo > REV_SHORT) return;
  for (int q = lo; q < hi; ++q) {
    const int j = __ldg(rs + q);
    const float gj = __fmul_rn(gs.at(!second, so + j), 2.0f);
#pragma unroll
    for (int c = 0; c < 3; ++c) acc[c] = __fadd_rn(acc[c], -__fmul_rn(gj, __fsub_rn(__ldg(Bp + 3 * j + c), a[c])));
  }
#pragma unroll
  for (int c = 0; c < 3; ++c) ga[3 * i + c] = acc[c];
}

// The long buckets (the maps' queues): one warp per target point.  The lanes load 32 sources at a time and form their terms
// in parallel; every lane then adds the 32 terms in source order from the shuffles, so the sum is the one the point kernel
// forms and a bucket of a whole cloud costs its serial adds, not a load latency per source.
template <typename GradSrc, bool SEG = false>
__global__ void __launch_bounds__(256) chamfer_bwd_det_long_kernel(const float *__restrict__ xyz1, const float *__restrict__ xyz2,
                                                                   const int *__restrict__ idx1, const int *__restrict__ idx2,
                                                                   const GradSrc gs, int n, int m, RevMap rev1, RevMap rev2,
                                                                   float *__restrict__ gx1, float *__restrict__ gx2) {
  const int lane = threadIdx.x & 31;
  const int n1 = __ldg(rev1.longq), n2 = __ldg(rev2.longq);
  const int stride = static_cast<int>((gridDim.x * blockDim.x) >> 5);
  for (int w = static_cast<int>((blockIdx.x * blockDim.x + threadIdx.x) >> 5); w < n1 + n2; w += stride) {
    const bool second = w >= n1;
    const int u = second ? __ldg(rev2.longq + 1 + (w - n1)) : __ldg(rev1.longq + 1 + w);
    const int t = second ? m : n;
    const size_t cloud = static_cast<size_t>(u / t);
    const int i = u - static_cast<int>(cloud) * t;
    const float *A, *Bp;
    const int *idx, *rp, *rs;
    float *ga;
    size_t o, so;
    if (!second) {
      A = xyz1 + cloud * n * 3; Bp = xyz2 + cloud * m * 3; idx = idx1 + cloud * n; o = cloud * n + i;
      ga = gx1 + cloud * n * 3; so = cloud * m;
      rp = rev1.ptr + cloud * (n + 1); rs = rev1.slot + cloud * m;
    } else {
      A = xyz2 + cloud * m * 3; Bp = xyz1 + cloud * n * 3; idx = idx2 + cloud * m; o = cloud * m + i;
      ga = gx2 + cloud * m * 3; so = cloud * n;
      rp = rev2.ptr + cloud * (m + 1); rs = rev2.slot + cloud * n;
    }
    const int j2 = __ldg(idx + i);
    const bool own = !SEG || j2 >= 0;  // SEG: a point without a match has no own term
    const float g = own ? __fmul_rn(gs.at(second, o), 2.0f) : 0.0f;
    float a[3], acc[3];
#pragma unroll
    for (int c = 0; c < 3; ++c) a[c] = __ldg(A + 3 * i + c);
#pragma unroll
    for (int c = 0; c < 3; ++c) acc[c] = own ? __fmul_rn(g, __fsub_rn(a[c], __ldg(Bp + 3 * j2 + c))) : 0.0f;
    // LW_ROUNDS x 32 sources per pass: their loads are all issued before the first add of the pass
    constexpr int LW_ROUNDS = 4;
    const int lo = __ldg(rp + i), hi = __ldg(rp + i + 1);
    for (int q0 = lo; q0 < hi; q0 += 32 * LW_ROUNDS) {
      int j[LW_ROUNDS];
      float v[LW_ROUNDS][3];
#pragma unroll
      for (int r = 0; r < LW_ROUNDS; ++r) j[r] = q0 + r * 32 + lane < hi ? __ldg(rs + q0 + r * 32 + lane) : -1;
#pragma unroll
      for (int r = 0; r < LW_ROUNDS; ++r) {
        v[r][0] = v[r][1] = v[r][2] = 0.f;
        if (j[r] >= 0) {
          const float gj = __fmul_rn(gs.at(!second, so + j[r]), 2.0f);
#pragma unroll
          for (int c = 0; c < 3; ++c) v[r][c] = -__fmul_rn(gj, __fsub_rn(__ldg(Bp + 3 * j[r] + c), a[c]));
        }
      }
#pragma unroll
      for (int r = 0; r < LW_ROUNDS; ++r) {
        const int cnt = min(32, hi - (q0 + r * 32));
        for (int l = 0; l < cnt; ++l) {
#pragma unroll
          for (int c = 0; c < 3; ++c) acc[c] = __fadd_rn(acc[c], __shfl_sync(0xffffffffu, v[r][c], l));
        }
      }
    }
    if (lane == 0) {
#pragma unroll
      for (int c = 0; c < 3; ++c) ga[3 * i + c] = acc[c];
    }
  }
}

static size_t chamfer_bwd_det_bytes(int b, int n, int m) {
  return (rev_map_bytes(b, m, n) + 255) / 256 * 256 + rev_map_bytes(b, n, m);
}

template <typename GradSrc, bool SEG = false>
static int launch_chamfer_bwd_det(const float *xyz1, const float *xyz2, const int *idx1, const int *idx2, const GradSrc &gs,
                                  int b, int n, int m, float *gx1, float *gx2, void *ws, cudaStream_t st) {
  const long long bpc = (static_cast<long long>(n) + m + 255) / 256;
  if (bpc * b > 0x7fffffffLL) return PDAE_E_UNSUPPORTED;
  RevMap rev1, rev2;
  unsigned char *w = static_cast<unsigned char *>(ws);
  int rc = rev_map_build(idx2, b, m, n, w, &rev1, st);
  if (rc) return rc;
  rc = rev_map_build(idx1, b, n, m, w + (rev_map_bytes(b, m, n) + 255) / 256 * 256, &rev2, st);
  if (rc) return rc;
  chamfer_bwd_det_kernel<GradSrc, SEG><<<static_cast<unsigned>(bpc * b), 256, 0, st>>>(xyz1, xyz2, idx1, idx2, gs, n, m,
                                                                                  static_cast<int>(bpc), rev1, rev2, gx1, gx2);
  PDAE_RETURN_IF_LAUNCH_FAILED();
  if (n > REV_SHORT || m > REV_SHORT) {  // otherwise no bucket can be long
    const long long most = static_cast<long long>(b) * (n / (REV_SHORT + 1) + m / (REV_SHORT + 1));  // long buckets at most
    const long long cap = 4LL * sm_count();
    const long long blocks = (most + 7) / 8 < cap ? (most + 7) / 8 : cap;
    chamfer_bwd_det_long_kernel<GradSrc, SEG><<<static_cast<unsigned>(blocks), 256, 0, st>>>(xyz1, xyz2, idx1, idx2, gs, n, m, rev1,
                                                                                        rev2, gx1, gx2);
    PDAE_RETURN_IF_LAUNCH_FAILED();
  }
  return 0;
}

}  // namespace pdae
