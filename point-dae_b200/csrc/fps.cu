// fps.cu -- furthest point sampling (+ fused centre gather) and gather / gather_grad.
//
// Semantics follow extensions/pointnet2/_ext_src/src/sampling_gpu.cu:72-176 of the reference
// (identical in pointnet2_ops): idx[0] = 0; every later sample maximises the running minimum
// squared distance over the points with (double)|p|^2 > 1e-3; ties are resolved the way the
// reference's block does it -- thread slot `k mod bs` in bit-reversed order first (its shared
// memory tree keeps the lower slot), then the smaller k (its per-thread strict `>`), with
// bs = opt_n_threads(n) (cuda_utils.h:15-21).  That order is encoded as a 32-bit rank so the
// arg-max becomes two warp-wide integer reductions (max of the value bits, then min of the rank
// among the lanes holding that value) instead of a 9-level shared-memory tree with 10 barriers.
//
// Design (latency bound: npoint-1 strictly sequential iterations, one CTA per cloud):
//   * every thread keeps its P points (x, y, z, running min) in registers for the whole call;
//     the cloud is also staged once in shared memory (float4 per point) so the coordinates of
//     the point just selected are one broadcast LDS.128 away;
//   * skipped points and padding carry min = -2, which no update can raise above the -1 a
//     thread starts from, so the inner loop is branch-free;
//   * one __syncthreads per iteration (double-buffered per-warp slots), REDUX for both levels.
//   * clouds too large for one CTA's registers fall back to a variant that keeps the running
//     minima in a global workspace (same arithmetic, same tie rule).
#include <math.h>
#include <stdio.h>
#include <stdlib.h>

#include <cooperative_groups.h>

#include "common.cuh"
#include "reverse.cuh"
#include "fps_rank.cuh"

namespace cg = cooperative_groups;

namespace pdae {

// block-wide arg-max for the register-resident kernel: per-warp winners are posted as ONE 64-bit key
// (value bits << 32 | ~rank: larger value first, then smaller rank) and every thread folds the W keys with a
// register tree after the barrier -- two broadcast LDS.128 and log2(W) dependent 64-bit max instead of a second pair
// of REDUX + uniform-to-vector moves on the critical path of every iteration.
template <int T>
__device__ __forceinline__ unsigned fps_block_argmax_keys(unsigned vb, unsigned rank, unsigned long long *slots /*[2][32]*/,
                                                          int it) {
  constexpr int W = T / 32;
  const unsigned full = 0xffffffffu;
  const unsigned m = __reduce_max_sync(full, vb);
  const unsigned r = __reduce_min_sync(full, vb == m ? rank : 0xffffffffu);
  if (W == 1) return r;
  if constexpr (W > 4) {  // 8+ keys per thread cost more than the second pair of REDUX (measured: 23.0 vs 20.5 us at W = 8)
    return fps_block_argmax<T>(vb, rank, reinterpret_cast<uint2 *>(slots), it);
  } else {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    unsigned long long *buf = slots + (it & 1) * 32;
    if (lane == 0) buf[warp] = (static_cast<unsigned long long>(m) << 32) | static_cast<unsigned>(~r);
    __syncthreads();
    unsigned long long kk[W];
#pragma unroll
    for (int w = 0; w < W; w += 2) {
      const ulonglong2 two = *reinterpret_cast<const ulonglong2 *>(buf + w);
      kk[w] = two.x;
      kk[w + 1] = two.y;
    }
#pragma unroll
    for (int stride = 1; stride < W; stride *= 2)
#pragma unroll
      for (int i = 0; i + stride < W; i += 2 * stride) kk[i] = kk[i] > kk[i + stride] ? kk[i] : kk[i + stride];
    return ~static_cast<unsigned>(kk[0]);
  }
}

// running minima of a thread's P points against the centre just selected.  PACKED: two points per step on the packed fp32
// forms (FADD2 / FMUL2 / FFMA2: IEEE per half, same rounding order as dist_yxz), 6 FMA-pipe instructions per two points
// instead of 12.  Measured on B200: with four warps per scheduler (512-thread CTAs, 8192 -> 512: 755 -> 681 us) the
// update is issue-bound and the packed form wins; with one warp per scheduler (128-thread CTAs, 2048 -> 64) the iteration
// is a latency chain and the packed form is slower (16.9 -> 20.0 us), so those keep the scalar form.
template <int P, bool PACKED>
__device__ __forceinline__ void fps_update(const float (&px)[P], const float (&py)[P], const float (&pz)[P], float (&pt)[P],
                                           float ox, float oy, float oz) {
  if constexpr (!PACKED) {
#pragma unroll
    for (int p = 0; p < P; ++p) {
      const float d = dist_yxz(__fsub_rn(px[p], ox), __fsub_rn(py[p], oy), __fsub_rn(pz[p], oz));
      pt[p] = fminf(d, pt[p]);
    }
    return;
  }
  const float2 ox2 = make_float2(ox, ox), oy2 = make_float2(oy, oy), oz2 = make_float2(oz, oz);
#pragma unroll
  for (int p = 0; p + 1 < P; p += 2) {
    const float2 d2 = dist_yxz2(sub2(make_float2(px[p], px[p + 1]), ox2), sub2(make_float2(py[p], py[p + 1]), oy2),
                                sub2(make_float2(pz[p], pz[p + 1]), oz2));
    pt[p] = fminf(d2.x, pt[p]);
    pt[p + 1] = fminf(d2.y, pt[p + 1]);
  }
  if (P & 1) {
    const float d = dist_yxz(__fsub_rn(px[P - 1], ox), __fsub_rn(py[P - 1], oy), __fsub_rn(pz[P - 1], oz));
    pt[P - 1] = fminf(d, pt[P - 1]);
  }
}

// ---- register-resident variant: n <= T*P -----------------------------------------------------
// S = log2(bs / T) when the CTA is narrower than the reference's block (T < bs = 512): a thread then owns
// 2^S different reference slots, and its registers are laid out in tie-rank order (slot sub-index
// bit-reversed first, then k / bs) so that the in-thread first-maximum scan still reproduces the rule.
// The tie rank of the point in register i needs no bit reversal in the loop: the reversed slot of a thread is a
// constant (its high part) plus the register's slot sub-index, and k / bs is linear in i.  The staged cloud is stored
// in RANK order -- position (reversed slot) * ceil(n / bs) + k / bs -- with the point's index in .w, so the winner's
// coordinates and index are one multiply-add and one LDS.128 away from the reduced rank.
template <int T, int P, int S>
__global__ void __launch_bounds__(T) fps_reg_kernel(const float *__restrict__ data, int n, int c, int m, int lg_bs,
                                                    int *__restrict__ idx, float *__restrict__ centers) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int npb = (n + (1 << lg_bs) - 1) >> lg_bs;               // points per reference slot (k / bs < npb)
  float4 *sp = reinterpret_cast<float4 *>(smem_raw);            // [bs * npb] staged cloud in rank order
  unsigned long long *slots = reinterpret_cast<unsigned long long *>(sp + (static_cast<size_t>(npb) << lg_bs));  // [2][32]
  const int tid = threadIdx.x;
  const float *__restrict__ cloud = data + static_cast<size_t>(blockIdx.x) * n * c;
  int *__restrict__ out = idx + static_cast<size_t>(blockIdx.x) * m;

  static_assert(P % (1 << S) == 0, "points per thread must cover whole slot groups");
  constexpr int PG = P >> S;  // points per slot sub-index
  constexpr int LOG2T = T == 128 ? 7 : T == 256 ? 8 : T == 512 ? 9 : 10;
  // rank of register i = rank_base + rank_of_reg(i):
  //   S == 0 (T >= bs): reversed slot = brev(tid mod bs), k / bs = (tid >> lg_bs) + i * (T >> lg_bs)
  //   S  > 0 (T <  bs): reversed slot = brev_T(tid) << S | sub(i), k / bs = i mod PG           (sub = i / PG)
  unsigned rank_base;
  if (S == 0) {
    const unsigned slot = static_cast<unsigned>(tid) & ((1u << lg_bs) - 1u);
    const unsigned rev = lg_bs ? (__brev(slot) >> (32 - lg_bs)) : 0u;
    rank_base = (rev << 22) | (static_cast<unsigned>(tid) >> lg_bs);
  } else {
    rank_base = (__brev(static_cast<unsigned>(tid)) >> (32 - LOG2T)) << (22 + S);
  }
  const unsigned hi_step = S == 0 ? static_cast<unsigned>(T >> lg_bs) : 1u;
  auto rank_of_reg = [&](int i) -> unsigned {
    if (S == 0) return rank_base + static_cast<unsigned>(i) * hi_step;
    return rank_base + (static_cast<unsigned>(i / PG) << 22) + static_cast<unsigned>(i % PG);
  };
  auto pos_of_rank = [&](unsigned r) -> unsigned { return (r >> 22) * static_cast<unsigned>(npb) + (r & 0x3fffffu); };

  float px[P], py[P], pz[P], pt[P];
#pragma unroll
  for (int p = 0; p < P; ++p) {
    const int k = tid + fps_point_of_reg<S, PG>(p) * T;
    float x = 0.f, y = 0.f, z = 0.f, t = -2.0f;
    if (k < n) {
      x = __ldg(cloud + static_cast<size_t>(k) * c);
      y = __ldg(cloud + static_cast<size_t>(k) * c + 1);
      z = __ldg(cloud + static_cast<size_t>(k) * c + 2);
      const float mag = dist_yxz(x, y, z);
      t = (static_cast<double>(mag) <= 1e-3) ? -2.0f : 1e10f;  // sampling_gpu.cu:103-104
      sp[pos_of_rank(rank_of_reg(p))] = make_float4(x, y, z, __int_as_float(k));
    }
    px[p] = x; py[p] = y; pz[p] = z; pt[p] = t;
  }
  if (tid == 0) out[0] = 0;
  __syncthreads();

  float4 o = sp[0];  // point 0 has rank 0
  for (int j = 1; j < m; ++j) {
    float v[P];
    int vi[P];
    fps_update<P, (T >= 512)>(px, py, pz, pt, o.x, o.y, o.z);
#pragma unroll
    for (int p = 0; p < P; ++p) {
      v[p] = pt[p];
      vi[p] = p;
    }
    // first-maximum tournament (strict `>` keeps the lower p on ties, like the reference's serial scan)
#pragma unroll
    for (int stride = 1; stride < P; stride *= 2) {
#pragma unroll
      for (int i = 0; i + stride < P; i += 2 * stride) {
        const bool take = v[i + stride] > v[i];
        v[i] = take ? v[i + stride] : v[i];
        vi[i] = take ? vi[i + stride] : vi[i];
      }
    }
    const bool any = v[0] > -1.0f;
    const float best = any ? v[0] : -1.0f;
    // a thread with no valid point reports (value -1, index 0) like the reference (:93-94); point 0 has rank 0
    const unsigned myrank = any ? rank_of_reg(vi[0]) : 0u;
    const unsigned r = fps_block_argmax_keys<T>(fps_val_bits(best), myrank, slots, j);
    o = sp[pos_of_rank(r)];
    if (tid == 0) out[j] = __float_as_int(o.w);
  }

  if (centers != nullptr) {  // fused utils/misc.py:18-19 gather of the sampled rows
    __syncthreads();
    float *__restrict__ cen = centers + static_cast<size_t>(blockIdx.x) * m * c;
    for (int e = tid; e < m * c; e += T) {
      const int j = e / c, ch = e - j * c;
      cen[e] = __ldg(cloud + static_cast<size_t>(out[j]) * c + ch);
    }
  }
}

// ---- scene-scale clouds (12 288 < n <= CS*512*P): one thread-block CLUSTER per cloud --------------------------------
// The cloud is split over the CS CTAs of a cluster (contiguous 512*P-point slices, all state still in registers +
// the CTA's own shared memory).  Per iteration every CTA finds its local arg-max as above, its warp 0 posts
// (value bits, rank, x, y, z) into the slot table of EVERY CTA of the cluster through distributed shared memory,
// one cluster barrier makes the posts visible, and every warp picks the global winner from its CTA's local table.
// Slot tables are double-buffered, so there is exactly one cluster barrier and one CTA barrier per iteration.
struct FpsSlot {
  unsigned vb, rank;
  float x, y, z;
  unsigned pad[3];
};

template <int P, int CS>
__global__ void __launch_bounds__(512) fps_cluster_kernel(const float *__restrict__ data, int n, int c, int m, int lg_bs,
                                                          int *__restrict__ idx, float *__restrict__ centers) {
  constexpr int T = 512;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float4 *sp = reinterpret_cast<float4 *>(smem_raw);                         // [T*P] this CTA's slice
  FpsSlot *table = reinterpret_cast<FpsSlot *>(sp + T * P);                  // [2][CS]
  uint2 *slots = reinterpret_cast<uint2 *>(table + 2 * CS);                  // [2][32] intra-CTA reduction
  cg::cluster_group cluster = cg::this_cluster();
  const int crank = static_cast<int>(cluster.block_rank());
  const int cloud_id = blockIdx.x / CS;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int base = crank * T * P;  // multiple of 512: k mod bs == tid for every point of a thread
  const float *__restrict__ cloud = data + static_cast<size_t>(cloud_id) * n * c;
  int *__restrict__ out = idx + static_cast<size_t>(cloud_id) * m;

  float px[P], py[P], pz[P], pt[P];
#pragma unroll
  for (int p = 0; p < P; ++p) {
    const int k = base + tid + p * T;
    float x = 0.f, y = 0.f, z = 0.f, t = -2.0f;
    if (k < n) {
      x = __ldg(cloud + static_cast<size_t>(k) * c);
      y = __ldg(cloud + static_cast<size_t>(k) * c + 1);
      z = __ldg(cloud + static_cast<size_t>(k) * c + 2);
      t = (static_cast<double>(dist_yxz(x, y, z)) <= 1e-3) ? -2.0f : 1e10f;
    }
    sp[tid + p * T] = make_float4(x, y, z, 0.f);
    px[p] = x; py[p] = y; pz[p] = z; pt[p] = t;
  }
  if (crank == 0 && tid == 0) out[0] = 0;
  float ox = __ldg(cloud), oy = __ldg(cloud + 1), oz = __ldg(cloud + 2);  // point 0
  __syncthreads();
  cluster.sync();

  for (int j = 1; j < m; ++j) {
    float v[P];
    int vi[P];
    fps_update<P, true>(px, py, pz, pt, ox, oy, oz);
#pragma unroll
    for (int p = 0; p < P; ++p) {
      v[p] = pt[p];
      vi[p] = p;
    }
#pragma unroll
    for (int stride = 1; stride < P; stride *= 2) {
#pragma unroll
      for (int i = 0; i + stride < P; i += 2 * stride) {
        const bool take = v[i + stride] > v[i];
        v[i] = take ? v[i + stride] : v[i];
        vi[i] = take ? vi[i + stride] : vi[i];
      }
    }
    const bool any = v[0] > -1.0f;
    const float best = any ? v[0] : -1.0f;
    const int bk = any ? base + tid + vi[0] * T : 0;
    const unsigned vb = fps_val_bits(best);
    const unsigned r = fps_block_argmax<T>(vb, fps_rank(bk, lg_bs), slots, j);
    // CTA-level value of the winner: recompute from the table of warp maxima (all warps hold the same r)
    const unsigned full = 0xffffffffu;
    const uint2 wv = lane < T / 32 ? slots[(j & 1) * 32 + lane] : make_uint2(0u, 0xffffffffu);
    const unsigned cta_vb = __reduce_max_sync(full, wv.x);
    FpsSlot *tab = table + (j & 1) * CS;
    if (warp == 0) {
      // local winner's coordinates (only meaningful when it is a real point of this CTA's slice)
      const int kl = fps_unrank(r, lg_bs) - base;
      const bool mine = cta_vb != 0u && kl >= 0 && kl < T * P;
      const float4 w = sp[mine ? kl : 0];
      if (lane < CS) {
        FpsSlot *remote = cluster.map_shared_rank(tab, lane) + crank;
        remote->vb = cta_vb;
        remote->rank = cta_vb != 0u ? r : 0u;  // "no valid point" posts (value -1, index 0) like the reference
        remote->x = w.x; remote->y = w.y; remote->z = w.z;
      }
    }
    cluster.sync();
    const FpsSlot sl = tab[lane < CS ? lane : 0];
    const unsigned gvb = __reduce_max_sync(full, lane < CS ? sl.vb : 0u);
    const unsigned gr = __reduce_min_sync(full, (lane < CS && sl.vb == gvb) ? sl.rank : 0xffffffffu);
    const unsigned who = __ballot_sync(full, lane < CS && sl.vb == gvb && sl.rank == gr);
    const int src = __ffs(who) - 1;
    const int old = gvb != 0u ? fps_unrank(gr, lg_bs) : 0;
    if (gvb != 0u) {
      ox = __shfl_sync(full, sl.x, src); oy = __shfl_sync(full, sl.y, src); oz = __shfl_sync(full, sl.z, src);
    } else {
      ox = __ldg(cloud); oy = __ldg(cloud + 1); oz = __ldg(cloud + 2);  // every point skipped: the reference re-selects index 0
    }
    if (crank == 0 && tid == 0) out[j] = old;
  }
  cluster.sync();  // no CTA may exit while peers can still write into its shared memory
  if (centers != nullptr && crank == 0) {
    __syncthreads();
    float *__restrict__ cen = centers + static_cast<size_t>(cloud_id) * m * c;
    for (int e = tid; e < m * c; e += T) {
      const int jj = e / c, ch = e - jj * c;
      cen[e] = cloud[static_cast<size_t>(out[jj]) * c + ch];
    }
  }
}

template <int P, int CS>
static int launch_fps_cluster(const float *data, int b, int n, int c, int m, int lg_bs, int *idx, float *centers,
                              cudaStream_t st) {
  const size_t smem = static_cast<size_t>(512) * P * sizeof(float4) + 2 * CS * sizeof(FpsSlot) + 2 * 32 * sizeof(uint2);
  auto kern = fps_cluster_kernel<P, CS>;
  PDAE_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
  if (CS > 8) PDAE_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(static_cast<unsigned>(b) * CS, 1, 1);
  cfg.blockDim = dim3(512, 1, 1);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CS;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  PDAE_CUDA_TRY(cudaLaunchKernelEx(&cfg, kern, data, n, c, m, lg_bs, idx, centers));
  return 0;
}

// ---- large-cloud fallback: running minima in a global workspace -------------------------------
template <int T>
__global__ void __launch_bounds__(T) fps_global_kernel(const float *__restrict__ data, int n, int c, int m, int lg_bs,
                                                       int *__restrict__ idx, float *__restrict__ centers,
                                                       float *__restrict__ temp_ws) {
  __shared__ uint2 slots[2 * 32];
  const int tid = threadIdx.x;
  const float *__restrict__ cloud = data + static_cast<size_t>(blockIdx.x) * n * c;
  float *__restrict__ temp = temp_ws + static_cast<size_t>(blockIdx.x) * n;
  int *__restrict__ out = idx + static_cast<size_t>(blockIdx.x) * m;
  for (int k = tid; k < n; k += T) {
    const float x = cloud[static_cast<size_t>(k) * c], y = cloud[static_cast<size_t>(k) * c + 1],
                z = cloud[static_cast<size_t>(k) * c + 2];
    temp[k] = (static_cast<double>(dist_yxz(x, y, z)) <= 1e-3) ? -2.0f : 1e10f;
  }
  if (tid == 0) out[0] = 0;
  __syncthreads();
  int old = 0;
  for (int j = 1; j < m; ++j) {
    const float ox = cloud[static_cast<size_t>(old) * c], oy = cloud[static_cast<size_t>(old) * c + 1],
                oz = cloud[static_cast<size_t>(old) * c + 2];
    float best = -1.0f;
    int bk = 0;
    // T is a multiple of bs, so a thread's points share one slot and ascending k is rank order
    for (int k = tid; k < n; k += T) {
      const float x = cloud[static_cast<size_t>(k) * c], y = cloud[static_cast<size_t>(k) * c + 1],
                  z = cloud[static_cast<size_t>(k) * c + 2];
      const float d = dist_yxz(__fsub_rn(x, ox), __fsub_rn(y, oy), __fsub_rn(z, oz));
      const float d2 = fminf(d, temp[k]);
      temp[k] = d2;
      const bool take = d2 > best;
      bk = take ? k : bk;
      best = take ? d2 : best;
    }
    if (best < 0.0f) bk = 0;
    const unsigned r = fps_block_argmax<T>(fps_val_bits(best), fps_rank(bk, lg_bs), slots, j);
    old = fps_unrank(r, lg_bs);
    if (tid == 0) out[j] = old;
  }
  if (centers != nullptr) {
    __syncthreads();
    float *__restrict__ cen = centers + static_cast<size_t>(blockIdx.x) * m * c;
    for (int e = tid; e < m * c; e += T) {
      const int j = e / c, ch = e - j * c;
      cen[e] = cloud[static_cast<size_t>(out[j]) * c + ch];
    }
  }
}

// ---- gather ------------------------------------------------------------------------------------
// reference: sampling_gpu.cu:11-23.  One thread per output element, idx read once per (b, j).
__global__ void __launch_bounds__(256) gather_kernel(const float *__restrict__ feat, const int *__restrict__ idx, int c,
                                                     int n, int m, long long total, float *__restrict__ out) {
  const long long e = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (e >= total) return;
  const int j = static_cast<int>(e % m);
  const long long bc = e / m;  // b*c + l
  const long long bi = bc / c;
  out[e] = __ldg(feat + bc * n + __ldg(idx + bi * m + j));
}

// reference: sampling_gpu.cu:37-50 (atomicAdd scatter into zeros).
__global__ void __launch_bounds__(256) gather_grad_kernel(const float *__restrict__ gout, const int *__restrict__ idx,
                                                          int c, int n, int m, long long total,
                                                          float *__restrict__ gfeat) {
  const long long e = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (e >= total) return;
  const int j = static_cast<int>(e % m);
  const long long bc = e / m;
  const long long bi = bc / c;
  atomicAdd(gfeat + bc * n + __ldg(idx + bi * m + j), __ldg(gout + e));
}

static int ilog2_floor(int v) {
  int l = 0;
  while ((1 << (l + 1)) <= v) ++l;
  return l;
}

template <int T, int P, int S = 0>
static int launch_fps_reg(const float *data, int b, int n, int c, int m, int lg_bs, int *idx, float *centers,
                          cudaStream_t st) {
  const size_t table = static_cast<size_t>((n + (1 << lg_bs) - 1) >> lg_bs) << lg_bs;  // rank-ordered positions, >= n
  const size_t smem = table * sizeof(float4) + 2 * 32 * sizeof(unsigned long long);
  if (smem > 48 * 1024) {
    PDAE_CUDA_TRY(cudaFuncSetAttribute(fps_reg_kernel<T, P, S>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       static_cast<int>(smem)));
  }
  fps_reg_kernel<T, P, S><<<b, T, smem, st>>>(data, n, c, m, lg_bs, idx, centers);
  PDAE_RETURN_IF_LAUNCH_FAILED();
  return 0;
}

constexpr int FPS_REG_MAX_N = 12288;
constexpr int FPS_T4096 = 512, FPS_P4096 = 8, FPS_S4096 = 0;  // 2049..4096 points: 51.5 us (4096 -> 128) vs 60.8 / 64.5 us for 256 x 16 / 128 x 32
constexpr int FPS_CLUSTER_MAX_N = 16 * 512 * 24;  // 196 608

static int fps_dispatch(const float *data, int b, int n, int c, int m, int *idx, float *centers, void *ws,
                        size_t ws_bytes, cudaStream_t st) {
  if (b < 0 || n < 0 || m < 0 || c < 3) return PDAE_E_INVALID;
  if (b == 0 || m == 0) return 0;
  if (!idx) return PDAE_E_INVALID;
  if (n == 0) {  // reference kernel would read out of bounds; define as all-zero indices
    PDAE_CUDA_TRY(cudaMemsetAsync(idx, 0, static_cast<size_t>(b) * m * sizeof(int), st));
    return 0;
  }
  if (!data) return PDAE_E_INVALID;
  const int bs = pdae_fps_block_size(n);
  const int lg_bs = ilog2_floor(bs);
  // thread count must be a multiple of bs so that ascending k inside a thread is rank order
  // (bs <= 512 and bs <= n, so every configuration below satisfies T % bs == 0 or is rejected).
#define PDAE_FPS_TRY(T, P)                                                                   \
  if (want_t == (T) && want_p == (P) && n <= (T) * (P)) {                                     \
    if ((T) % bs == 0) return launch_fps_reg<T, P, 0>(data, b, n, c, m, lg_bs, idx, centers, st); \
    if constexpr ((T) == 256 && (P) % 2 == 0) {                                               \
      if (bs == 512) return launch_fps_reg<T, P, 1>(data, b, n, c, m, lg_bs, idx, centers, st); \
    }                                                                                         \
    if constexpr ((T) == 128 && (P) % 4 == 0) {                                               \
      if (bs == 512) return launch_fps_reg<T, P, 2>(data, b, n, c, m, lg_bs, idx, centers, st); \
    }                                                                                         \
    if constexpr ((T) == 128 && (P) % 2 == 0) {                                               \
      if (bs == 256) return launch_fps_reg<T, P, 1>(data, b, n, c, m, lg_bs, idx, centers, st); \
    }                                                                                         \
  }
  int want_t = 0, want_p = 0;
  if (const char *e = getenv("PDAE_FPS_CFG")) {  // tuning hook: "T,P"
    if (sscanf(e, "%d,%d", &want_t, &want_p) == 2) {
      PDAE_FPS_TRY(128, 8) PDAE_FPS_TRY(128, 16) PDAE_FPS_TRY(128, 32) PDAE_FPS_TRY(256, 4) PDAE_FPS_TRY(256, 8)
      PDAE_FPS_TRY(256, 16) PDAE_FPS_TRY(256, 32) PDAE_FPS_TRY(512, 2) PDAE_FPS_TRY(512, 4) PDAE_FPS_TRY(512, 8)
      PDAE_FPS_TRY(512, 16) PDAE_FPS_TRY(1024, 4) PDAE_FPS_TRY(1024, 8)
    }
  }
#undef PDAE_FPS_TRY
  // defaults from profiles/tune_kernels.py on B200: one warp per scheduler (128 threads) gives the shortest iteration
  // once the block reduction is a 4-key register tree (2048 -> 64: 16.7 us against 23.0 us with 256 threads)
  if (n <= 128) return launch_fps_reg<128, 1>(data, b, n, c, m, lg_bs, idx, centers, st);
  if (n < 256) return launch_fps_reg<128, 2>(data, b, n, c, m, lg_bs, idx, centers, st);       // bs == 128
  if (n < 512) return launch_fps_reg<128, 4, 1>(data, b, n, c, m, lg_bs, idx, centers, st);    // bs == 256
  // from here on bs == 512: the narrower CTAs use the rank-ordered register layout (S = log2(512 / T))
  if (n <= 1024) return launch_fps_reg<128, 8, 2>(data, b, n, c, m, lg_bs, idx, centers, st);
  if (n <= 2048) return launch_fps_reg<128, 16, 2>(data, b, n, c, m, lg_bs, idx, centers, st);
  if (n <= 4096) return launch_fps_reg<FPS_T4096, FPS_P4096, FPS_S4096>(data, b, n, c, m, lg_bs, idx, centers, st);
  if (n <= 8192) return launch_fps_reg<512, 16>(data, b, n, c, m, lg_bs, idx, centers, st);  // 366 us vs 392 us for 256 x 32 (8192 -> 512)
  if (n <= FPS_REG_MAX_N) return launch_fps_reg<512, 24>(data, b, n, c, m, lg_bs, idx, centers, st);
  // scene-scale clouds: a 16-CTA cluster per cloud (state in registers + DSMEM exchange), up to 196 608 points
  if (n <= 16 * 512 * 8) return launch_fps_cluster<8, 16>(data, b, n, c, m, lg_bs, idx, centers, st);
  if (n <= 16 * 512 * 13) return launch_fps_cluster<13, 16>(data, b, n, c, m, lg_bs, idx, centers, st);
  if (n <= FPS_CLUSTER_MAX_N) return launch_fps_cluster<24, 16>(data, b, n, c, m, lg_bs, idx, centers, st);
  const size_t need = static_cast<size_t>(b) * n * sizeof(float);
  if (!ws || ws_bytes < need) return PDAE_E_WORKSPACE;
  fps_global_kernel<1024><<<b, 1024, 0, st>>>(data, n, c, m, lg_bs, idx, centers, static_cast<float *>(ws));
  PDAE_RETURN_IF_LAUNCH_FAILED();
  return 0;
}

}  // namespace pdae

using namespace pdae;

// reference: cuda_utils.h:15-21.  Evaluated with the same double log() expression so the tie
// rule can never disagree with the reference about the block size.
extern "C" int pdae_fps_block_size(int n) {
  if (n <= 0) return 1;
  const int pow_2 = static_cast<int>(log(static_cast<double>(n)) / log(2.0));
  int t = 1 << pow_2;
  if (t > 512) t = 512;
  if (t < 1) t = 1;
  return t;
}

extern "C" size_t pdae_fps_workspace_bytes(int b, int n, int m) {
  (void)m;
  if (b <= 0 || n <= FPS_CLUSTER_MAX_N) return 0;
  return static_cast<size_t>(b) * n * sizeof(float);
}

extern "C" int pdae_fps_f32(const float *xyz, int b, int n, int m, int *idx, void *workspace, size_t workspace_bytes,
                            pdae_stream_t stream) {
  return fps_dispatch(xyz, b, n, 3, m, idx, nullptr, workspace, workspace_bytes, static_cast<cudaStream_t>(stream));
}

extern "C" int pdae_fps_gather_f32(const float *data, int b, int n, int c, int m, int *idx, float *centers,
                                   void *workspace, size_t workspace_bytes, pdae_stream_t stream) {
  if (b > 0 && m > 0 && !centers) return PDAE_E_INVALID;
  if (n == 0 && b > 0 && m > 0) return PDAE_E_INVALID;
  return fps_dispatch(data, b, n, c, m, idx, centers, workspace, workspace_bytes, static_cast<cudaStream_t>(stream));
}

extern "C" int pdae_gather_f32(const float *feat, const int *idx, int b, int c, int n, int m, float *out,
                               pdae_stream_t stream) {
  if (b < 0 || c < 0 || n < 0 || m < 0) return PDAE_E_INVALID;
  const long long total = static_cast<long long>(b) * c * m;
  if (total == 0) return 0;
  if (!feat || !idx || !out || n == 0) return PDAE_E_INVALID;
  const long long grid = (total + 255) / 256;
  if (grid > 0x7fffffffLL) return PDAE_E_UNSUPPORTED;
  gather_kernel<<<static_cast<unsigned>(grid), 256, 0, static_cast<cudaStream_t>(stream)>>>(feat, idx, c, n, m, total,
                                                                                           out);
  PDAE_RETURN_IF_LAUNCH_FAILED();
  return 0;
}

extern "C" int pdae_gather_grad_f32(const float *gout, const int *idx, int b, int c, int n, int m, float *gfeat,
                                    pdae_stream_t stream) {
  if (b < 0 || c < 0 || n < 0 || m < 0) return PDAE_E_INVALID;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const size_t gsz = static_cast<size_t>(b) * c * n;
  if (gsz) {
    if (!gfeat) return PDAE_E_INVALID;
    PDAE_CUDA_TRY(cudaMemsetAsync(gfeat, 0, gsz * sizeof(float), st));
  }
  const long long total = static_cast<long long>(b) * c * m;
  if (total == 0 || gsz == 0) return 0;
  if (!gout || !idx) return PDAE_E_INVALID;
  const long long grid = (total + 255) / 256;
  if (grid > 0x7fffffffLL) return PDAE_E_UNSUPPORTED;
  gather_grad_kernel<<<static_cast<unsigned>(grid), 256, 0, st>>>(gout, idx, c, n, m, total, gfeat);
  PDAE_RETURN_IF_LAUNCH_FAILED();
  return 0;
}

// deterministic form: gfeat[b][l][p] = +0 (+) gout[b][l][j] for every j with idx[b][j] == p, j ascending (reverse.cuh)
extern "C" size_t pdae_gather_grad_det_workspace_bytes(int b, int n, int m) {
  if (b <= 0 || n < 0 || m < 0) return 0;
  return rev_map_bytes(b, m, n);
}

extern "C" int pdae_gather_grad_det_f32(const float *gout, const int *idx, int b, int c, int n, int m, float *gfeat,
                                        void *workspace, size_t workspace_bytes, pdae_stream_t stream) {
  if (b < 0 || c < 0 || n < 0 || m < 0) return PDAE_E_INVALID;
  const size_t gsz = static_cast<size_t>(b) * c * n;
  if (gsz == 0) return 0;
  if (!gfeat || (m && (!gout || !idx))) return PDAE_E_INVALID;
  if (!workspace || workspace_bytes < pdae_gather_grad_det_workspace_bytes(b, n, m)) return PDAE_E_WORKSPACE;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  RevMap map;
  const int rc = rev_map_build(idx, b, m, n, workspace, &map, st);
  if (rc) return rc;
  return rev_gather_channel_major(gout, nullptr, b, c, m, n, 1, map, gfeat, st);
}
