// knn.cu -- brute-force k nearest neighbours (knn_cuda.KNN), the fused Group tail
// (kNN + gather + centre-subtract) and the low-dimensional DGCNN kNN.
//
// Semantics: KNN_CUDA 0.2 (un-vendored dependency of the reference; algorithm restated in
// oracle/pdae_oracle.c): squared distance accumulated as sequential fma over the dims in order,
// the k smallest kept in ascending order with strict `<` insertion, i.e. ascending by
// (distance, index); Euclidean (sqrt) distances and 0-based int64 indices are returned.
// Call sites: models/PointCAE_transformer.py:59,76 (transpose_mode=True, k=32, dim 3),
// models/MaskSurf_v2.py:79,124 (transpose_mode=False).  DGCNN kNN: models/dgcnn_util.py:7-12.
//
// Design: the reference launches ~12 kernels per cloud from a Python loop; here the whole batch
// is one launch.  A CTA stages a tile of the reference cloud in shared memory as planes and each
// warp owns one query at a time: every lane evaluates one reference point per step, candidates
// below the running k-th key are appended to a per-warp queue with a ballot, and a full queue
// (32 entries) is bitonic-sorted and merged into the warp-resident sorted list (one key per lane
// per 32 of k).  Keys are (float bits << 32 | index), so the unsigned order *is* the
// (distance, lower index first) order and the selection is exact and deterministic.
#include "knn_select.cuh"

#include <cstdlib>

namespace pdae {

struct KnnArgs {
  const float *ref;    // PLANAR ? (b, dim, r) : (b, r, dim)
  const float *query;  // PLANAR ? unused (queries are the reference points) : (b, q, dim)
  float *dist;         // optional, Euclidean
  int64_t *idx;        // optional
  float *group;        // optional (b, q, k, 3): ref[idx] - query   (dim == 3, !PLANAR)
  uint64_t *keys;      // optional (b, q, k): raw (squared-distance bits << 32 | ref_offset + index) for sharded merges
  uint32_t ref_offset; // global index of ref[0] (keys output only)
  int raw_group;       // 1: `group` receives ref[idx] itself instead of ref[idx] - query
  int r, q, dim, k;
  int tile;            // reference points per shared-memory tile (multiple of 32)
  int qpw;             // queries per warp (1 when the cloud spans several tiles)
  int out_kq;          // 1: outputs laid out (b, k, q)
};

template <int D /*0 = runtime*/, bool PLANAR, int NS>
__global__ void __launch_bounds__(KNN_THREADS) knn_kernel(const KnnArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  uint64_t *queue_all = reinterpret_cast<uint64_t *>(smem_raw);              // [KNN_WARPS][64]
  float *planes = reinterpret_cast<float *>(queue_all + KNN_WARPS * 64);     // [dim][tile]
  const int dim = D ? D : a.dim;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int cloud = blockIdx.y;
  const int r = a.r, q = a.q, k = a.k, tile = a.tile;
  const float *__restrict__ R = a.ref + static_cast<size_t>(cloud) * r * dim;
  const float *__restrict__ Qp = PLANAR ? R : a.query + static_cast<size_t>(cloud) * q * dim;
  uint64_t *queue = queue_all + warp * 64;
  const int ntiles = (r + tile - 1) / tile;
  const int kslot = (k - 1) >> 5, klane = (k - 1) & 31;

  for (int qi = 0; qi < a.qpw; ++qi) {
    const int qidx = (blockIdx.x * KNN_WARPS + warp) * a.qpw + qi;
    const bool qvalid = qidx < q;
    float q0 = 0.f, q1 = 0.f, q2 = 0.f;
    if (D == 3 && qvalid) {
      if (PLANAR) {
        q0 = __ldg(Qp + qidx); q1 = __ldg(Qp + r + qidx); q2 = __ldg(Qp + 2 * r + qidx);
      } else {
        q0 = __ldg(Qp + 3 * qidx); q1 = __ldg(Qp + 3 * qidx + 1); q2 = __ldg(Qp + 3 * qidx + 2);
      }
    }
    WarpSelect<NS> sel;
    sel.init();

    for (int tl = 0; tl < ntiles; ++tl) {
      const int tbase = tl * tile;
      const int tn = (r - tbase) < tile ? (r - tbase) : tile;
      if (ntiles > 1 || qi == 0) {
        __syncthreads();  // previous tile fully consumed
        if (PLANAR) {
          for (int c = 0; c < dim; ++c)
            for (int p = tid; p < tn; p += KNN_THREADS) planes[c * tile + p] = __ldg(R + static_cast<size_t>(c) * r + tbase + p);
        } else {
          const float *src = R + static_cast<size_t>(tbase) * dim;
          for (int f = tid; f < tn * dim; f += KNN_THREADS) {
            const int p = f / dim, c = f - p * dim;
            planes[c * tile + p] = __ldg(src + f);
          }
        }
        __syncthreads();
      }
      if (!qvalid) continue;
      for (int j0 = 0; j0 < tn; j0 += 32) {
        const int j = j0 + lane;
        const bool in = j < tn;
        float d = 0.f;
        if (in) {
          if (D == 3) {
            d = dist_seq3(__fsub_rn(planes[j], q0), __fsub_rn(planes[tile + j], q1), __fsub_rn(planes[2 * tile + j], q2));
          } else {
            for (int c = 0; c < dim; ++c) {
              const float qc = PLANAR ? __ldg(Qp + static_cast<size_t>(c) * r + qidx) : __ldg(Qp + static_cast<size_t>(qidx) * dim + c);
              const float t = __fsub_rn(planes[c * tile + j], qc);
              d = __fmaf_rn(t, t, d);
            }
          }
        }
        const uint64_t key = pack_key(d, static_cast<uint32_t>(tbase + j));
        sel.offer(in && key < sel.tau, key, queue, lane, kslot, klane);
      }
    }
    if (!qvalid) continue;
    sel.finish(queue, lane);
    // ---- epilogue: ascending list -> outputs -------------------------------------------------
    const size_t bq = static_cast<size_t>(cloud) * q + qidx;
#pragma unroll
    for (int s = 0; s < NS; ++s) {
      const int p = s * 32 + lane;
      if (p < k) {
        const uint64_t key = sel.L[s];
        const uint32_t ji = static_cast<uint32_t>(key);
        const size_t o = a.out_kq ? (static_cast<size_t>(cloud) * k + p) * q + qidx : bq * k + p;
        if (a.idx) a.idx[o] = static_cast<int64_t>(ji);
        if (a.dist) a.dist[o] = __fsqrt_rn(__uint_as_float(static_cast<uint32_t>(key >> 32)));
        if (a.keys) a.keys[bq * k + p] = key == KEY_INF ? KEY_INF : key + a.ref_offset;
        if (D == 3 && !PLANAR && a.group) {
          const bool raw = a.raw_group != 0;
          float *g = a.group + (bq * k + p) * 3;
          const float x = __ldg(R + 3 * static_cast<size_t>(ji)), y = __ldg(R + 3 * static_cast<size_t>(ji) + 1);
          const float z = __ldg(R + 3 * static_cast<size_t>(ji) + 2);
          g[0] = raw ? x : __fsub_rn(x, q0);
          g[1] = raw ? y : __fsub_rn(y, q1);
          g[2] = raw ? z : __fsub_rn(z, q2);
        }
      }
    }
  }
}

template <int D, bool PLANAR>
static int launch_knn(const KnnArgs &a, int b, cudaStream_t st) {
  const int ns = (a.k + 31) / 32;
  const size_t smem = static_cast<size_t>(KNN_WARPS) * 64 * sizeof(uint64_t) + static_cast<size_t>(a.dim) * a.tile * sizeof(float);
  const dim3 grid(ceil_div(a.q, KNN_WARPS * a.qpw), b);
  if (b > 65535) return PDAE_E_UNSUPPORTED;
#define PDAE_KNN_LAUNCH(NS)                                                                              \
  do {                                                                                                   \
    if (smem > 48 * 1024)                                                                                \
      PDAE_CUDA_TRY(cudaFuncSetAttribute(knn_kernel<D, PLANAR, NS>, cudaFuncAttributeMaxDynamicSharedMemorySize, \
                                         static_cast<int>(smem)));                                      \
    knn_kernel<D, PLANAR, NS><<<grid, KNN_THREADS, smem, st>>>(a);                                       \
  } while (0)
  if (ns == 1) PDAE_KNN_LAUNCH(1);
  else if (ns == 2) PDAE_KNN_LAUNCH(2);
  else PDAE_KNN_LAUNCH(4);
#undef PDAE_KNN_LAUNCH
  PDAE_RETURN_IF_LAUNCH_FAILED();
  return 0;
}

static int knn_plan(KnnArgs &a, int b) {
  // tile: whole cloud when it fits in ~96 KB of planes, else 2048-point tiles (dim <= 11) or less
  const int dim = a.dim;
  const int budget_floats = (96 * 1024) / 4;
  int tile_cap = (budget_floats / dim) & ~31;
  if (tile_cap < 32) return PDAE_E_UNSUPPORTED;  // dim > 768
  const int r32 = (a.r + 31) & ~31;
  if (r32 <= tile_cap) {
    a.tile = r32;
    long long per = (static_cast<long long>(b) * a.q) / (148LL * KNN_WARPS * 3);
    a.qpw = per < 1 ? 1 : (per > 8 ? 8 : static_cast<int>(per));
  } else {
    a.tile = tile_cap > 2048 ? 2048 : tile_cap;
    a.qpw = 1;
  }
  return 0;
}

}  // namespace pdae

using namespace pdae;

static int knn_dim3(const float *ref, const float *query, int b, int r, int q, int k, int out_kq, float *dist, int64_t *idx,
                    float *group, cudaStream_t st, uint64_t *keys, uint32_t off, int raw, void *ws, size_t ws_bytes) {
  const int rc = knn4_points(ref, query, b, r, q, k, out_kq, dist, idx, group, st, keys, off, raw, nullptr, ws, ws_bytes);
  if (rc != PDAE_E_UNSUPPORTED) return rc;
  // clouds beyond the 16-bit step numbers of one chunk (> 8 M points without a workspace): streaming warp-select
  KnnArgs a{ref, query, dist, idx, group, keys, off, raw, r, q, 3, k, 0, 1, out_kq};
  const int prc = knn_plan(a, b);
  if (prc) return prc;
  return launch_knn<3, false>(a, b, st);
}

extern "C" size_t pdae_knn_workspace_bytes(int b, int r, int q, int dim, int k) {
  return dim == 3 ? knn4_workspace_bytes(b, r, q, k) : 0;
}

extern "C" int pdae_knn_ws_f32(const float *ref, const float *query, int b, int r, int q, int dim, int k, int out_kq,
                               float *dist, int64_t *idx, void *workspace, size_t workspace_bytes, pdae_stream_t stream) {
  if (b < 0 || r < 0 || q < 0 || dim <= 0 || k <= 0) return PDAE_E_INVALID;
  if (b == 0 || q == 0) return 0;
  if (k > r || k > KNN_MAX_K) return PDAE_E_INVALID;
  if (!ref || !query || (!dist && !idx)) return PDAE_E_INVALID;
  if (dim == 3 && k <= 64)
    return knn_dim3(ref, query, b, r, q, k, out_kq ? 1 : 0, dist, idx, nullptr, static_cast<cudaStream_t>(stream), nullptr, 0u,
                    0, workspace, workspace_bytes);
  return pdae_knn_f32(ref, query, b, r, q, dim, k, out_kq, dist, idx, stream);
}

extern "C" int pdae_knn_f32(const float *ref, const float *query, int b, int r, int q, int dim, int k, int out_kq,
                            float *dist, int64_t *idx, pdae_stream_t stream) {
  if (b < 0 || r < 0 || q < 0 || dim <= 0 || k <= 0) return PDAE_E_INVALID;
  if (b == 0 || q == 0) return 0;
  if (k > r || k > KNN_MAX_K) return PDAE_E_INVALID;
  if (!ref || !query || (!dist && !idx)) return PDAE_E_INVALID;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (dim == 3 && k <= 64) return knn_dim3(ref, query, b, r, q, k, out_kq ? 1 : 0, dist, idx, nullptr, st, nullptr, 0u, 0, nullptr, 0);
  KnnArgs a{ref, query, dist, idx, nullptr, nullptr, 0u, 0, r, q, dim, k, 0, 1, out_kq ? 1 : 0};
  const int rc = knn_plan(a, b);
  if (rc) return rc;
  return dim == 3 ? launch_knn<3, false>(a, b, st) : launch_knn<0, false>(a, b, st);
}

// ---- reference-set sharding (scene-scale clouds, SURVEY.md 8e): per-rank top-k as packed keys + W-way merge ----
// A rank scans all queries against its slice of the reference cloud and emits, per query, its k best candidates
// as ascending (squared-distance bits << 32 | global index) keys; the ranks all-gather the lists (W*Q*k*8 bytes)
// and every rank merges them: the k smallest keys overall are exactly the unsharded result, because the key order
// is the (distance, lower index first) order of the single-GPU kernel.
__global__ void __launch_bounds__(256) knn_merge_keys_kernel(const uint64_t *__restrict__ keys /*(w, nq, k)*/, int w,
                                                             long long nq, int q, int k, int out_kq,
                                                             float *__restrict__ dist, int64_t *__restrict__ idx) {
  const long long t = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;  // (cloud, query)
  if (t >= nq) return;
  int head[16];
#pragma unroll
  for (int s = 0; s < 16; ++s) head[s] = 0;
  const long long cloud = t / q, qi = t - cloud * q;
  for (int p = 0; p < k; ++p) {
    uint64_t best = KEY_INF;
    int who = 0;
#pragma unroll
    for (int s = 0; s < 16; ++s) {
      if (s < w && head[s] < k) {
        const uint64_t c = keys[(static_cast<long long>(s) * nq + t) * k + head[s]];
        if (c < best) best = c, who = s;
      }
    }
#pragma unroll
    for (int s = 0; s < 16; ++s) head[s] += (s == who && best != KEY_INF) ? 1 : 0;
    const long long o = out_kq ? (cloud * k + p) * q + qi : t * k + p;
    if (idx) idx[o] = static_cast<int64_t>(static_cast<uint32_t>(best));
    if (dist) dist[o] = __fsqrt_rn(__uint_as_float(static_cast<uint32_t>(best >> 32)));
  }
}

// k <= 64: a warp per query keeps the running k best in registers (one key per lane and 32 of k) and folds every rank's
// ascending list in with the bitonic warp merge -- the thread-per-query walk above is latency-bound (2048 threads for the
// scene-scale shape)
template <int E>
__global__ void __launch_bounds__(128) knn_merge_keys_warp_kernel(const uint64_t *__restrict__ keys /*(w, nq, k)*/, int w,
                                                                  long long nq, int q, int k, int out_kq,
                                                                  float *__restrict__ dist, int64_t *__restrict__ idx) {
  const int lane = threadIdx.x & 31;
  const long long t = (static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  if (t >= nq) return;
  uint64_t L[E];
#pragma unroll
  for (int e = 0; e < E; ++e) L[e] = KEY_INF;
  for (int s = 0; s < w; ++s) {
    const uint64_t *src = keys + (static_cast<long long>(s) * nq + t) * k;
    for (int p0 = 0; p0 < k; p0 += 32) {
      const uint64_t c = (p0 + lane) < k ? __ldg(src + p0 + lane) : KEY_INF;
      warp_merge<E>(L, c, lane);
    }
  }
  const long long cloud = t / q, qi = t - cloud * q;
#pragma unroll
  for (int e = 0; e < E; ++e) {
    const int p = e * 32 + lane;
    if (p < k) {
      const long long o = out_kq ? (cloud * k + p) * q + qi : t * k + p;
      if (idx) idx[o] = static_cast<int64_t>(static_cast<uint32_t>(L[e]));
      if (dist) dist[o] = __fsqrt_rn(__uint_as_float(static_cast<uint32_t>(L[e] >> 32)));
    }
  }
}

extern "C" int pdae_knn_keys_u64(const float *ref_local, const float *query, int b, int r_local, int q, int dim, int k,
                                 long long ref_offset, uint64_t *keys, pdae_stream_t stream) {
  if (b < 0 || r_local < 0 || q < 0 || dim <= 0 || k <= 0 || ref_offset < 0 || ref_offset + r_local > 0xffffffffLL)
    return PDAE_E_INVALID;
  if (b == 0 || q == 0) return 0;
  if (k > KNN_MAX_K || !query || !keys || (r_local && !ref_local)) return PDAE_E_INVALID;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const uint32_t off = static_cast<uint32_t>(ref_offset);
  if (r_local == 0) {  // empty slice: every candidate is +inf
    PDAE_CUDA_TRY(cudaMemsetAsync(keys, 0xff, static_cast<size_t>(b) * q * k * sizeof(uint64_t), st));
    return 0;
  }
  if (dim == 3 && k <= 64) return knn_dim3(ref_local, query, b, r_local, q, k, 0, nullptr, nullptr, nullptr, st, keys, off, 0, nullptr, 0);
  KnnArgs a{ref_local, query, nullptr, nullptr, nullptr, keys, off, 0, r_local, q, dim, k, 0, 1, 0};
  const int rc = knn_plan(a, b);
  if (rc) return rc;
  return dim == 3 ? launch_knn<3, false>(a, b, st) : launch_knn<0, false>(a, b, st);
}

extern "C" int pdae_knn_merge_keys_u64(const uint64_t *keys_all, int w, int b, int q, int k, int out_kq, float *dist,
                                       int64_t *idx, pdae_stream_t stream) {
  if (w <= 0 || w > 16 || b < 0 || q < 0 || k <= 0) return PDAE_E_INVALID;
  const long long nq = static_cast<long long>(b) * q;
  if (nq == 0) return 0;
  if (!keys_all || (!dist && !idx)) return PDAE_E_INVALID;
  if (k <= 64) {
    const long long wgrid = (nq + 3) / 4;
    if (wgrid > 0x7fffffffLL) return PDAE_E_UNSUPPORTED;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (k <= 32) knn_merge_keys_warp_kernel<1><<<static_cast<unsigned>(wgrid), 128, 0, st>>>(keys_all, w, nq, q, k, out_kq ? 1 : 0, dist, idx);
    else knn_merge_keys_warp_kernel<2><<<static_cast<unsigned>(wgrid), 128, 0, st>>>(keys_all, w, nq, q, k, out_kq ? 1 : 0, dist, idx);
    PDAE_RETURN_IF_LAUNCH_FAILED();
    return 0;
  }
  const long long grid = (nq + 255) / 256;
  if (grid > 0x7fffffffLL) return PDAE_E_UNSUPPORTED;
  knn_merge_keys_kernel<<<static_cast<unsigned>(grid), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      keys_all, w, nq, q, k, out_kq ? 1 : 0, dist, idx);
  PDAE_RETURN_IF_LAUNCH_FAILED();
  return 0;
}

static int group_impl(const float *xyz, const float *center, int b, int n, int g, int m, int64_t *idx, float *neighborhood,
                      bool raw, cudaStream_t st, void *ws = nullptr, size_t ws_bytes = 0) {
  if (b < 0 || n < 0 || g < 0 || m <= 0) return PDAE_E_INVALID;
  if (b == 0 || g == 0) return 0;
  if (m > n || m > KNN_MAX_K) return PDAE_E_INVALID;
  if (!xyz || !center || !neighborhood) return PDAE_E_INVALID;
  if (m <= 64) return knn_dim3(xyz, center, b, n, g, m, 0, nullptr, idx, neighborhood, st, nullptr, 0u, raw ? 1 : 0, ws, ws_bytes);
  KnnArgs a{xyz, center, nullptr, idx, neighborhood, nullptr, 0u, raw ? 1 : 0, n, g, 3, m, 0, 1, 0};
  const int rc = knn_plan(a, b);
  if (rc) return rc;
  return launch_knn<3, false>(a, b, st);
}

extern "C" int pdae_group_f32(const float *xyz, const float *center, int b, int n, int g, int m, int64_t *idx,
                              float *neighborhood, pdae_stream_t stream) {
  return group_impl(xyz, center, b, n, g, m, idx, neighborhood, false, static_cast<cudaStream_t>(stream));
}

extern "C" int pdae_group_ws_f32(const float *xyz, const float *center, int b, int n, int g, int m, int64_t *idx,
                                 float *neighborhood, void *workspace, size_t workspace_bytes, pdae_stream_t stream) {
  return group_impl(xyz, center, b, n, g, m, idx, neighborhood, false, static_cast<cudaStream_t>(stream), workspace,
                    workspace_bytes);
}

extern "C" int pdae_group_gather_f32(const float *xyz, const float *center, int b, int n, int g, int m, int64_t *idx,
                                     float *patches, pdae_stream_t stream) {
  return group_impl(xyz, center, b, n, g, m, idx, patches, true, static_cast<cudaStream_t>(stream));
}

// DGCNN kNN: x (b, c, n) channel-major, every point is a query.  Low channel counts (the first
// EdgeConv layer, c = 3) use the planar variant of the kernel above; wide feature layers are
// served by featknn.cu.
int pdae::feat_knn_generic(const float *x, int b, int c, int n, int k, int64_t *idx, cudaStream_t st) {
  if (b < 0 || c <= 0 || n < 0 || k <= 0) return PDAE_E_INVALID;
  if (b == 0 || n == 0) return 0;
  if (k > n || k > KNN_MAX_K) return PDAE_E_INVALID;
  if (!x || !idx) return PDAE_E_INVALID;
  if (c == 3 && k <= 64) return knn4_planar(x, b, n, k, idx, st);
  KnnArgs a{x, nullptr, nullptr, idx, nullptr, nullptr, 0u, 0, n, n, c, k, 0, 1, 0};
  const int rc = knn_plan(a, b);
  if (rc) return rc;
  return c == 3 ? launch_knn<3, true>(a, b, st) : launch_knn<0, true>(a, b, st);
}
