// chamfer.cu -- Chamfer distance forward (fused min/argmin, both directions in one launch),
// backward (gradient scatter through the saved argmin) and the reference-set-sharded variant
// that emits packed (distance, index) keys for a MIN all-reduce.
//
// Semantics follow extensions/chamfer_dist/chamfer.cu:15-145 (forward) and :173-201 (backward)
// of the reference: dist = min_k fma(dz,dz, fma(dx,dx, dy*dy)) with d* = b_k - a, idx = lowest k
// attaining it; backward g = 2*grad_dist, v = g*(a - b_idx), gx1[j] += v, gx2[idx] -= v.
//
// Design (FP32 FMA-pipe bound, see DESIGN.md):
//   * a CTA owns QT*CH_THREADS query points held in registers (each coordinate duplicated into a
//     64-bit register pair) and streams the other cloud through shared memory in planar
//     (SoA) tiles, so one LDS.128 feeds two packed FADD2/FMUL2/FFMA2 evaluations per query;
//   * the inner loop carries no index: the running minimum is updated with one FMNMX3 per two
//     pairs; the only bookkeeping is "which group of 16 reference points last lowered the
//     minimum" (one FSETP + SEL per sixteen pairs).  Every instruction that is not FMA-pipe work
//     costs a dispatch slot the FMA pipe could have used (packed ops take two), so the loop is
//     built to minimise them: 6 FMA-pipe slots + ~1.06 other slots per point pair;
//   * after the scan every thread re-evaluates the single 16-point group recorded for each of
//     its queries and takes the first point whose distance equals the minimum bit-for-bit ->
//     the lowest index, as the reference's strict `<` does.
#include <stdlib.h>

#include "chamfer_core.cuh"

namespace pdae {

struct ChamferDir {
  const float *q;   // (b, nq, 3) query cloud
  const float *r;   // (b, nr, 3) reference cloud (or local slice)
  float *dist;      // (b, nq) or null
  int *idx;         // (b, nq) or null
  uint64_t *keys;   // (b, nq) packed output (sharded mode) or null
  uint64_t *colkeys;  // (b, nr) symmetric mode: (min over the queries, 32*QT-query group id), RED.MIN target
  int nq, nr;
  int qtiles;       // CTAs per cloud for this direction (0 = direction absent)
  int ref_offset;   // global index of r[0] (sharded mode)
  int csplit;       // column chunks per row block (0 or 1 = a CTA streams the whole reference cloud); > 1 needs `keys`,
                    // pre-filled with the MIN identity: the chunks merge their (row minimum, lowest index) with RED.MIN
};

// chamfer_min_body (the scan of one row block) lives in chamfer_core.cuh.  QT = 4 queries per thread, or 1 for the
// two-scan path of clouds up to 256 points (see launch_min).
template <int QT, bool SYM>
__global__ void __launch_bounds__(CH_THREADS, 1) chamfer_min_kernel(const ChamferDir d0, const ChamferDir d1) {
  constexpr int W = CH_THREADS / 32;
  __shared__ __align__(16) float tile[2][3][CH_TILE];
  __shared__ __align__(16) unsigned colmin[SYM ? 2 : 1][W][SYM ? CH_TILE : 4];

  // column split (symmetric forward only, d1 absent): consecutive blocks are the chunks of one row block
  const int nc = d0.csplit > 1 ? d0.csplit : 1;
  const int per_cloud = (d0.qtiles + d1.qtiles) * nc;
  const int cloud = blockIdx.x / per_cloud;
  int t = blockIdx.x - cloud * per_cloud;
  const int chunk = t % nc;
  t /= nc;
  const bool second = t >= d0.qtiles;
  if (second) t -= d0.qtiles;
  const ChamferDir &d = second ? d1 : d0;
  int tile_begin = 0, tile_end = 0x7fffffff;
  if (nc > 1) {
    const int ntiles = (d.nr + CH_TILE - 1) / CH_TILE, tpc = (ntiles + nc - 1) / nc;
    tile_begin = chunk * tpc;
    tile_end = tile_begin + tpc;
    if (tile_begin >= ntiles) return;  // uniform for the CTA
  }
  chamfer_min_body<QT, SYM>(
      d.q + static_cast<size_t>(cloud) * d.nq * 3, d.r + static_cast<size_t>(cloud) * d.nr * 3, d.nq, d.nr,
      t * (QT * CH_THREADS), static_cast<size_t>(cloud), d.dist, d.idx, d.keys, d.ref_offset, d.colkeys, tile, colmin,
      tile_begin, tile_end, nc > 1);
}

// ---- tiny clouds (both sides <= SMALL_MAX points): one warp per (cloud, direction) -----------
// The reference spends a (32,16)x512 grid on these; Point-DAE's fine loss runs ~5000 clouds of
// 32..36 points per step (models/PointCAE_transformer.py:1066).  Mirrors the reference's
// `k == 0 || d < best` scan literally (including its NaN behaviour).
constexpr int SMALL_MAX = 128;
constexpr int SMALL_WARPS = 8;

__global__ void __launch_bounds__(SMALL_WARPS * 32) chamfer_small_kernel(const float *__restrict__ xyz1,
                                                                         const float *__restrict__ xyz2, int b, int n,
                                                                         int m, float *__restrict__ dist1,
                                                                         float *__restrict__ dist2, int *__restrict__ idx1,
                                                                         int *__restrict__ idx2) {
  __shared__ float sref[SMALL_WARPS][3 * SMALL_MAX];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long gw = static_cast<long long>(blockIdx.x) * SMALL_WARPS + warp;
  if (gw >= 2LL * b) return;
  const int cloud = static_cast<int>(gw >> 1);
  const bool second = gw & 1;
  const int nq = second ? m : n, nr = second ? n : m;
  const float *__restrict__ Q = (second ? xyz2 : xyz1) + static_cast<size_t>(cloud) * nq * 3;
  const float *__restrict__ R = (second ? xyz1 : xyz2) + static_cast<size_t>(cloud) * nr * 3;
  float *dist = (second ? dist2 : dist1) + static_cast<size_t>(cloud) * nq;
  int *idx = (second ? idx2 : idx1) + static_cast<size_t>(cloud) * nq;
  float *s = sref[warp];
  for (int i = lane; i < nr * 3; i += 32) s[i] = __ldg(R + i);
  __syncwarp();
  for (int q = lane; q < nq; q += 32) {
    const float x1 = __ldg(Q + 3 * q), y1 = __ldg(Q + 3 * q + 1), z1 = __ldg(Q + 3 * q + 2);
    float best = 0.0f;
    int besti = 0;
#pragma unroll 4
    for (int k = 0; k < nr; ++k) {
      const float d = dist_yxz(__fsub_rn(s[3 * k], x1), __fsub_rn(s[3 * k + 1], y1), __fsub_rn(s[3 * k + 2], z1));
      const bool take = (k == 0) || (d < best);
      best = take ? d : best;
      besti = take ? k : besti;
    }
    dist[q] = best;
    idx[q] = besti;
  }
}


// ---- fused mean losses: (mean f(dist1), mean f(dist2)) with f = identity (L2) or sqrt (L1) ------------------
// reference: extensions/chamfer_dist/__init__.py:43 (L2: mean + mean) and :413-417 (L1: (mean sqrt + mean sqrt) / 2),
// there two or four torch kernels plus the add.  Deterministic: fixed-size partial sums in fp32 per CTA (fp64 across
// the CTA partials), summed in a fixed order by the second launch.
constexpr int LOSS_BLOCKS = 128;

__global__ void __launch_bounds__(256) chamfer_loss_partial_kernel(const float *__restrict__ dist1, const float *__restrict__ dist2,
                                                                   long long c1, long long c2, int l1,
                                                                   float *__restrict__ partial /*[2][LOSS_BLOCKS]*/) {
  __shared__ float red[2][8];
  float acc[2] = {0.f, 0.f};
#pragma unroll
  for (int side = 0; side < 2; ++side) {
    const float *__restrict__ d = side ? dist2 : dist1;
    const long long cnt = side ? c2 : c1;
    // four strided loads in flight per round (the sum is latency-bound: 8 values per thread at the headline shape)
    constexpr long long STRIDE = 256LL * LOSS_BLOCKS;
    for (long long i = static_cast<long long>(blockIdx.x) * 256 + threadIdx.x; i < cnt; i += 4 * STRIDE) {
      float v[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) v[u] = i + u * STRIDE < cnt ? __ldg(d + i + u * STRIDE) : 0.f;
#pragma unroll
      for (int u = 0; u < 4; ++u) acc[side] += l1 ? __fsqrt_rn(v[u]) : v[u];
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc[side] += __shfl_xor_sync(0xffffffffu, acc[side], o);
    if ((threadIdx.x & 31) == 0) red[side][threadIdx.x >> 5] = acc[side];
  }
  __syncthreads();
  if (threadIdx.x < 2) {
    float t = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) t += red[threadIdx.x][w];
    partial[threadIdx.x * LOSS_BLOCKS + blockIdx.x] = t;
  }
}

__global__ void __launch_bounds__(32) chamfer_loss_final_kernel(const float *__restrict__ partial, long long c1, long long c2,
                                                                int l1, float *__restrict__ out /*[3]*/) {
  // lanes 0-15 sum the first term's partials, lanes 16-31 the second's: 8 each, then a fixed shuffle tree (deterministic)
  const int side = threadIdx.x >> 4, l = threadIdx.x & 15;
  double t = 0.0;
#pragma unroll
  for (int i = 0; i < LOSS_BLOCKS / 16; ++i) t += static_cast<double>(partial[side * LOSS_BLOCKS + l * (LOSS_BLOCKS / 16) + i]);
#pragma unroll
  for (int o = 8; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
  const long long cnt = side ? c2 : c1;
  const float mean = static_cast<float>(t / static_cast<double>(cnt));  // 0/0 = NaN like torch.mean of an empty tensor
  const float other = __shfl_xor_sync(0xffffffffu, mean, 16);
  if (l == 0) out[1 + side] = mean;
  if (threadIdx.x == 0) out[0] = l1 ? __fmul_rn(__fadd_rn(mean, other), 0.5f) : __fadd_rn(mean, other);
}

__global__ void __launch_bounds__(256) unpack_keys_kernel(const uint64_t *__restrict__ keys, long long count,
                                                          float *__restrict__ dist, int *__restrict__ idx) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= count) return;
  const uint64_t k = keys[i];
  dist[i] = __uint_as_float(static_cast<uint32_t>(k >> 32));
  idx[i] = static_cast<int>(static_cast<uint32_t>(k));
}

// queries per CTA of the kernel launch_min will pick (the callers size `qtiles` with it)
static int chamfer_qpc(int nq_max, bool sym) { return !sym && nq_max <= 256 ? CH_THREADS : 4 * CH_THREADS; }

template <bool SYM>
static int launch_min(const ChamferDir &d0, const ChamferDir &d1, int b, cudaStream_t st) {
  const long long per_cloud = (static_cast<long long>(d0.qtiles) + d1.qtiles) * (d0.csplit > 1 ? d0.csplit : 1);
  const long long grid = per_cloud * b;
  if (grid <= 0) return 0;
  if (grid > 0x7fffffffLL) return PDAE_E_UNSUPPORTED;
  const unsigned g = static_cast<unsigned>(grid);
  const int nq_max = d0.nq > d1.nq ? d0.nq : d1.nq;
  if (chamfer_qpc(nq_max, SYM) == CH_THREADS) chamfer_min_kernel<1, false><<<g, CH_THREADS, 0, st>>>(d0, d1);
  else chamfer_min_kernel<4, SYM><<<g, CH_THREADS, 0, st>>>(d0, d1);
  PDAE_RETURN_IF_LAUNCH_FAILED();
  return 0;
}

// identity of the MIN reduction over packed keys: larger than every real key both as uint64 and as
// int64 (torch / NCCL reduce the keys as signed 64-bit; real keys have a clear top bit because d >= 0).
constexpr uint64_t CHAMFER_KEY_IDENTITY = 0x7fffffffffffffffull;

__global__ void __launch_bounds__(256) fill_keys_kernel(uint64_t *__restrict__ keys, long long count) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i < count) keys[i] = CHAMFER_KEY_IDENTITY;
}

// rows per column-key group: the 32*QT queries of one warp of the symmetric scan, chamfer_min_kernel<4, true>
constexpr int RECOVER_QPG = 32 * 4;
// the list recovery serves clouds up to this many row groups, the warp-per-column recovery larger ones
constexpr int RECOVER_LIST_GROUPS = 128;

// symmetric mode, second half: the column recovery.  colkeys[j] = (min_i d(a_i, b_j), id of the QPG-query group holding
// a minimiser; lowest such group), QPG = RECOVER_QPG.  Scanning that group in index order and taking the first query
// whose distance equals the minimum bit for bit yields the lowest index overall.
// Warp-per-column form, for clouds above RECOVER_LIST_GROUPS groups: one warp per column point b_j.  A group's queries
// are contiguous, so each lane takes QPG/32 consecutive ones (float4 loads when the cloud base is 16-byte aligned) and
// the whole group is examined in one step; lanes are in index order, hence ballot + ffs gives the lowest index.  A warp
// resolves RPW consecutive column points with all their loads issued up front: the kernel is pure load latency
// (key -> group rows), so the memory-level parallelism per warp is what sets its speed.
template <int QPG, int RPW>
__global__ void __launch_bounds__(256) chamfer_col_recover_kernel(const float *__restrict__ rows, const float *__restrict__ cols,
                                                                  const uint64_t *__restrict__ colkeys, int n_rows,
                                                                  int n_cols,
                                                                  float *__restrict__ dist, int *__restrict__ idx) {
  constexpr int PER = QPG / 32;  // consecutive queries per lane
  const int lane = threadIdx.x & 31;
  const int j0 = ((blockIdx.x * blockDim.x + threadIdx.x) >> 5) * RPW;  // first column point of the warp
  if (j0 >= n_cols) return;
  const size_t cloud = blockIdx.y;
  const float *__restrict__ A = rows + cloud * n_rows * 3;
  const bool vec = (n_rows & 3) == 0 && PER % 4 == 0;
  uint64_t key[RPW];
  float bx[RPW], by[RPW], bz[RPW];
#pragma unroll
  for (int u = 0; u < RPW; ++u) {
    const int j = j0 + u < n_cols ? j0 + u : n_cols - 1;
    const size_t gw = cloud * n_cols + j;
    key[u] = colkeys[gw];
    bx[u] = __ldg(cols + 3 * gw); by[u] = __ldg(cols + 3 * gw + 1); bz[u] = __ldg(cols + 3 * gw + 2);
  }
  float c[RPW][3 * PER];
  int base[RPW];
#pragma unroll
  for (int u = 0; u < RPW; ++u) {
    base[u] = static_cast<int>(static_cast<uint32_t>(key[u])) * QPG + lane * PER;
    if (vec && base[u] + PER <= n_rows) {
      const float4 *p4 = reinterpret_cast<const float4 *>(A + 3 * static_cast<size_t>(base[u]));
#pragma unroll
      for (int t = 0; t < 3 * PER / 4; ++t) {
        const float4 w = __ldg(p4 + t);
        c[u][4 * t] = w.x; c[u][4 * t + 1] = w.y; c[u][4 * t + 2] = w.z; c[u][4 * t + 3] = w.w;
      }
    } else {
#pragma unroll
      for (int t = 0; t < 3 * PER; ++t)
        c[u][t] = (base[u] + t / 3 < n_rows) ? __ldg(A + 3 * static_cast<size_t>(base[u]) + t) : __int_as_float(0x7fc00000);
    }
  }
#pragma unroll
  for (int u = 0; u < RPW; ++u) {
    const float v = __uint_as_float(static_cast<uint32_t>(key[u] >> 32));
    int first = PER;  // first matching query of this lane
#pragma unroll
    for (int t = PER - 1; t >= 0; --t) {
      const float d = dist_yxz(__fsub_rn(bx[u], c[u][3 * t]), __fsub_rn(by[u], c[u][3 * t + 1]), __fsub_rn(bz[u], c[u][3 * t + 2]));
      first = (d == v) ? t : first;  // NaN padding never matches
    }
    const unsigned mk = __ballot_sync(0xffffffffu, first < PER);
    const int src = mk ? __ffs(mk) - 1 : 0;
    const int found = __shfl_sync(0xffffffffu, base[u] + first, src);
    if (lane == 0 && j0 + u < n_cols) {
      const size_t gw = cloud * n_cols + j0 + u;
      dist[gw] = v;
      idx[gw] = mk ? found : 0;
    }
  }
}

// List form of the recovery, for clouds up to RECOVER_LIST_GROUPS groups: the CTA of (cloud, group) stages the
// group's QPG rows in shared memory as planes, every thread tests a strided share of the cloud's column keys and
// appends the columns won by this group to a shared list, and then ONE THREAD PER LISTED COLUMN walks the group's rows
// (broadcast LDS.64 of two rows per plane, packed distance, compare with the recorded minimum bit for bit), back to
// front so that the lowest matching row is the one kept.  No shuffles or ballots in the walk: ~6.5 instructions per
// (column, row).  The warp-per-column kernel above re-reads a whole group (12*QPG bytes) per column; here the traffic
// is the keys once per group (8*n_cols bytes per CTA), which grows with n_rows*n_cols/QPG -- hence the size limit.
constexpr int RECOVER_LIST_MAX = 4096;  // columns examined per pass (list of int in shared memory)

template <int QPG>
__global__ void __launch_bounds__(256) chamfer_col_recover_list_kernel(const float *__restrict__ rows,
                                                                       const float *__restrict__ cols,
                                                                       const uint64_t *__restrict__ colkeys, int n_rows,
                                                                       int n_cols, float *__restrict__ dist,
                                                                       int *__restrict__ idx,
                                                                       const uint64_t *__restrict__ rowkeys,
                                                                       float *__restrict__ drow, int *__restrict__ irow) {
  __shared__ __align__(16) float sx[QPG], sy[QPG], sz[QPG];
  __shared__ int list[RECOVER_LIST_MAX];
  __shared__ int count;
  const unsigned g = blockIdx.x;
  const size_t cloud = blockIdx.y;
  const float *__restrict__ A = rows + cloud * n_rows * 3;
  const uint64_t *__restrict__ K = colkeys + cloud * n_cols;
  const float *__restrict__ C = cols + cloud * n_cols * 3;
  const int tid = threadIdx.x;
  if (tid == 0) count = 0;
  if (rowkeys != nullptr) {  // column-split forward: this CTA's rows leave their merged keys here (no extra launch)
    for (int r = tid; r < QPG; r += 256) {
      const long long row = static_cast<long long>(g) * QPG + r;
      if (row < n_rows) {
        const uint64_t key = rowkeys[cloud * n_rows + row];
        drow[cloud * n_rows + row] = __uint_as_float(static_cast<uint32_t>(key >> 32));
        irow[cloud * n_rows + row] = static_cast<int>(static_cast<uint32_t>(key));
      }
    }
  }
  for (int e = tid; e < 3 * QPG; e += 256) {  // coalesced AoS read of the group's rows; NaN padding never matches
    const int r = e / 3, c = e - 3 * r;
    const long long row = static_cast<long long>(g) * QPG + r;
    const float v = row < n_rows ? __ldg(A + row * 3 + c) : __int_as_float(0x7fc00000);
    (c == 0 ? sx : c == 1 ? sy : sz)[r] = v;
  }
  __syncthreads();
  constexpr int UNR = 8;
  for (int c0 = 0; c0 < n_cols; c0 += RECOVER_LIST_MAX) {  // the list holds one chunk of columns at a time
    const int c1 = c0 + RECOVER_LIST_MAX < n_cols ? c0 + RECOVER_LIST_MAX : n_cols;
    for (int j0 = c0 + tid; j0 < c1; j0 += 256 * UNR) {
      uint32_t gid[UNR];
#pragma unroll
      for (int u = 0; u < UNR; ++u) {
        const int j = j0 + u * 256;
        gid[u] = j < c1 ? static_cast<uint32_t>(K[j]) : 0xffffffffu;
      }
#pragma unroll
      for (int u = 0; u < UNR; ++u)
        if (gid[u] == g) list[atomicAdd(&count, 1)] = j0 + u * 256;
    }
    __syncthreads();
    const int total = count;
    for (int m = tid; m < total; m += 256) {
      const int j = list[m];
      const float want = __uint_as_float(static_cast<uint32_t>(K[j] >> 32));
      const float bx = __ldg(C + 3 * j), by = __ldg(C + 3 * j + 1), bz = __ldg(C + 3 * j + 2);
      const float2 cx = make_float2(bx, bx), cy = make_float2(by, by), cz = make_float2(bz, bz);
      int found = 0;
#pragma unroll 8
      for (int r = QPG - 2; r >= 0; r -= 2) {
        const float2 d = dist_yxz2(sub2(cx, *reinterpret_cast<const float2 *>(sx + r)),
                                   sub2(cy, *reinterpret_cast<const float2 *>(sy + r)),
                                   sub2(cz, *reinterpret_cast<const float2 *>(sz + r)));
        found = (d.y == want) ? r + 1 : found;
        found = (d.x == want) ? r : found;
      }
      dist[cloud * n_cols + j] = want;
      idx[cloud * n_cols + j] = static_cast<int>(g) * QPG + found;
    }
    __syncthreads();
    if (tid == 0) count = 0;
    __syncthreads();
  }
}

// true when the list kernel recovers a cloud of n_rows rows.  It visits every row exactly once, so it also unpacks the
// row keys of an (unphased) column-split forward.
static bool recover_unpacks_rows(int n_rows) {
  return (static_cast<long long>(n_rows) + RECOVER_QPG - 1) / RECOVER_QPG <= RECOVER_LIST_GROUPS;
}

// second half of the symmetric forward: picks the recovery kernel by cloud size
static int launch_col_recover(const float *rows, const float *cols, const uint64_t *ck, int b, int n_rows, int n_cols,
                              float *dcol, int *icol, cudaStream_t st, const uint64_t *rowkeys = nullptr,
                              float *drow = nullptr, int *irow = nullptr) {
  if (recover_unpacks_rows(n_rows)) {
    const dim3 ggrid(static_cast<unsigned>(ceil_div(n_rows, RECOVER_QPG)), b);
    chamfer_col_recover_list_kernel<RECOVER_QPG><<<ggrid, 256, 0, st>>>(rows, cols, ck, n_rows, n_cols, dcol, icol, rowkeys,
                                                                        drow, irow);
  } else {
    if (rowkeys) return PDAE_E_INVALID;
    // 4 column points per warp, 8 warps per CTA (splitting a warp across points was measured slower)
    const dim3 rgrid(static_cast<unsigned>((n_cols + 31) / 32), b);
    chamfer_col_recover_kernel<RECOVER_QPG, 4><<<rgrid, 256, 0, st>>>(rows, cols, ck, n_rows, n_cols, dcol, icol);
  }
  PDAE_RETURN_IF_LAUNCH_FAILED();
  return 0;
}

}  // namespace pdae

using namespace pdae;

// column keys of the smaller cloud + (for column-split units) row keys of the larger one.  A workspace of only the
// first part (b * min(n, m) keys, the size this function returned before the split existed) is still accepted: the
// forward then runs unsplit.
extern "C" size_t pdae_chamfer_fwd_workspace_bytes(int b, int n, int m) {
  if (b <= 0 || n <= 0 || m <= 0) return 0;
  if (n <= SMALL_MAX && m <= SMALL_MAX) return 0;
  return static_cast<size_t>(b) * (static_cast<size_t>(n) + m) * sizeof(uint64_t);
}

// Column chunks per 512-row block for the symmetric forward.  One 4-warp CTA saturates an SM's FMA issue, so an SM
// works through its CTAs at a fixed rate and the kernel ends when the SM with the most CTAs ends: with U equal units
// on S SMs that is ceil(U / S) unit times.  512 row blocks on 148 SMs (128 x 2048^2) make 4 against an average of
// 3.46; cutting every block's column sweep in two makes 7 half-units against 6.92.  A unit costs its tiles plus a
// fixed prologue / epilogue (first tile not overlapped, query loads, 16-point rescan, key posts), put at a quarter
// of a 512-point tile.  PDAE_CHAMFER_SPLIT forces a value (1 = never split).
static int g_chamfer_split = -1;
static int chamfer_split_forced() {
  if (g_chamfer_split < 0) {
    const char *e = getenv("PDAE_CHAMFER_SPLIT");
    g_chamfer_split = e ? atoi(e) : 0;
  }
  return g_chamfer_split;
}
static int chamfer_csplit(long long row_units, int ntiles) {
  const int forced = chamfer_split_forced();
  if (ntiles <= 1) return 1;
  if (forced > 0) return forced < ntiles ? forced : ntiles;
  const long long sms = sm_count();
  int best_nc = 1;
  double best_cost = 0.0;
  for (int nc = 1; nc <= ntiles && nc <= 16; ++nc) {
    const int tpc = (ntiles + nc - 1) / nc;
    const long long chunks = (ntiles + tpc - 1) / tpc;  // chunks that actually hold tiles
    const long long waves = (row_units * chunks + sms - 1) / sms;
    const double cost = static_cast<double>(waves) * (tpc + 0.25);
    if (nc == 1 || cost < best_cost * 0.97) {  // split only for a clear (> 3 %) gain
      best_cost = cost;
      best_nc = nc;
    }
  }
  return best_nc;
}

// phase 0: the whole forward; 1: everything except the column recovery of the symmetric path (the "scan": row
// results final, column minima parked in the workspace); 2: only that recovery.  Paths without a separate recovery
// (tiny clouds, two-scan, empty inputs) do all their work in phase 1 and nothing in phase 2.
static int chamfer_fwd_impl(const float *xyz1, const float *xyz2, int b, int n, int m, float *dist1, float *dist2,
                            int *idx1, int *idx2, void *workspace, size_t workspace_bytes, pdae_stream_t stream,
                            int phase) {
  if (b < 0 || n < 0 || m < 0) return PDAE_E_INVALID;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const size_t bn = static_cast<size_t>(b) * n, bm = static_cast<size_t>(b) * m;
  if ((bn && (!xyz1 || !dist1 || !idx1)) || (bm && (!xyz2 || !dist2 || !idx2))) return PDAE_E_INVALID;
  if (b == 0) return 0;
  const int nq_max = n > m ? n : m;
  const size_t need = static_cast<size_t>(b) * (n < m ? n : m) * sizeof(uint64_t);  // column keys (the row keys are optional)
  const bool sym = n > 0 && m > 0 && !(n <= SMALL_MAX && m <= SMALL_MAX) && workspace != nullptr &&
                   workspace_bytes >= need && nq_max > 256 &&
                   b <= 65535;  // the recovery kernels index clouds with gridDim.y; larger batches take the two-scan path
  if (phase == 2 && !sym) return 0;
  if (n == 0 || m == 0) {  // reference: outputs stay at their zero initialisation (chamfer.cu:152-157)
    if (bn) {
      PDAE_CUDA_TRY(cudaMemsetAsync(dist1, 0, bn * sizeof(float), st));
      PDAE_CUDA_TRY(cudaMemsetAsync(idx1, 0, bn * sizeof(int), st));
    }
    if (bm) {
      PDAE_CUDA_TRY(cudaMemsetAsync(dist2, 0, bm * sizeof(float), st));
      PDAE_CUDA_TRY(cudaMemsetAsync(idx2, 0, bm * sizeof(int), st));
    }
    return 0;
  }
  if (n <= SMALL_MAX && m <= SMALL_MAX) {
    const long long warps = 2LL * b;
    const long long grid = (warps + SMALL_WARPS - 1) / SMALL_WARPS;
    if (grid > 0x7fffffffLL) return PDAE_E_UNSUPPORTED;
    chamfer_small_kernel<<<static_cast<unsigned>(grid), SMALL_WARPS * 32, 0, st>>>(xyz1, xyz2, b, n, m, dist1, dist2,
                                                                                  idx1, idx2);
    PDAE_RETURN_IF_LAUNCH_FAILED();
    return 0;
  }
  if (chamfer_tc_applies(b, n, m, workspace ? workspace_bytes : 0)) {  // tensor-core filter + exact evaluation (chamfer_tc.cu)
    if (phase == 2) return 0;
    return chamfer_tc_forward(xyz1, xyz2, b, n, m, dist1, dist2, idx1, idx2, workspace, workspace_bytes, st);
  }
  if (sym) {
    // rows (register-resident queries) = the larger cloud, columns = the smaller one
    const bool swap = m > n;
    const float *rows = swap ? xyz2 : xyz1, *cols = swap ? xyz1 : xyz2;
    const int nr_rows = swap ? m : n, nr_cols = swap ? n : m;
    float *drow = swap ? dist2 : dist1, *dcol = swap ? dist1 : dist2;
    int *irow = swap ? idx2 : idx1, *icol = swap ? idx1 : idx2;
    uint64_t *ck = static_cast<uint64_t *>(workspace);
    const long long ncol = static_cast<long long>(b) * nr_cols;
    const long long nrow = static_cast<long long>(b) * nr_rows;
    // column split: only with room for the row keys
    const int nsplit = workspace_bytes >= static_cast<size_t>(ncol + nrow) * sizeof(uint64_t)
                           ? chamfer_csplit(static_cast<long long>(b) * ceil_div(nr_rows, 512), ceil_div(nr_cols, 512))
                           : 1;
    // the whole forward in one call: the list recovery writes the rows' results while it is there
    const bool fused_unpack = nsplit > 1 && phase == 0 && recover_unpacks_rows(nr_rows);
    if (phase != 2) {
      const long long nfill = nsplit > 1 ? ncol + nrow : ncol;
      fill_keys_kernel<<<static_cast<unsigned>((nfill + 255) / 256), 256, 0, st>>>(ck, nfill);
      PDAE_RETURN_IF_LAUNCH_FAILED();
      const int qpc = chamfer_qpc(nr_rows, true);
      ChamferDir d0{rows, cols, drow, irow, nullptr, ck, nr_rows, nr_cols, ceil_div(nr_rows, qpc), 0};
      ChamferDir d1{nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, 0, 0, 0, 0};
      if (nsplit > 1) {  // rows leave as merged keys instead of dist / idx
        d0.csplit = nsplit;
        d0.keys = ck + ncol;
        d0.dist = nullptr;
        d0.idx = nullptr;
      }
      const int rc = launch_min<true>(d0, d1, b, st);
      if (rc) return rc;
      if (nsplit > 1 && !fused_unpack) {  // merged row keys -> dist / idx of the larger cloud
        unpack_keys_kernel<<<static_cast<unsigned>((nrow + 255) / 256), 256, 0, st>>>(ck + ncol, nrow, drow, irow);
        PDAE_RETURN_IF_LAUNCH_FAILED();
      }
    }
    if (phase == 1) return 0;
    if (fused_unpack) return launch_col_recover(rows, cols, ck, b, nr_rows, nr_cols, dcol, icol, st, ck + ncol, drow, irow);
    return launch_col_recover(rows, cols, ck, b, nr_rows, nr_cols, dcol, icol, st);
  }
  const int qpc = chamfer_qpc(nq_max, false);
  ChamferDir d0{xyz1, xyz2, dist1, idx1, nullptr, nullptr, n, m, ceil_div(n, qpc), 0};
  ChamferDir d1{xyz2, xyz1, dist2, idx2, nullptr, nullptr, m, n, ceil_div(m, qpc), 0};
  return launch_min<false>(d0, d1, b, st);
}

// tuning / test hook: force the number of column chunks inside one process (0 = automatic, 1 = never split);
// returns the previous setting, a negative argument only queries.
extern "C" int pdae_tune_chamfer_split(int nc) {
  const int old = chamfer_split_forced();
  if (nc >= 0) g_chamfer_split = nc;
  return old;
}

extern "C" int pdae_chamfer_fwd_f32(const float *xyz1, const float *xyz2, int b, int n, int m, float *dist1,
                                    float *dist2, int *idx1, int *idx2, void *workspace, size_t workspace_bytes,
                                    pdae_stream_t stream) {
  return chamfer_fwd_impl(xyz1, xyz2, b, n, m, dist1, dist2, idx1, idx2, workspace, workspace_bytes, stream, 0);
}

extern "C" int pdae_chamfer_fwd_phase_f32(const float *xyz1, const float *xyz2, int b, int n, int m, float *dist1,
                                          float *dist2, int *idx1, int *idx2, void *workspace, size_t workspace_bytes,
                                          int phase, pdae_stream_t stream) {
  if (phase != 1 && phase != 2) return PDAE_E_INVALID;
  return chamfer_fwd_impl(xyz1, xyz2, b, n, m, dist1, dist2, idx1, idx2, workspace, workspace_bytes, stream, phase);
}

extern "C" int pdae_chamfer_min_keys_u64(const float *queries, const float *refs, int b, int nq, int nr,
                                         int ref_offset, uint64_t *keys, pdae_stream_t stream) {
  if (b < 0 || nq < 0 || nr < 0 || ref_offset < 0) return PDAE_E_INVALID;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const size_t bq = static_cast<size_t>(b) * nq;
  if (bq == 0) return 0;
  if (!queries || !keys || (nr && !refs)) return PDAE_E_INVALID;
  if (nr == 0) {  // empty slice: identity of MIN
    fill_keys_kernel<<<static_cast<unsigned>((bq + 255) / 256), 256, 0, st>>>(keys, static_cast<long long>(bq));
    PDAE_RETURN_IF_LAUNCH_FAILED();
    return 0;
  }
  const int qpc = chamfer_qpc(nq, false);
  ChamferDir d0{queries, refs, nullptr, nullptr, keys, nullptr, nq, nr, ceil_div(nq, qpc), ref_offset};
  ChamferDir d1{nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, 0, 0, 0, 0};
  const int nsplit = nq > 256 ? chamfer_csplit(static_cast<long long>(b) * ceil_div(nq, 512), ceil_div(nr, 512)) : 1;
  if (nsplit > 1) {  // column-split units merge into the output keys
    fill_keys_kernel<<<static_cast<unsigned>((bq + 255) / 256), 256, 0, st>>>(keys, static_cast<long long>(bq));
    PDAE_RETURN_IF_LAUNCH_FAILED();
    d0.csplit = nsplit;
  }
  return launch_min<false>(d0, d1, b, st);
}

// one rank's share of a reference-set-sharded Chamfer forward: all of xyz1 against the local slice of xyz2,
// every pair evaluated once (symmetric kernel): row minima leave as packed keys for the MIN all-reduce, column
// minima are already final for the slice because every rank sees all of xyz1.
extern "C" int pdae_chamfer_sharded_f32(const float *xyz1, const float *xyz2_local, int b, int n, int m_local,
                                        int ref_offset, uint64_t *keys1, float *dist2_local, int *idx2_local,
                                        void *workspace, size_t workspace_bytes, pdae_stream_t stream) {
  if (b < 0 || n < 0 || m_local < 0 || ref_offset < 0) return PDAE_E_INVALID;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const size_t bn = static_cast<size_t>(b) * n, bm = static_cast<size_t>(b) * m_local;
  if (b == 0) return 0;
  if (bn && (!xyz1 || !keys1)) return PDAE_E_INVALID;
  if (bm && (!xyz2_local || !dist2_local || !idx2_local)) return PDAE_E_INVALID;
  if (b > 65535) return PDAE_E_UNSUPPORTED;
  if (m_local == 0) {
    if (bn) {
      fill_keys_kernel<<<static_cast<unsigned>((bn + 255) / 256), 256, 0, st>>>(keys1, static_cast<long long>(bn));
      PDAE_RETURN_IF_LAUNCH_FAILED();
    }
    return 0;
  }
  if (n == 0) {  // reference: outputs stay zero
    PDAE_CUDA_TRY(cudaMemsetAsync(dist2_local, 0, bm * sizeof(float), st));
    PDAE_CUDA_TRY(cudaMemsetAsync(idx2_local, 0, bm * sizeof(int), st));
    return 0;
  }
  if (!workspace || workspace_bytes < bm * sizeof(uint64_t)) return PDAE_E_WORKSPACE;
  if (chamfer_tc_sharded_applies(b, n, m_local))  // tensor-core filter in column chunks; same keys (chamfer_tc.cu)
    return chamfer_tc_sharded(xyz1, xyz2_local, b, n, m_local, ref_offset, keys1, dist2_local, idx2_local, workspace,
                              workspace_bytes, st);
  uint64_t *ck = static_cast<uint64_t *>(workspace);
  fill_keys_kernel<<<static_cast<unsigned>((bm + 255) / 256), 256, 0, st>>>(ck, static_cast<long long>(bm));
  PDAE_RETURN_IF_LAUNCH_FAILED();
  const int qpc = chamfer_qpc(n, true);
  ChamferDir d0{xyz1, xyz2_local, nullptr, nullptr, keys1, ck, n, m_local, ceil_div(n, qpc), ref_offset};
  ChamferDir d1{nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, 0, 0, 0, 0};
  // a single scene-scale cloud gives few row blocks (100 000 points: 196 for 148 SMs): column-split units, merged
  // through the very keys this call returns
  const int nsplit = chamfer_csplit(static_cast<long long>(b) * ceil_div(n, 512), ceil_div(m_local, 512));
  if (nsplit > 1) {
    fill_keys_kernel<<<static_cast<unsigned>((bn + 255) / 256), 256, 0, st>>>(keys1, static_cast<long long>(bn));
    PDAE_RETURN_IF_LAUNCH_FAILED();
    d0.csplit = nsplit;
  }
  const int rc = launch_min<true>(d0, d1, b, st);
  if (rc) return rc;
  return launch_col_recover(xyz1, xyz2_local, ck, b, n, m_local, dist2_local, idx2_local, st);
}

extern "C" int pdae_chamfer_unpack_keys(const uint64_t *keys, long long count, float *dist, int *idx,
                                        pdae_stream_t stream) {
  if (count < 0) return PDAE_E_INVALID;
  if (count == 0) return 0;
  if (!keys || !dist || !idx) return PDAE_E_INVALID;
  const long long grid = (count + 255) / 256;
  if (grid > 0x7fffffffLL) return PDAE_E_UNSUPPORTED;
  unpack_keys_kernel<<<static_cast<unsigned>(grid), 256, 0, static_cast<cudaStream_t>(stream)>>>(keys, count, dist, idx);
  PDAE_RETURN_IF_LAUNCH_FAILED();
  return 0;
}

extern "C" int pdae_chamfer_bwd_f32(const float *xyz1, const float *xyz2, const int *idx1, const int *idx2,
                                    const float *gd1, const float *gd2, int b, int n, int m, float *gx1, float *gx2,
                                    pdae_stream_t stream) {
  if (b < 0 || n < 0 || m < 0) return PDAE_E_INVALID;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const long long t1 = static_cast<long long>(b) * n, t2 = static_cast<long long>(b) * m;
  if ((t1 && (!xyz1 || !gx1)) || (t2 && (!xyz2 || !gx2))) return PDAE_E_INVALID;
  if (n == 0 || m == 0 || b == 0) {  // reference: the loops never execute, grads stay zero
    if (t1) PDAE_CUDA_TRY(cudaMemsetAsync(gx1, 0, static_cast<size_t>(t1) * 3 * sizeof(float), st));
    if (t2) PDAE_CUDA_TRY(cudaMemsetAsync(gx2, 0, static_cast<size_t>(t2) * 3 * sizeof(float), st));
    return 0;
  }
  if (!idx1 || !idx2 || !gd1 || !gd2) return PDAE_E_INVALID;
  return launch_chamfer_bwd(xyz1, xyz2, idx1, idx2, GradArrays{gd1, gd2}, b, n, m, gx1, gx2, st);
}

extern "C" size_t pdae_chamfer_loss_workspace_bytes(void) { return 2 * LOSS_BLOCKS * sizeof(float); }

extern "C" int pdae_chamfer_loss_f32(const float *dist1, const float *dist2, int b, int n, int m, int l1, float *loss3,
                                     void *workspace, size_t workspace_bytes, pdae_stream_t stream) {
  if (b < 0 || n < 0 || m < 0 || !loss3) return PDAE_E_INVALID;
  if (!workspace || workspace_bytes < pdae_chamfer_loss_workspace_bytes()) return PDAE_E_WORKSPACE;
  const long long c1 = static_cast<long long>(b) * n, c2 = static_cast<long long>(b) * m;
  if ((c1 && !dist1) || (c2 && !dist2)) return PDAE_E_INVALID;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  float *partial = static_cast<float *>(workspace);
  chamfer_loss_partial_kernel<<<LOSS_BLOCKS, 256, 0, st>>>(dist1, dist2, c1, c2, l1 ? 1 : 0, partial);
  PDAE_RETURN_IF_LAUNCH_FAILED();
  chamfer_loss_final_kernel<<<1, 32, 0, st>>>(partial, c1, c2, l1 ? 1 : 0, loss3);
  PDAE_RETURN_IF_LAUNCH_FAILED();
  return 0;
}

extern "C" int pdae_chamfer_loss_bwd_f32(const float *xyz1, const float *xyz2, const int *idx1, const int *idx2,
                                         const float *dist1, const float *dist2, const float *gloss, float w1, float w2,
                                         int b, int n, int m, int l1, float *gx1, float *gx2, pdae_stream_t stream) {
  if (b < 0 || n < 0 || m < 0) return PDAE_E_INVALID;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const long long t1 = static_cast<long long>(b) * n, t2 = static_cast<long long>(b) * m;
  if ((t1 && (!xyz1 || !gx1)) || (t2 && (!xyz2 || !gx2))) return PDAE_E_INVALID;
  if (n == 0 || m == 0 || b == 0) {
    if (t1) PDAE_CUDA_TRY(cudaMemsetAsync(gx1, 0, static_cast<size_t>(t1) * 3 * sizeof(float), st));
    if (t2) PDAE_CUDA_TRY(cudaMemsetAsync(gx2, 0, static_cast<size_t>(t2) * 3 * sizeof(float), st));
    return 0;
  }
  if (!idx1 || !idx2 || !gloss || (l1 && (!dist1 || !dist2))) return PDAE_E_INVALID;
  const float n1 = static_cast<float>(t1), n2 = static_cast<float>(t2);
  return launch_chamfer_bwd(xyz1, xyz2, idx1, idx2, GradMean{gloss, dist1, dist2, w1 / n1, w2 / n2, l1 ? 1 : 0}, b, n, m, gx1,
                            gx2, st);
}

extern "C" size_t pdae_chamfer_bwd_det_workspace_bytes(int b, int n, int m) {
  if (b <= 0 || n <= 0 || m <= 0) return 0;
  return chamfer_bwd_det_bytes(b, n, m);
}

extern "C" int pdae_chamfer_bwd_det_f32(const float *xyz1, const float *xyz2, const int *idx1, const int *idx2,
                                        const float *gd1, const float *gd2, int b, int n, int m, float *gx1, float *gx2,
                                        void *workspace, size_t workspace_bytes, pdae_stream_t stream) {
  if (b < 0 || n < 0 || m < 0) return PDAE_E_INVALID;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const long long t1 = static_cast<long long>(b) * n, t2 = static_cast<long long>(b) * m;
  if ((t1 && (!xyz1 || !gx1)) || (t2 && (!xyz2 || !gx2))) return PDAE_E_INVALID;
  if (n == 0 || m == 0 || b == 0) {
    if (t1) PDAE_CUDA_TRY(cudaMemsetAsync(gx1, 0, static_cast<size_t>(t1) * 3 * sizeof(float), st));
    if (t2) PDAE_CUDA_TRY(cudaMemsetAsync(gx2, 0, static_cast<size_t>(t2) * 3 * sizeof(float), st));
    return 0;
  }
  if (!idx1 || !idx2 || !gd1 || !gd2) return PDAE_E_INVALID;
  if (!workspace || workspace_bytes < pdae_chamfer_bwd_det_workspace_bytes(b, n, m)) return PDAE_E_WORKSPACE;
  return launch_chamfer_bwd_det(xyz1, xyz2, idx1, idx2, GradArrays{gd1, gd2}, b, n, m, gx1, gx2, workspace, st);
}

extern "C" int pdae_chamfer_loss_bwd_det_f32(const float *xyz1, const float *xyz2, const int *idx1, const int *idx2,
                                             const float *dist1, const float *dist2, const float *gloss, float w1, float w2,
                                             int b, int n, int m, int l1, float *gx1, float *gx2, void *workspace,
                                             size_t workspace_bytes, pdae_stream_t stream) {
  if (b < 0 || n < 0 || m < 0) return PDAE_E_INVALID;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const long long t1 = static_cast<long long>(b) * n, t2 = static_cast<long long>(b) * m;
  if ((t1 && (!xyz1 || !gx1)) || (t2 && (!xyz2 || !gx2))) return PDAE_E_INVALID;
  if (n == 0 || m == 0 || b == 0) {
    if (t1) PDAE_CUDA_TRY(cudaMemsetAsync(gx1, 0, static_cast<size_t>(t1) * 3 * sizeof(float), st));
    if (t2) PDAE_CUDA_TRY(cudaMemsetAsync(gx2, 0, static_cast<size_t>(t2) * 3 * sizeof(float), st));
    return 0;
  }
  if (!idx1 || !idx2 || !gloss || (l1 && (!dist1 || !dist2))) return PDAE_E_INVALID;
  if (!workspace || workspace_bytes < pdae_chamfer_bwd_det_workspace_bytes(b, n, m)) return PDAE_E_WORKSPACE;
  const float n1 = static_cast<float>(t1), n2 = static_cast<float>(t2);
  return launch_chamfer_bwd_det(xyz1, xyz2, idx1, idx2, GradMean{gloss, dist1, dist2, w1 / n1, w2 / n2, l1 ? 1 : 0}, b, n, m,
                                gx1, gx2, workspace, st);
}
