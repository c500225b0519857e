// featknn.cu -- DGCNN `knn` dispatch and the fused `get_graph_feature` gather (+ backward).
//
// Semantics follow models/dgcnn_util.py:7-36 of the reference: idx = k nearest neighbours of
// every point in feature space (self included, nearest first); feature = cat(x_j - x_i, x_i)
// returned as a (B, 2C, N, k) view of a physically (B, N, k, 2C) tensor.  The neighbour order is
// this repo's canonical one (direct-form distance, ties -> lower index; SURVEY.md appendix A.5).
//
// The graph-feature kernels are HBM-bound (output B*N*k*2C*4 bytes): x is transposed once into a
// (B, N, C) workspace so every neighbour row is one contiguous read, and the reference's
// index-select + repeat + cat + permute chain (4 passes) becomes one write pass.
#include <stdlib.h>

#include "knn_select.cuh"
#include "reverse.cuh"

namespace pdae {

// (b, rows, cols) -> (b, cols, rows), 32x32 shared-memory tiles
__global__ void __launch_bounds__(256) transpose_kernel(const float *__restrict__ in, float *__restrict__ out, int rows,
                                                        int cols) {
  __shared__ float t[32][33];
  const size_t base = static_cast<size_t>(blockIdx.z) * rows * cols;
  const int c0 = blockIdx.x * 32, r0 = blockIdx.y * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;  // 32 x 8
#pragma unroll
  for (int i = 0; i < 32; i += 8) {
    const int r = r0 + ty + i, c = c0 + tx;
    if (r < rows && c < cols) t[ty + i][tx] = __ldg(in + base + static_cast<size_t>(r) * cols + c);
  }
  __syncthreads();
#pragma unroll
  for (int i = 0; i < 32; i += 8) {
    const int c = c0 + ty + i, r = r0 + tx;
    if (r < rows && c < cols) out[base + static_cast<size_t>(c) * rows + r] = t[tx][ty + i];
  }
}

static int launch_transpose(const float *in, float *out, int b, int rows, int cols, cudaStream_t st) {
  if (b > 65535) return PDAE_E_UNSUPPORTED;
  const dim3 grid(ceil_div(cols, 32), ceil_div(rows, 32), b);
  if (grid.y > 65535) return PDAE_E_UNSUPPORTED;
  transpose_kernel<<<grid, 256, 0, st>>>(in, out, rows, cols);
  PDAE_RETURN_IF_LAUNCH_FAILED();
  return 0;
}

// one thread per output element; xt is (b, n, c).  out row (b,i,p) = [xt[j] - xt[i], xt[i]].
__global__ void __launch_bounds__(256) graph_feature_kernel(const float *__restrict__ xt, const int64_t *__restrict__ idx,
                                                            int c, int n, int k, long long total,
                                                            float *__restrict__ out) {
  const long long e = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (e >= total) return;
  const int c2 = 2 * c;
  const long long row = e / c2;  // (b*n + i)*k + p
  const int col = static_cast<int>(e - row * c2);
  const long long bi = row / k;  // b*n + i
  const long long bb = bi / n;
  const int ch = col < c ? col : col - c;
  const float ctr = __ldg(xt + bi * c + ch);
  float v = ctr;
  if (col < c) {
    const long long j = __ldg(idx + row);
    v = __fsub_rn(__ldg(xt + (bb * n + j) * c + ch), ctr);
  }
  out[e] = v;
}

// vectorised variant (c % 4 == 0, fewer than 2^31 float4 outputs): one thread per float4 of the output, 32-bit
// index arithmetic, 128-bit loads of the transposed rows and 128-bit streaming stores.
__global__ void __launch_bounds__(256) graph_feature_v4_kernel(const float4 *__restrict__ xt4, const int64_t *__restrict__ idx,
                                                               int c4 /* c/4 */, int n, int k, unsigned total4,
                                                               float4 *__restrict__ out4) {
  const unsigned e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= total4) return;
  const unsigned c24 = 2u * c4;
  const unsigned row = e / c24;  // (b*n + i)*k + p
  const unsigned col = e - row * c24;
  const unsigned bi = row / k;   // b*n + i
  const unsigned bb = bi / n;
  const unsigned ch = col < static_cast<unsigned>(c4) ? col : col - c4;
  const float4 ctr = __ldg(xt4 + static_cast<size_t>(bi) * c4 + ch);
  float4 v = ctr;
  if (col < static_cast<unsigned>(c4)) {
    const long long j = __ldg(idx + row);
    const float4 nb = __ldg(xt4 + (static_cast<size_t>(bb) * n + j) * c4 + ch);
    v = make_float4(__fsub_rn(nb.x, ctr.x), __fsub_rn(nb.y, ctr.y), __fsub_rn(nb.z, ctr.z), __fsub_rn(nb.w, ctr.w));
  }
  __stcs(out4 + e, v);
}

// row-per-CTA variant (c % 4 == 0): a CTA owns one point i of one cloud: its k x 2c/4 float4 outputs are contiguous
// (k * 2c * 4 bytes, 20 KB at c = 128), the centre row is read once, and every thread walks the row with a stride of the
// block size -- no per-element divisions (the thread-per-element kernel spends its issue slots on three integer
// divisions per float4 and reaches 60 % of the HBM write peak at c = 128).
template <int THREADS>
__global__ void __launch_bounds__(THREADS) graph_feature_row_kernel(const float4 *__restrict__ xt4, const int64_t *__restrict__ idx,
                                                                    int c4 /* c/4 */, int n, int k, float4 *__restrict__ out4) {
  __shared__ long long nb[64];
  const unsigned bi = blockIdx.x;  // b*n + i
  const unsigned bb = bi / n;
  const int c24 = 2 * c4;
  for (int p = threadIdx.x; p < k; p += THREADS) nb[p] = __ldg(idx + static_cast<size_t>(bi) * k + p);
  __syncthreads();
  const float4 *ctr_row = xt4 + static_cast<size_t>(bi) * c4;
  const float4 *cloud_rows = xt4 + static_cast<size_t>(bb) * n * c4;
  float4 *dst = out4 + static_cast<size_t>(bi) * k * c24;
  const int total = k * c24;
  // thread t handles elements t, t + THREADS, ...: (p, col) advance incrementally
  int p = threadIdx.x / c24, col = threadIdx.x - p * c24;
  const int dp = THREADS / c24, dcol = THREADS - dp * c24;
  for (int e = threadIdx.x; e < total; e += THREADS) {
    const int ch = col < c4 ? col : col - c4;
    const float4 ctr = __ldg(ctr_row + ch);
    float4 v = ctr;
    if (col < c4) {
      const float4 q = __ldg(cloud_rows + static_cast<size_t>(nb[p]) * c4 + ch);
      v = make_float4(__fsub_rn(q.x, ctr.x), __fsub_rn(q.y, ctr.y), __fsub_rn(q.z, ctr.z), __fsub_rn(q.w, ctr.w));
    }
    __stcs(dst + e, v);
    p += dp, col += dcol;
    if (col >= c24) col -= c24, ++p;
  }
}

// backward, scatter part: gxt[b, idx, ch] += G[row, ch]          (thread per (row, ch))
__global__ void __launch_bounds__(256) graph_feature_grad_scatter_kernel(const float *__restrict__ gout,
                                                                         const int64_t *__restrict__ idx, int c, int n,
                                                                         int k, long long total,
                                                                         float *__restrict__ gxt) {
  const long long e = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (e >= total) return;
  const long long row = e / c;
  const int ch = static_cast<int>(e - row * c);
  const long long bb = row / (static_cast<long long>(k) * n);
  const long long j = __ldg(idx + row);
  atomicAdd(gxt + (bb * n + j) * c + ch, __ldg(gout + row * 2 * c + ch));
}

// backward, centre part: gxt[b, i, ch] += sum_p (G[.., c+ch] - G[.., ch])   (thread per (b,i,ch))
__global__ void __launch_bounds__(256) graph_feature_grad_center_kernel(const float *__restrict__ gout, int c, int k,
                                                                        long long total, float *__restrict__ gxt) {
  const long long e = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (e >= total) return;
  const long long bi = e / c;
  const int ch = static_cast<int>(e - bi * c);
  const float *g = gout + bi * k * 2 * c;
  float s = 0.f;
  for (int p = 0; p < k; ++p) s += __ldg(g + static_cast<size_t>(p) * 2 * c + c + ch) - __ldg(g + static_cast<size_t>(p) * 2 * c + ch);
  atomicAdd(gxt + e, s);
}

// backward, deterministic: gxt[b, j, ch] = centre term of row j (p ascending), then (+) G[b, i, p, ch] for every edge
// with idx[b][i][p] == j, slot i * k + p ascending (the ordered reverse map of idx)       (thread per (b,j,ch))
__global__ void __launch_bounds__(256) graph_feature_grad_det_kernel(const float *__restrict__ gout, int c, int n, int k,
                                                                     long long total, RevMap map, float *__restrict__ gxt) {
  const long long e = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (e >= total) return;
  const long long bj = e / c;
  const int ch = static_cast<int>(e - bj * c);
  const long long bb = bj / n;
  const int j = static_cast<int>(bj - bb * n);
  const float *g = gout + bj * k * 2 * c;
  float s = 0.f;
  for (int p = 0; p < k; ++p)
    s = __fadd_rn(s, __fsub_rn(__ldg(g + static_cast<size_t>(p) * 2 * c + c + ch), __ldg(g + static_cast<size_t>(p) * 2 * c + ch)));
  const int *rp = map.ptr + bb * (n + 1);
  const int *rs = map.slot + bb * n * k;
  const float *gc = gout + bb * n * k * 2 * c + ch;
  const int lo = __ldg(rp + j), hi = __ldg(rp + j + 1);
  for (int q = lo; q < hi; ++q) s = __fadd_rn(s, __ldg(gc + static_cast<size_t>(__ldg(rs + q)) * 2 * c));
  gxt[e] = s;
}

// backward, fused and vectorised (c % 4 == 0): one thread per (point, 4 channels) walks its k neighbour rows once:
// 128-bit loads of both halves of the row, the centre term accumulated in registers, the neighbour term scattered
// with one 128-bit RED.ADD (atomicAdd on float4, sm_90+) per row.
__global__ void __launch_bounds__(256) graph_feature_grad_v4_kernel(const float4 *__restrict__ gout4, const int64_t *__restrict__ idx,
                                                                    int c4, int n, int k, unsigned total,
                                                                    float4 *__restrict__ gxt4) {
  const unsigned e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= total) return;
  const unsigned bi = e / c4;           // b*n + i
  const unsigned ch = e - bi * c4;
  const unsigned bb = bi / n;
  const float4 *g = gout4 + static_cast<size_t>(bi) * k * 2 * c4 + ch;
  const int64_t *ip = idx + static_cast<size_t>(bi) * k;
  float4 cs = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int p = 0; p < k; ++p) {
    const float4 g1 = __ldcs(g + static_cast<size_t>(p) * 2 * c4);
    const float4 g2 = __ldcs(g + static_cast<size_t>(p) * 2 * c4 + c4);
    cs.x += g2.x - g1.x; cs.y += g2.y - g1.y; cs.z += g2.z - g1.z; cs.w += g2.w - g1.w;
    const long long j = __ldg(ip + p);
    atomicAdd(gxt4 + (static_cast<size_t>(bb) * n + j) * c4 + ch, g1);
  }
  atomicAdd(gxt4 + static_cast<size_t>(bi) * c4 + ch, cs);
}

// ---- DGCNN kNN in feature space, wide channel counts (C >= 8): register-tiled direct-form distances ----------
// d(i,j) = sum_c (x_jc - x_ic)^2 accumulated with fma in channel order (the repo's canonical definition, bit-exact
// with the oracle); the reference materialises a B x N x N matrix through cuBLAS and runs topk on it
// (models/dgcnn_util.py:7-12).  A CTA owns 64 queries and walks the cloud in 128-point tiles: each thread
// accumulates a 4 x 8 block of pair distances over the channels (packed FADD2/FFMA2: 3 LDS.128 per 32 packed
// ops; operand stages of 16 channels are double-buffered, the next stage's global loads fly during the FMAs),
// the 64 x 128 distance tile is parked in shared memory and each warp feeds its 8 queries' streaming
// warp-select (state and candidate queue per query kept in shared memory between tiles).  FP32 FMA-pipe bound:
// 2 lane-ops per pair and channel; tensor cores would change the rounding and therefore the neighbour order.
constexpr int FT_Q = 64, FT_R = 128, FT_K = 16, FT_THREADS = 256, FT_DPAD = 4;

__global__ void __launch_bounds__(FT_THREADS, 2) feat_knn_tiled_kernel(const float *__restrict__ x, int c, int n, int k,
                                                                       int64_t *__restrict__ idx) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  uint64_t *queues = reinterpret_cast<uint64_t *>(smem_raw);                          // [64 queries][64] candidate queues
  uint64_t *sel_l = queues + FT_Q * 64;                                               // [64 queries][32] sorted lists
  uint64_t *sel_tau = sel_l + FT_Q * 32;                                              // [64 queries]
  int *sel_qn = reinterpret_cast<int *>(sel_tau + FT_Q);                              // [64 queries]
  float *ops0 = reinterpret_cast<float *>(sel_qn + FT_Q);                             // operand stage, 2 buffers
  float *dt = ops0 + 2 * FT_K * (FT_Q + FT_R);                                        // [FT_Q][FT_R + FT_DPAD]
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int ty = tid >> 4, tx = tid & 15;  // 16 x 16 threads: 4 queries x (4 + 4) references each
  const int cloud = blockIdx.y;
  const int q0 = blockIdx.x * FT_Q;
  const float *__restrict__ X = x + static_cast<size_t>(cloud) * c * n;
  const float INF = __int_as_float(0x7f800000);
  const int klane = k - 1;
  constexpr int LD = FT_K * (FT_Q + FT_R) / FT_THREADS;  // floats staged per thread per stage (12)

  // per-query selection state lives in shared memory between tiles so that the selection code exists once
  // (8 unrolled copies of a sort/merge network thrashed the instruction cache: 'no instruction' was the top stall)
  for (int e = tid; e < FT_Q * 32; e += FT_THREADS) sel_l[e] = KEY_INF;
  for (int e = tid; e < FT_Q; e += FT_THREADS) { sel_tau[e] = KEY_INF; sel_qn[e] = 0; }

  const int nst = (c + FT_K - 1) / FT_K;              // channel stages per reference tile
  const int ntiles = (n + FT_R - 1) / FT_R;
  const int total = nst * ntiles;
  float pre[LD];
  // staging map (compile-time per element i, e = tid + i*256): i < 4 -> query operand, channel (tid>>6) + 4i, column
  // tid & 63; i >= 4 -> reference operand, channel (tid>>7) + 2(i-4), column tid & 127.  Everything that does not
  // depend on the stage is hoisted into two per-thread base pointers and two predicates.
  static_assert(FT_K * FT_Q == 4 * FT_THREADS && FT_K * FT_R == 8 * FT_THREADS && FT_Q == 64 && FT_R == 128, "staging map");
  const float *__restrict__ pq = X + static_cast<size_t>(tid >> 6) * n + q0 + (tid & 63);
  const float *__restrict__ pr = X + static_cast<size_t>(tid >> 7) * n + (tid & 127);
  const bool q_ok = q0 + (tid & 63) < n;
  auto fetch = [&](int st) {
    const int tile_i = st / nst;
    const int r0 = tile_i * FT_R, c0 = (st - tile_i * nst) * FT_K;
    const int kc = c - c0;  // channels left (>= 1); rows >= kc of the stage are zero-filled
    const bool r_ok = r0 + (tid & 127) < n;
    const float *bq = pq + static_cast<size_t>(c0) * n;
    const float *br = pr + static_cast<size_t>(c0) * n + r0;
#pragma unroll
    for (int i = 0; i < 4; ++i)
      pre[i] = (q_ok && (tid >> 6) + 4 * i < kc) ? __ldg(bq + static_cast<size_t>(4 * i) * n) : 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i)
      pre[4 + i] = (r_ok && (tid >> 7) + 2 * i < kc) ? __ldg(br + static_cast<size_t>(2 * i) * n) : 0.f;
  };
  auto stash = [&](int buf) {
    float *dst = ops0 + buf * FT_K * (FT_Q + FT_R);
#pragma unroll
    for (int i = 0; i < LD; ++i) dst[tid + i * FT_THREADS] = pre[i];
  };

  fetch(0);
  stash(0);
  __syncthreads();
  float2 acc[4][4];
  for (int st = 0; st < total; ++st) {
    const int tile_i = st / nst, si = st - tile_i * nst;
    const int r0 = tile_i * FT_R, c0 = si * FT_K;
    if (si == 0) {
#pragma unroll
      for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b) acc[a][b] = make_float2(0.f, 0.f);
    }
    if (st + 1 < total) fetch(st + 1);  // global loads of the next stage fly during this stage's FMAs
    const float *qs = ops0 + (st & 1) * FT_K * (FT_Q + FT_R);
    const float *rs = qs + FT_K * FT_Q;
    const int kc = (c - c0) < FT_K ? (c - c0) : FT_K;
#pragma unroll 4
    for (int cc = 0; cc < kc; ++cc) {
      const float4 qv = *reinterpret_cast<const float4 *>(qs + cc * FT_Q + ty * 4);
      const float4 ra = *reinterpret_cast<const float4 *>(rs + cc * FT_R + tx * 4);
      const float4 rb = *reinterpret_cast<const float4 *>(rs + cc * FT_R + 64 + tx * 4);
      const float2 rp[4] = {make_float2(ra.x, ra.y), make_float2(ra.z, ra.w), make_float2(rb.x, rb.y), make_float2(rb.z, rb.w)};
      const float qq[4] = {qv.x, qv.y, qv.z, qv.w};
#pragma unroll
      for (int a = 0; a < 4; ++a) {
        const float2 q2 = make_float2(qq[a], qq[a]);
#pragma unroll
        for (int b = 0; b < 4; ++b) {
          const float2 t = sub2(rp[b], q2);
          acc[a][b] = fma2(t, t, acc[a][b]);
        }
      }
    }
    if (st + 1 < total) stash((st + 1) & 1);
    if (si == nst - 1) {
      // all channels of this reference tile done: park the 64 x 128 distances (references 4tx..4tx+3 and 64+4tx..)
#pragma unroll
      for (int a = 0; a < 4; ++a) {
        float *row = dt + (ty * 4 + a) * (FT_R + FT_DPAD);
        *reinterpret_cast<float4 *>(row + tx * 4) = make_float4(acc[a][0].x, acc[a][0].y, acc[a][1].x, acc[a][1].y);
        *reinterpret_cast<float4 *>(row + 64 + tx * 4) = make_float4(acc[a][2].x, acc[a][2].y, acc[a][3].x, acc[a][3].y);
      }
    }
    __syncthreads();
    if (si == nst - 1) {
      // ---- selection: warp w serves queries 8w .. 8w+7 of the tile (dt is rewritten only after >= 1 more barrier)
      // Streaming warp-select per query; its state (sorted list, threshold, queue fill) lives in shared memory
      // between tiles so the selection code exists once.  (Measured alternatives, both slower on B200: rank
      // insertion per candidate with an always-exact threshold, 0.70 ms; parallel threshold scan + per-lane
      // insertion sort by two rotating warps, 0.88 ms; this version 0.65 ms at C=64, N=2048, B=16.)
#pragma unroll 1
      for (int i = 0; i < 8; ++i) {
        const int ql = warp * 8 + i;
        if (q0 + ql >= n) continue;
        const float *row = dt + ql * (FT_R + FT_DPAD);
        const uint64_t tau_in = sel_tau[ql];
        uint64_t key[4];
        bool anyp = false;
#pragma unroll
        for (int h = 0; h < 4; ++h) {
          const int r = h * 32 + lane;
          const bool in = r0 + r < n;
          key[h] = in ? pack_key(row[r], static_cast<uint32_t>(r0 + r)) : KEY_INF;
          anyp |= key[h] < tau_in;
        }
        if (!__any_sync(0xffffffffu, anyp)) continue;
        WarpSelect<1> s;
        s.L[0] = sel_l[ql * 32 + lane];
        s.tau = tau_in;
        s.qn = sel_qn[ql];
        uint64_t *queue = queues + ql * 64;
#pragma unroll 1
        for (int h = 0; h < 4; ++h) {
          const uint64_t kk = h == 0 ? key[0] : (h == 1 ? key[1] : (h == 2 ? key[2] : key[3]));
          s.offer(kk < s.tau, kk, queue, lane, 0, klane);  // tau may have dropped after a flush in this loop
        }
        sel_l[ql * 32 + lane] = s.L[0];
        if (lane == 0) { sel_tau[ql] = s.tau; sel_qn[ql] = s.qn; }
        __syncwarp();
      }
      if (nst == 1) __syncthreads();  // single-stage tiles: the next stage's park would otherwise race the selection
    }
  }
  // ---- epilogue ----------------------------------------------------------------------------------------------------
#pragma unroll 1
  for (int i = 0; i < 8; ++i) {
    const int ql = warp * 8 + i, qg = q0 + ql;
    if (qg < n) {
      WarpSelect<1> s;
      s.L[0] = sel_l[ql * 32 + lane];
      s.tau = sel_tau[ql];
      s.qn = sel_qn[ql];
      s.finish(queues + ql * 64, lane);
      if (lane < k) idx[(static_cast<size_t>(cloud) * n + qg) * k + lane] = static_cast<int64_t>(static_cast<uint32_t>(s.L[0]));
    }
  }
}

// ---- the same search through a materialised distance matrix (default when a workspace is given) -------------------------
// ncu on the fused kernel above (C = 64, N = 2048, B = 16): 364 M warp instructions of which only 134 M are the packed
// FMA work -- the streaming selection (about k ln(N/k) + k insertions per query, a ballot / queue append per candidate,
// a bitonic flush every 32) costs more issue slots than the distances.  On B200 writing the B x N x N fp32 matrix the
// reference also materialises is cheap (268 MB at that shape: ~40 us each way at the measured 6.5 TB/s), so the distances
// go to global memory and a warp per query selects from its stored row.
// The search is a SELF-kNN: d(i,j) and d(j,i) are the same bits (the operands of every subtraction only change sign), so
// each unordered pair is evaluated once.  A CTA owns 64 queries and walks only the 128-point reference tiles from its own
// diagonal tile on; besides its rows it stores the TRANSPOSED block D[r][q] (for every reference four consecutive
// queries = one 128-bit store; the two 16-row halves of a warp fill whole 32-byte sectors), which is exactly the part of
// the lower triangle no CTA computes directly.  Executed FMA work: (ntiles + 1) / (2 ntiles) of the full matrix.
// A CTA does not see its rows' lower-triangle distances, so the selection kernel takes its threshold tau0 from the stored
// row itself: 64 segment minima per query (one FMNMX3 per two values), k-th smallest by one 32-bit bitonic sort -- the
// pass 1 of knn4.cu -- then the row is read again (L1 / L2 hit), the ~1.2 k points with d <= tau0 go to lane-private
// lists (predicated stores), are compacted, sorted as 64-bit (distance, index) keys and the first k written.  Overflow
// (mass ties) -> exact streaming warp-select over the stored row.  Same distances, same (distance, lower index first)
// order: bit-identical to the fused kernel and the oracle.
constexpr int FS_LC = 8;  // lane-private candidate slots of the selection kernel

__global__ void __launch_bounds__(FT_THREADS, 2) feat_dist_sym_kernel(const float *__restrict__ x, int c, int n,
                                                                      float *__restrict__ dmat /*(b, n, n)*/) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float *ops0 = reinterpret_cast<float *>(smem_raw);  // operand stage, 2 buffers
  const int tid = threadIdx.x;
  const int ty = tid >> 4, tx = tid & 15;  // 16 x 16 threads: 4 queries x (4 + 4) references each
  // grid (clouds, query blocks): the dispatcher hands out blockIdx.x fastest, so ALL clouds' heaviest query blocks (block 0
  // walks every tile, the last block one) start first and the light ones fill the tail -- longest-processing-time order
  const int cloud = blockIdx.x;
  const int q0 = blockIdx.y * FT_Q;
  const float *__restrict__ X = x + static_cast<size_t>(cloud) * c * n;
  float *__restrict__ D = dmat + static_cast<size_t>(cloud) * n * n;
  constexpr int LD = FT_K * (FT_Q + FT_R) / FT_THREADS;
  const int nst = (c + FT_K - 1) / FT_K;
  const int ntiles = (n + FT_R - 1) / FT_R;
  const int t_first = q0 / FT_R;  // the diagonal tile of this query block
  const int total = nst * (ntiles - t_first);
  float pre[LD];
  const float *__restrict__ pq = X + static_cast<size_t>(tid >> 6) * n + q0 + (tid & 63);
  const float *__restrict__ pr = X + static_cast<size_t>(tid >> 7) * n + (tid & 127);
  const bool q_ok = q0 + (tid & 63) < n;
  auto fetch = [&](int st) {
    const int tile_i = t_first + st / nst;
    const int r0 = tile_i * FT_R, c0 = (st % nst) * FT_K;
    const int kc = c - c0;
    const bool r_ok = r0 + (tid & 127) < n;
    const float *bq = pq + static_cast<size_t>(c0) * n;
    const float *br = pr + static_cast<size_t>(c0) * n + r0;
#pragma unroll
    for (int i = 0; i < 4; ++i)
      pre[i] = (q_ok && (tid >> 6) + 4 * i < kc) ? __ldg(bq + static_cast<size_t>(4 * i) * n) : 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i)
      pre[4 + i] = (r_ok && (tid >> 7) + 2 * i < kc) ? __ldg(br + static_cast<size_t>(2 * i) * n) : 0.f;
  };
  auto stash = [&](int buf) {
    float *dst = ops0 + buf * FT_K * (FT_Q + FT_R);
#pragma unroll
    for (int i = 0; i < LD; ++i) dst[tid + i * FT_THREADS] = pre[i];
  };
  const bool vec = (n & 3) == 0;

  fetch(0);
  stash(0);
  __syncthreads();
  float2 acc[4][4];
  for (int st = 0; st < total; ++st) {
    const int tile_i = t_first + st / nst, si = st % nst;
    const int r0 = tile_i * FT_R, c0 = si * FT_K;
    if (si == 0) {
#pragma unroll
      for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b) acc[a][b] = make_float2(0.f, 0.f);
    }
    if (st + 1 < total) fetch(st + 1);
    const float *qs = ops0 + (st & 1) * FT_K * (FT_Q + FT_R);
    const float *rs = qs + FT_K * FT_Q;
    const int kc = (c - c0) < FT_K ? (c - c0) : FT_K;
#pragma unroll 4
    for (int cc = 0; cc < kc; ++cc) {
      const float4 qv = *reinterpret_cast<const float4 *>(qs + cc * FT_Q + ty * 4);
      const float4 ra = *reinterpret_cast<const float4 *>(rs + cc * FT_R + tx * 4);
      const float4 rb = *reinterpret_cast<const float4 *>(rs + cc * FT_R + 64 + tx * 4);
      const float2 rp[4] = {make_float2(ra.x, ra.y), make_float2(ra.z, ra.w), make_float2(rb.x, rb.y), make_float2(rb.z, rb.w)};
      const float qq[4] = {qv.x, qv.y, qv.z, qv.w};
#pragma unroll
      for (int a = 0; a < 4; ++a) {
        const float2 q2 = make_float2(qq[a], qq[a]);
#pragma unroll
        for (int b = 0; b < 4; ++b) {
          const float2 t = sub2(rp[b], q2);
          acc[a][b] = fma2(t, t, acc[a][b]);
        }
      }
    }
    if (st + 1 < total) stash((st + 1) & 1);
    if (si == nst - 1) {
      const int ra0 = r0 + tx * 4, rb0 = r0 + 64 + tx * 4;  // first reference of each half
      float v[4][8];
#pragma unroll
      for (int a = 0; a < 4; ++a) {
        v[a][0] = acc[a][0].x, v[a][1] = acc[a][0].y, v[a][2] = acc[a][1].x, v[a][3] = acc[a][1].y;
        v[a][4] = acc[a][2].x, v[a][5] = acc[a][2].y, v[a][6] = acc[a][3].x, v[a][7] = acc[a][3].y;
      }
      // rows of this query block
#pragma unroll
      for (int a = 0; a < 4; ++a) {
        const int qg = q0 + ty * 4 + a;
        if (qg < n) {
          float *row = D + static_cast<size_t>(qg) * n;
          if (vec) {
            if (ra0 < n) *reinterpret_cast<float4 *>(row + ra0) = make_float4(v[a][0], v[a][1], v[a][2], v[a][3]);
            if (rb0 < n) *reinterpret_cast<float4 *>(row + rb0) = make_float4(v[a][4], v[a][5], v[a][6], v[a][7]);
          } else {
#pragma unroll
            for (int e = 0; e < 8; ++e) {
              const int r = e < 4 ? ra0 + e : rb0 + e - 4;
              if (r < n) row[r] = v[a][e];
            }
          }
        }
      }
      // the transposed block: rows = this tile's references, columns = this block's queries (tiles above the diagonal)
      if (tile_i > t_first) {
        const int qa = q0 + ty * 4;
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          const int r = e < 4 ? ra0 + e : rb0 + e - 4;
          if (r < n) {
            float *col = D + static_cast<size_t>(r) * n + qa;
            if (vec && qa + 3 < n) {
              *reinterpret_cast<float4 *>(col) = make_float4(v[0][e], v[1][e], v[2][e], v[3][e]);
            } else {
#pragma unroll
              for (int a = 0; a < 4; ++a)
                if (qa + a < n) col[a] = v[a][e];
            }
          }
        }
      }
    }
    __syncthreads();
  }
}

__global__ void __launch_bounds__(256) feat_select2_kernel(const float *__restrict__ dmat, int n, int k, int64_t *__restrict__ idx) {
  __shared__ uint64_t queue_all[8][64];
  __shared__ uint64_t lq_all[8][FS_LC * 32];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int q = blockIdx.x * 8 + warp;
  const size_t cloud = blockIdx.y;
  if (q >= n) return;
  const float *__restrict__ row = dmat + (cloud * n + q) * n;
  uint64_t *queue = queue_all[warp], *lq = lq_all[warp];
  const float INF = __int_as_float(0x7f800000);
  const bool vec = (n & 3) == 0;
  // ---- pass 1: 64 segment minima (2 per lane) -> tau0 = their k-th smallest (k <= 32) ---------------------------------
  float ma = INF, mb = INF;
  if (vec) {
    for (int j0 = 0; j0 < n; j0 += 128) {
      const int j = j0 + 4 * lane;
      if (j < n) {
        const float4 d = __ldg(reinterpret_cast<const float4 *>(row + j));
        ma = min3(ma, d.x, d.y);
        mb = min3(mb, d.z, d.w);
      }
    }
  } else {
    for (int j = lane; j < n; j += 64) ma = fminf(ma, __ldg(row + j));
    for (int j = lane + 32; j < n; j += 64) mb = fminf(mb, __ldg(row + j));
  }
  uint32_t sv[2] = {__float_as_uint(ma), __float_as_uint(mb)};  // distances are >= 0: bit patterns order like values
  warp_sort_u32<2>(sv, lane, warp_sort_dir_mask(lane));
  const float tau0 = __uint_as_float(__shfl_sync(0xffffffffu, sv[0], k - 1));
  // ---- pass 2: every point with d <= tau0 -> lane-private lists -> exact order ---------------------------------------------
  const bool degenerate = !(tau0 < INF);
  int cnt = 0;
  if (vec) {
    for (int j0 = 0; j0 < n; j0 += 128) {
      const int j = j0 + 4 * lane;
      if (j < n) {
        const float4 d = __ldg(reinterpret_cast<const float4 *>(row + j));
        if (min3(d.x, d.y, fminf(d.z, d.w)) <= tau0) {
          const float v[4] = {d.x, d.y, d.z, d.w};
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const bool cnd = v[e] <= tau0;
            if (cnd && cnt < FS_LC) lq[cnt * 32 + lane] = pack_key(v[e], static_cast<uint32_t>(j + e));
            cnt += cnd;
          }
        }
      }
    }
  } else {
    for (int j = lane; j < n; j += 32) {
      const float v = __ldg(row + j);
      const bool cnd = v <= tau0;
      if (cnd && cnt < FS_LC) lq[cnt * 32 + lane] = pack_key(v, static_cast<uint32_t>(j));
      cnt += cnd;
    }
  }
  if (degenerate) cnt = FS_LC + 1;
  int incl = cnt;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int t = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += t;
  }
  const int totalc = __shfl_sync(0xffffffffu, incl, 31);
  const bool overflow = __any_sync(0xffffffffu, cnt > FS_LC) || totalc > 64;
  uint64_t keys[2];
  if (!overflow) {
    const int off = incl - cnt;
    for (int i = 0; i < cnt; ++i) queue[off + i] = lq[i * 32 + lane];
    __syncwarp();
#pragma unroll
    for (int e = 0; e < 2; ++e) keys[e] = (e * 32 + lane) < totalc ? queue[e * 32 + lane] : KEY_INF;
    __syncwarp();
    warp_sort_multi<2>(keys, lane);
  } else {  // exact fallback: streaming warp-select over the stored row
    WarpSelect<1> sel;
    sel.init();
    for (int j0 = 0; j0 < n; j0 += 32) {
      const int j = j0 + lane;
      const bool in = j < n;
      const uint64_t key = in ? pack_key(__ldg(row + j), static_cast<uint32_t>(j)) : KEY_INF;
      sel.offer(in && key < sel.tau, key, queue, lane, 0, k - 1);
    }
    sel.finish(queue, lane);
    keys[0] = sel.L[0];
    keys[1] = KEY_INF;
  }
  if (lane < k) idx[(cloud * n + q) * k + lane] = static_cast<int64_t>(static_cast<uint32_t>(keys[0]));
}

static size_t feat_matrix_bytes_per_cloud(int n) { return (static_cast<size_t>(n) * n + n) * sizeof(float); }

static int launch_feat_knn_matrix(const float *x, int b, int c, int n, int k, int64_t *idx, void *workspace,
                                  size_t workspace_bytes, cudaStream_t st) {
  const size_t per = feat_matrix_bytes_per_cloud(n);
  long long chunk = static_cast<long long>(workspace_bytes / per);
  if (chunk < 1) return PDAE_E_WORKSPACE;
  if (chunk > 65535) chunk = 65535;
  const size_t smem = 2 * static_cast<size_t>(FT_K) * (FT_Q + FT_R) * sizeof(float);
  for (long long b0 = 0; b0 < b; b0 += chunk) {
    const int nb = static_cast<int>(b - b0 < chunk ? b - b0 : chunk);
    float *dmat = static_cast<float *>(workspace);
    const int nqb = ceil_div(n, FT_Q);
    if (nqb > 65535) return PDAE_E_UNSUPPORTED;
    feat_dist_sym_kernel<<<dim3(nb, nqb), FT_THREADS, smem, st>>>(x + static_cast<size_t>(b0) * c * n, c, n, dmat);
    PDAE_RETURN_IF_LAUNCH_FAILED();
    feat_select2_kernel<<<dim3(ceil_div(n, 8), nb), 256, 0, st>>>(dmat, n, k, idx + static_cast<size_t>(b0) * n * k);
    PDAE_RETURN_IF_LAUNCH_FAILED();
  }
  return 0;
}

static int launch_feat_knn_tiled(const float *x, int b, int c, int n, int k, int64_t *idx, cudaStream_t st) {
  if (b > 65535) return PDAE_E_UNSUPPORTED;
  const size_t smem = (static_cast<size_t>(FT_Q) * 64 + FT_Q * 32 + FT_Q) * sizeof(uint64_t) + FT_Q * sizeof(int) +
                      (2 * static_cast<size_t>(FT_K) * (FT_Q + FT_R) + static_cast<size_t>(FT_Q) * (FT_R + FT_DPAD)) * sizeof(float);
  static_assert(FT_K * (FT_Q + FT_R) % FT_THREADS == 0, "operand stage must split evenly over the CTA");
  PDAE_CUDA_TRY(cudaFuncSetAttribute(feat_knn_tiled_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
  const dim3 grid(ceil_div(n, FT_Q), b);
  feat_knn_tiled_kernel<<<grid, FT_THREADS, smem, st>>>(x, c, n, k, idx);
  PDAE_RETURN_IF_LAUNCH_FAILED();
  return 0;
}

}  // namespace pdae

using namespace pdae;

extern "C" int pdae_feat_knn_f32(const float *x, int b, int c, int n, int k, int64_t *idx, pdae_stream_t stream) {
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (b > 0 && n > 0 && x && idx && c >= 8 && k >= 1 && k <= 32 && k <= n) return launch_feat_knn_tiled(x, b, c, n, k, idx, st);
  return feat_knn_generic(x, b, c, n, k, idx, st);  // c == 3 -> knn4 planar fast path; other shapes -> streaming warp-select
}

// workspace of the matrix path: whole clouds' worth of (n x n distances + n spare floats), capped at 1 GiB (the host
// function walks the batch in chunks); 0 when the shape takes another path or one cloud alone exceeds the cap.
extern "C" size_t pdae_feat_knn_workspace_bytes(int b, int c, int n, int k) {
  if (b <= 0 || n <= 0 || c < 8 || k < 1 || k > 32 || k > n) return 0;
  const size_t per = feat_matrix_bytes_per_cloud(n), cap = static_cast<size_t>(1) << 30;
  if (per > cap) return 0;
  size_t clouds = cap / per;
  if (clouds > static_cast<size_t>(b)) clouds = static_cast<size_t>(b);
  return clouds * per;
}

extern "C" int pdae_feat_knn_ws_f32(const float *x, int b, int c, int n, int k, int64_t *idx, void *workspace,
                                    size_t workspace_bytes, pdae_stream_t stream) {
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (b > 0 && n > 0 && x && idx && c >= 8 && k >= 1 && k <= 32 && k <= n && workspace &&
      workspace_bytes >= feat_matrix_bytes_per_cloud(n))
    return launch_feat_knn_matrix(x, b, c, n, k, idx, workspace, workspace_bytes, st);
  return pdae_feat_knn_f32(x, b, c, n, k, idx, stream);
}

extern "C" size_t pdae_graph_feature_workspace_bytes(int b, int c, int n) {
  if (b <= 0 || c <= 0 || n <= 0) return 0;
  return static_cast<size_t>(b) * c * n * sizeof(float);
}

extern "C" int pdae_graph_feature_f32(const float *x, const int64_t *idx, int b, int c, int n, int k, float *out,
                                      void *workspace, size_t workspace_bytes, pdae_stream_t stream) {
  if (b < 0 || c <= 0 || n < 0 || k < 0) return PDAE_E_INVALID;
  const long long total = static_cast<long long>(b) * n * k * 2 * c;
  if (total == 0) return 0;
  if (!x || !idx || !out) return PDAE_E_INVALID;
  if (!workspace || workspace_bytes < pdae_graph_feature_workspace_bytes(b, c, n)) return PDAE_E_WORKSPACE;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  float *xt = static_cast<float *>(workspace);
  const int rc = launch_transpose(x, xt, b, c, n, st);  // (b,c,n) -> (b,n,c)
  if (rc) return rc;
  if ((c & 3) == 0 && k <= 64 && c >= 16 && static_cast<long long>(b) * n < 0x7fffffffLL && getenv("PDAE_GRAPHFEAT_ELEMENTWISE") == nullptr) {
    graph_feature_row_kernel<256><<<static_cast<unsigned>(static_cast<long long>(b) * n), 256, 0, st>>>(
        reinterpret_cast<const float4 *>(xt), idx, c / 4, n, k, reinterpret_cast<float4 *>(out));
    PDAE_RETURN_IF_LAUNCH_FAILED();
    return 0;
  }
  if ((c & 3) == 0 && total / 4 < 0x7fffffffLL) {
    const unsigned total4 = static_cast<unsigned>(total / 4);
    graph_feature_v4_kernel<<<(total4 + 255) / 256, 256, 0, st>>>(reinterpret_cast<const float4 *>(xt), idx, c / 4, n, k, total4,
                                                               reinterpret_cast<float4 *>(out));
    PDAE_RETURN_IF_LAUNCH_FAILED();
    return 0;
  }
  const long long grid = (total + 255) / 256;
  if (grid > 0x7fffffffLL) return PDAE_E_UNSUPPORTED;
  graph_feature_kernel<<<static_cast<unsigned>(grid), 256, 0, st>>>(xt, idx, c, n, k, total, out);
  PDAE_RETURN_IF_LAUNCH_FAILED();
  return 0;
}

extern "C" int pdae_graph_feature_grad_f32(const float *gout, const int64_t *idx, int b, int c, int n, int k,
                                           float *gx, void *workspace, size_t workspace_bytes, pdae_stream_t stream) {
  if (b < 0 || c <= 0 || n < 0 || k < 0) return PDAE_E_INVALID;
  const size_t gsz = static_cast<size_t>(b) * c * n;
  if (gsz == 0) return 0;
  if (!gx) return PDAE_E_INVALID;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (k == 0) {
    PDAE_CUDA_TRY(cudaMemsetAsync(gx, 0, gsz * sizeof(float), st));
    return 0;
  }
  if (!gout || !idx) return PDAE_E_INVALID;
  if (!workspace || workspace_bytes < pdae_graph_feature_workspace_bytes(b, c, n)) return PDAE_E_WORKSPACE;
  float *gxt = static_cast<float *>(workspace);
  PDAE_CUDA_TRY(cudaMemsetAsync(gxt, 0, gsz * sizeof(float), st));
  const long long tc = static_cast<long long>(b) * n * c;
  const long long ts = tc * k;
  if ((c & 3) == 0 && tc / 4 < 0x7fffffffLL) {
    const unsigned total = static_cast<unsigned>(tc / 4);
    graph_feature_grad_v4_kernel<<<(total + 255) / 256, 256, 0, st>>>(reinterpret_cast<const float4 *>(gout), idx, c / 4, n, k, total,
                                                                    reinterpret_cast<float4 *>(gxt));
    PDAE_RETURN_IF_LAUNCH_FAILED();
    return launch_transpose(gxt, gx, b, n, c, st);  // (b,n,c) -> (b,c,n)
  }
  if ((ts + 255) / 256 > 0x7fffffffLL) return PDAE_E_UNSUPPORTED;
  graph_feature_grad_center_kernel<<<static_cast<unsigned>((tc + 255) / 256), 256, 0, st>>>(gout, c, k, tc, gxt);
  PDAE_RETURN_IF_LAUNCH_FAILED();
  graph_feature_grad_scatter_kernel<<<static_cast<unsigned>((ts + 255) / 256), 256, 0, st>>>(gout, idx, c, n, k, ts,
                                                                                          gxt);
  PDAE_RETURN_IF_LAUNCH_FAILED();
  return launch_transpose(gxt, gx, b, n, c, st);  // (b,n,c) -> (b,c,n)
}

extern "C" size_t pdae_graph_feature_grad_det_workspace_bytes(int b, int c, int n, int k) {
  if (b <= 0 || c <= 0 || n <= 0 || k < 0 || static_cast<long long>(n) * k > 0x7fffffffLL) return 0;
  return align256(rev_map_bytes(b, n * k, n)) + static_cast<size_t>(b) * c * n * sizeof(float);
}

extern "C" int pdae_graph_feature_grad_det_f32(const float *gout, const int64_t *idx, int b, int c, int n, int k, float *gx,
                                               void *workspace, size_t workspace_bytes, pdae_stream_t stream) {
  if (b < 0 || c <= 0 || n < 0 || k < 0) return PDAE_E_INVALID;
  const size_t gsz = static_cast<size_t>(b) * c * n;
  if (gsz == 0) return 0;
  if (!gx) return PDAE_E_INVALID;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (k == 0) {
    PDAE_CUDA_TRY(cudaMemsetAsync(gx, 0, gsz * sizeof(float), st));
    return 0;
  }
  if (!gout || !idx || static_cast<long long>(n) * k > 0x7fffffffLL) return PDAE_E_INVALID;
  if (!workspace || workspace_bytes < pdae_graph_feature_grad_det_workspace_bytes(b, c, n, k)) return PDAE_E_WORKSPACE;
  RevMap map;
  int rc = rev_map_build(idx, b, n * k, n, workspace, &map, st);
  if (rc) return rc;
  float *gxt = reinterpret_cast<float *>(static_cast<unsigned char *>(workspace) + align256(rev_map_bytes(b, n * k, n)));
  const long long tc = static_cast<long long>(b) * n * c;
  if ((tc + 255) / 256 > 0x7fffffffLL) return PDAE_E_UNSUPPORTED;
  graph_feature_grad_det_kernel<<<static_cast<unsigned>((tc + 255) / 256), 256, 0, st>>>(gout, c, n, k, tc, map, gxt);
  PDAE_RETURN_IF_LAUNCH_FAILED();
  return launch_transpose(gxt, gx, b, n, c, st);  // (b,n,c) -> (b,c,n)
}
