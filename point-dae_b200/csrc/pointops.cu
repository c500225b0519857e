// pointops.cu -- variable-size clouds packed in one batch: segment FPS and segment kNN (the reference's
// extensions/pointops: furthestsampling_cuda, knnquery_cuda).
//
// Layout: xyz (N_total, 3) holds the clouds back to back; offset[s] is the cumulative end of cloud s, so cloud s is
// [offset[s-1], offset[s]) with offset[-1] = 0.  new_offset does the same for the samples / queries.  Offsets are read
// on the device only (no host synchronisation) and are clamped into the tensors, so no value makes an access leave them.
// Every index written is global (into the packed tensor).  Semantics and rounding: include/pointdae_b200.h.
//
// FPS: one CTA per segment.  The tie rule of the reference's block tree (bit-reversed slot (k - start) mod bs first,
// then the smaller k) is the rank of fps_rank.cuh taken relative to the segment start, with bs from `n` (cap 1024).
// Every CTA width is a multiple of bs, so ascending k inside a thread is ascending rank and the in-thread scan keeps the
// reference's strict `>`.  Segments up to T*P points keep (x, y, z, running minimum) in registers; larger ones -- or any
// segment when `n` asks for more than the register form holds -- run the same loop with the running minima in global
// memory (the caller's tmp, or the workspace).
//
// kNN: a one-CTA pre-pass turns new_offset into a table of 8-query blocks that never straddle a segment; the main
// kernel's CTAs beyond the table exit.  Each warp owns one query and streams its segment through shared-memory tiles
// with the warp-select of knn_select.cuh: keys (d^2 bits << 32 | global index), so the kept set and its order are the
// exact (d^2, index) order whatever the grid.  No atomics anywhere; results do not depend on launch shape or stream.
#include "fps_rank.cuh"
#include "knn_select.cuh"

#include <math.h>

namespace pdae {

constexpr float SEG_INIT = 1e10f;  // the reference's tmp fill and heap initial distance
constexpr int SEG_FPS_T = 1024;    // widest CTA: a multiple of every bs <= 1024
constexpr int SEG_REG_MAX_N = SEG_FPS_T * 8;
constexpr int SEG_KNN_WARPS = 8;   // queries per kNN block (one per warp)
constexpr int SEG_KNN_TILE = 2048; // points per shared-memory tile
constexpr int SEG_KNN_MAX_K = 100; // the reference's fixed per-thread heap

// [lo, hi) of segment s in a tensor of `total` rows, clamped into it
__device__ __forceinline__ void seg_bounds(const int *__restrict__ off, int s, int total, int &lo, int &hi) {
  int a = s ? __ldg(off + s - 1) : 0, e = __ldg(off + s);
  a = min(max(a, 0), total);
  e = min(max(e, a), total);
  lo = a;
  hi = e;
}

// value -> monotone unsigned over every value a thread can report (> -1, or the "no point" -1); -0 folds into +0,
// which the reference's `>` does not distinguish either
__device__ __forceinline__ unsigned seg_val_key(float v) {
  const unsigned u = __float_as_uint(__fadd_rn(v, 0.0f));
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

struct SegFpsArgs {
  const float *xyz;
  const int *offset, *new_offset;
  float *tmp;  // caller's running minima (N_total) or null
  float *ws;   // N_total floats, used when tmp is null and a segment takes the global loop
  int *idx;
  int n_total, m_total, lg_bs;
};

// the running minima in global memory: any segment size, same arithmetic and tie rule as the register form.
// A thread only ever touches its own k = tid + i*T, so the minima need no barrier.
template <int T>
__device__ void seg_fps_global(const SegFpsArgs &a, int sn, int cnt, int sm, int cnt_m, uint2 *slots) {
  const int tid = threadIdx.x;
  const float *__restrict__ P = a.xyz + static_cast<size_t>(sn) * 3;
  float *run = (a.tmp ? a.tmp : a.ws) + sn;
  if (!a.tmp)
    for (int k = tid; k < cnt; k += T) run[k] = SEG_INIT;
  int old = 0;
  for (int j = 1; j < cnt_m; ++j) {
    const float ox = __ldg(P + 3 * old), oy = __ldg(P + 3 * old + 1), oz = __ldg(P + 3 * old + 2);
    float best = -1.0f;
    int bk = -1;
    for (int k = tid; k < cnt; k += T) {
      const float d = dist_yxz(__fsub_rn(__ldg(P + 3 * k), ox), __fsub_rn(__ldg(P + 3 * k + 1), oy),
                               __fsub_rn(__ldg(P + 3 * k + 2), oz));
      const float d2 = fminf(d, run[k]);
      run[k] = d2;
      if (d2 > best) {
        best = d2;
        bk = k;
      }
    }
    // a thread without a taken point reports (-1, start) like the reference; rank 0 unranks to the segment start
    const unsigned r = fps_block_argmax<T>(seg_val_key(best), bk >= 0 ? fps_rank(bk, a.lg_bs) : 0u, slots, j);
    old = fps_unrank(r, a.lg_bs);
    if (tid == 0) a.idx[sm + j] = sn + old;
  }
}

// common prologue: segment bounds, empty segments, the first sample.  false: nothing left to do.
template <int T>
__device__ __forceinline__ bool seg_fps_begin(const SegFpsArgs &a, int &sn, int &cnt, int &sm, int &cnt_m) {
  int en, em;
  seg_bounds(a.offset, blockIdx.x, a.n_total, sn, en);
  seg_bounds(a.new_offset, blockIdx.x, a.m_total, sm, em);
  cnt = en - sn;
  cnt_m = em - sm;
  if (cnt_m == 0) return false;
  if (cnt == 0) {  // the reference's tree then returns the start index for every sample
    for (int j = threadIdx.x; j < cnt_m; j += T) a.idx[sm + j] = sn;
    return false;
  }
  if (threadIdx.x == 0) a.idx[sm] = sn;
  return true;
}

template <int T>
__global__ void __launch_bounds__(T) seg_fps_global_kernel(const SegFpsArgs a) {
  __shared__ uint2 slots[2 * 32];
  int sn, cnt, sm, cnt_m;
  if (!seg_fps_begin<T>(a, sn, cnt, sm, cnt_m)) return;
  seg_fps_global<T>(a, sn, cnt, sm, cnt_m, slots);
}

// register form: thread tid holds points k = tid + p*T (k relative to the segment start) in registers; the segment is
// also staged in shared memory so the winner's coordinates are one LDS.128 away.  Padding carries -1, which the
// reference's `d2 > best` (best starting at -1) never takes and fminf never raises.
template <int T, int P>
__global__ void __launch_bounds__(T) seg_fps_reg_kernel(const SegFpsArgs a) {
  __shared__ uint2 slots[2 * 32];
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float4 *sp = reinterpret_cast<float4 *>(smem_raw);  // [T*P]
  int sn, cnt, sm, cnt_m;
  if (!seg_fps_begin<T>(a, sn, cnt, sm, cnt_m)) return;
  if (cnt > T * P) {  // the segment is larger than `n` announced: same results from the global loop
    seg_fps_global<T>(a, sn, cnt, sm, cnt_m, slots);
    return;
  }
  const int tid = threadIdx.x;
  const float *__restrict__ Pt = a.xyz + static_cast<size_t>(sn) * 3;
  float px[P], py[P], pz[P], pt[P];
#pragma unroll
  for (int p = 0; p < P; ++p) {
    const int k = tid + p * T;
    float x = 0.f, y = 0.f, z = 0.f, t = -1.0f;
    if (k < cnt) {
      x = __ldg(Pt + 3 * k);
      y = __ldg(Pt + 3 * k + 1);
      z = __ldg(Pt + 3 * k + 2);
      t = a.tmp ? a.tmp[sn + k] : SEG_INIT;
      sp[k] = make_float4(x, y, z, 0.f);
    }
    px[p] = x; py[p] = y; pz[p] = z; pt[p] = t;
  }
  __syncthreads();
  float4 o = sp[0];
  for (int j = 1; j < cnt_m; ++j) {
    float best = -1.0f;
    int bp = -1;
#pragma unroll
    for (int p = 0; p < P; ++p) {
      const float d = dist_yxz(__fsub_rn(px[p], o.x), __fsub_rn(py[p], o.y), __fsub_rn(pz[p], o.z));
      pt[p] = fminf(d, pt[p]);
      if (pt[p] > best) {
        best = pt[p];
        bp = p;
      }
    }
    const unsigned r = fps_block_argmax<T>(seg_val_key(best), bp >= 0 ? fps_rank(tid + bp * T, a.lg_bs) : 0u, slots, j);
    const int w = fps_unrank(r, a.lg_bs);
    o = sp[w];
    if (tid == 0) a.idx[sm + j] = sn + w;
  }
  if (a.tmp) {
#pragma unroll
    for (int p = 0; p < P; ++p) {
      const int k = tid + p * T;
      if (k < cnt) a.tmp[sn + k] = pt[p];
    }
  }
}

template <int T, int P>
static int launch_seg_fps_reg(const SegFpsArgs &a, int b, cudaStream_t st) {
  const size_t smem = static_cast<size_t>(T) * P * sizeof(float4);
  if (smem > 48 * 1024)
    PDAE_CUDA_TRY(cudaFuncSetAttribute(seg_fps_reg_kernel<T, P>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       static_cast<int>(smem)));
  seg_fps_reg_kernel<T, P><<<b, T, smem, st>>>(a);
  PDAE_RETURN_IF_LAUNCH_FAILED();
  return 0;
}

// ---- kNN -----------------------------------------------------------------------------------------------------------
// inclusive block-wide scan (sum or max) of one int per thread of a 1024-thread CTA; `total` gets the last value
__device__ __forceinline__ int block_scan_incl(int v, int *warp_tot /*[32]*/, int &total, bool is_max) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const int o = __shfl_up_sync(0xffffffffu, v, d);
    if (lane >= d) v = is_max ? max(v, o) : v + o;
  }
  if (lane == 31) warp_tot[warp] = v;
  __syncthreads();
  if (warp == 0) {
    int w = warp_tot[lane];
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const int o = __shfl_up_sync(0xffffffffu, w, d);
      if (lane >= d) w = is_max ? max(w, o) : w + o;
    }
    warp_tot[lane] = w;
  }
  __syncthreads();
  if (warp > 0) v = is_max ? max(v, warp_tot[warp - 1]) : v + warp_tot[warp - 1];
  total = warp_tot[31];
  __syncthreads();
  return v;
}

// one CTA of 1024 threads.  Table entry: points [sn, en) of the segment, queries [p0, p1) (at most SEG_KNN_WARPS).
// Query p belongs to the first segment s with p < new_offset[s] (the reference's
// get_bt_idx), i.e. to [max(new_offset[0..s-1]), new_offset[s]); rows from max(new_offset) up to m get the padding.
__global__ void __launch_bounds__(1024) seg_knn_table_kernel(const int *__restrict__ offset, const int *__restrict__ new_offset,
                                                             int b, int n_total, int m, int nsample, int4 *__restrict__ table,
                                                             int *__restrict__ count, int *__restrict__ idx,
                                                             float *__restrict__ dist2) {
  __shared__ int warp_tot[32];
  __shared__ int incl[1024];
  const int tid = threadIdx.x;
  int blocks_before = 0, q_before = 0;  // carried across chunks of 1024 segments
  for (int base = 0; base < b; base += 1024) {
    const int s = base + tid;
    int hi = 0;
    if (s < b) hi = min(max(__ldg(new_offset + s), 0), m);
    int qmax_total;
    const int qhi = max(block_scan_incl(hi, warp_tot, qmax_total, true), q_before);  // running max, inclusive
    incl[tid] = qhi;
    __syncthreads();
    const int lo = tid ? incl[tid - 1] : q_before;
    int sn = 0, en = 0;
    if (s < b) seg_bounds(offset, s, n_total, sn, en);
    const int nq = s < b ? qhi - lo : 0;
    const int nb = (nq + SEG_KNN_WARPS - 1) / SEG_KNN_WARPS;
    int nb_total;
    const int first = blocks_before + block_scan_incl(nb, warp_tot, nb_total, false) - nb;
    for (int t = 0; t < nb; ++t) {
      const int p0 = lo + t * SEG_KNN_WARPS;
      table[first + t] = make_int4(sn, en, p0, min(p0 + SEG_KNN_WARPS, qhi));
    }
    blocks_before += nb_total;
    q_before = max(q_before, qmax_total);
  }
  if (tid == 0) *count = blocks_before;
  for (long long e = static_cast<long long>(q_before) * nsample + tid; e < static_cast<long long>(m) * nsample; e += 1024) {
    idx[e] = -1;
    dist2[e] = SEG_INIT;
  }
}

template <int NS>
__global__ void __launch_bounds__(SEG_KNN_WARPS * 32) seg_knn_kernel(const float *__restrict__ xyz,
                                                                     const float *__restrict__ new_xyz, int nsample,
                                                                     const int4 *__restrict__ table,
                                                                     const int *__restrict__ count, int *__restrict__ idx,
                                                                     float *__restrict__ dist2) {
  __shared__ uint64_t queue_all[SEG_KNN_WARPS * 64];
  __shared__ float planes[3 * SEG_KNN_TILE];
  if (static_cast<int>(blockIdx.x) >= __ldg(count)) return;
  const int4 e = __ldg(table + blockIdx.x);
  const int sn = e.x, en = e.y;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int p = e.z + warp;
  const bool valid = p < e.w;
  uint64_t *queue = queue_all + warp * 64;
  const int kslot = (nsample - 1) >> 5, klane = (nsample - 1) & 31;
  float q0 = 0.f, q1 = 0.f, q2 = 0.f;
  if (valid) {
    q0 = __ldg(new_xyz + 3 * static_cast<size_t>(p));
    q1 = __ldg(new_xyz + 3 * static_cast<size_t>(p) + 1);
    q2 = __ldg(new_xyz + 3 * static_cast<size_t>(p) + 2);
  }
  WarpSelect<NS> sel;
  sel.init();
  for (int tbase = sn; tbase < en; tbase += SEG_KNN_TILE) {
    const int tn = min(SEG_KNN_TILE, en - tbase);
    __syncthreads();  // previous tile consumed
    const float *src = xyz + static_cast<size_t>(tbase) * 3;
    for (int f = tid; f < tn * 3; f += SEG_KNN_WARPS * 32) {
      const int q = f / 3, c = f - q * 3;
      planes[c * SEG_KNN_TILE + q] = __ldg(src + f);
    }
    __syncthreads();
    if (!valid) continue;
    for (int j0 = 0; j0 < tn; j0 += 32) {
      const int j = j0 + lane;
      const bool in = j < tn;
      float d = 0.f;
      if (in)
        d = dist_seq3(__fsub_rn(planes[j], q0), __fsub_rn(planes[SEG_KNN_TILE + j], q1),
                      __fsub_rn(planes[2 * SEG_KNN_TILE + j], q2));
      const uint64_t key = pack_key(d, static_cast<uint32_t>(tbase + j));
      // `d < 1e10` is the reference's admission test against its heap's initial root (it also drops NaN)
      sel.offer(in && d < SEG_INIT && key < sel.tau, key, queue, lane, kslot, klane);
    }
  }
  if (!valid) return;
  sel.finish(queue, lane);
  int *__restrict__ oi = idx + static_cast<size_t>(p) * nsample;
  float *__restrict__ od = dist2 + static_cast<size_t>(p) * nsample;
#pragma unroll
  for (int s = 0; s < NS; ++s) {
    const int pos = s * 32 + lane;
    if (pos < nsample) {
      const uint64_t key = sel.L[s];
      const bool filled = key != KEY_INF;
      oi[pos] = filled ? static_cast<int>(static_cast<uint32_t>(key)) : sn;
      od[pos] = filled ? __uint_as_float(static_cast<uint32_t>(key >> 32)) : SEG_INIT;
    }
  }
}

static int seg_knn_blocks(int b, int m) { return ceil_div(m, SEG_KNN_WARPS) + b; }

}  // namespace pdae

using namespace pdae;

// opt_n_threads of the reference's pointops (cuda_utils.h), evaluated with the same double log() expression
static int seg_fps_block_size(int n) {
  if (n <= 0) return 1;
  const int pow_2 = static_cast<int>(log(static_cast<double>(n)) / log(2.0));
  int t = 1 << pow_2;
  if (t > 1024) t = 1024;
  if (t < 1) t = 1;
  return t;
}

extern "C" size_t pdae_seg_fps_workspace_bytes(int n_total) {
  if (n_total <= 0) return 0;
  return align256(static_cast<size_t>(n_total) * sizeof(float));
}

extern "C" int pdae_seg_fps_f32(const float *xyz, int n_total, const int *offset, const int *new_offset, int b, int n,
                                int m_total, float *tmp, int *idx, void *workspace, size_t workspace_bytes,
                                pdae_stream_t stream) {
  if (b < 0 || n < 0 || n_total < 0 || m_total < 0) return PDAE_E_INVALID;
  if (b == 0 || m_total == 0) return 0;
  if (!offset || !new_offset || !idx || (n_total > 0 && !xyz)) return PDAE_E_INVALID;
  const int bs = seg_fps_block_size(n);
  int lg_bs = 0;
  while ((1 << (lg_bs + 1)) <= bs) ++lg_bs;
  if ((static_cast<long long>(n_total) >> lg_bs) >= (1LL << 22)) return PDAE_E_UNSUPPORTED;  // tie rank: 22 bits of k / bs
  if (!tmp && n_total > 0 && (!workspace || workspace_bytes < pdae_seg_fps_workspace_bytes(n_total))) return PDAE_E_WORKSPACE;
  SegFpsArgs a;
  a.xyz = xyz;
  a.offset = offset;
  a.new_offset = new_offset;
  a.tmp = tmp;
  a.ws = static_cast<float *>(workspace);
  a.idx = idx;
  a.n_total = n_total;
  a.m_total = m_total;
  a.lg_bs = lg_bs;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  // CTA width max(128, bs) (a multiple of bs) and 2 points per thread cover n < 2 bs; from bs = 1024 on, P grows
  if (n < 1024) {
    if (bs <= 128) return launch_seg_fps_reg<128, 2>(a, b, st);
    if (bs == 256) return launch_seg_fps_reg<256, 2>(a, b, st);
    return launch_seg_fps_reg<512, 2>(a, b, st);
  }
  if (n <= 2048) return launch_seg_fps_reg<SEG_FPS_T, 2>(a, b, st);
  if (n <= 4096) return launch_seg_fps_reg<SEG_FPS_T, 4>(a, b, st);
  if (n <= SEG_REG_MAX_N) return launch_seg_fps_reg<SEG_FPS_T, 8>(a, b, st);
  seg_fps_global_kernel<SEG_FPS_T><<<b, SEG_FPS_T, 0, st>>>(a);
  PDAE_RETURN_IF_LAUNCH_FAILED();
  return 0;
}

extern "C" size_t pdae_seg_knn_workspace_bytes(int b, int m) {
  if (b < 0 || m <= 0) return 0;
  return 256 + align256(static_cast<size_t>(seg_knn_blocks(b, m)) * sizeof(int4));
}

extern "C" int pdae_seg_knn_f32(const float *xyz, int n_total, const float *new_xyz, int m, const int *offset,
                                const int *new_offset, int b, int nsample, int *idx, float *dist2, void *workspace,
                                size_t workspace_bytes, pdae_stream_t stream) {
  if (b < 0 || m < 0 || n_total < 0 || nsample < 1 || nsample > SEG_KNN_MAX_K) return PDAE_E_INVALID;
  if (m == 0) return 0;
  if (!new_xyz || !idx || !dist2 || (b > 0 && (!offset || !new_offset)) || (n_total > 0 && !xyz)) return PDAE_E_INVALID;
  if (!workspace || workspace_bytes < pdae_seg_knn_workspace_bytes(b, m)) return PDAE_E_WORKSPACE;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int *count = static_cast<int *>(workspace);
  int4 *table = reinterpret_cast<int4 *>(static_cast<unsigned char *>(workspace) + 256);
  seg_knn_table_kernel<<<1, 1024, 0, st>>>(offset, new_offset, b, n_total, m, nsample, table, count, idx, dist2);
  PDAE_RETURN_IF_LAUNCH_FAILED();
  const int grid = seg_knn_blocks(b, m);
  const int ns = (nsample + 31) / 32;
  if (ns == 1) seg_knn_kernel<1><<<grid, SEG_KNN_WARPS * 32, 0, st>>>(xyz, new_xyz, nsample, table, count, idx, dist2);
  else if (ns == 2) seg_knn_kernel<2><<<grid, SEG_KNN_WARPS * 32, 0, st>>>(xyz, new_xyz, nsample, table, count, idx, dist2);
  else if (ns == 3) seg_knn_kernel<3><<<grid, SEG_KNN_WARPS * 32, 0, st>>>(xyz, new_xyz, nsample, table, count, idx, dist2);
  else seg_knn_kernel<4><<<grid, SEG_KNN_WARPS * 32, 0, st>>>(xyz, new_xyz, nsample, table, count, idx, dist2);
  PDAE_RETURN_IF_LAUNCH_FAILED();
  return 0;
}
