// reverse.cu -- per-cloud reverse index (see reverse.cuh): count, scan and cursor fill build the CSR; the ordering pass
// then sorts every bucket, which makes the map -- and every gradient gathered through it -- independent of the order in
// which the fill's atomics ran.
#include <limits.h>

#include "reverse.cuh"

namespace pdae {

template <typename I>
__global__ void __launch_bounds__(256) rev_count_kernel(const I *__restrict__ idx, int s, int t, long long total,
                                                        int *__restrict__ cnt) {
  const long long e = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (e >= total) return;
  const long long cloud = e / s;
  const long long v = static_cast<long long>(__ldg(idx + e));
  if (v < 0 || v >= t) return;
  atomicAdd(cnt + cloud * t + v, 1);
}

// one CTA per cloud (blockDim a power of two <= 1024): ptr = exclusive prefix sum of cnt (t + 1 entries); cnt is zeroed
// for its second life as the fill's cursor
__global__ void __launch_bounds__(1024) rev_scan_kernel(int *__restrict__ cnt, int t, int *__restrict__ ptr) {
  __shared__ int part[1024];
  const int T = blockDim.x;
  int *c = cnt + static_cast<size_t>(blockIdx.x) * t;
  int *p = ptr + static_cast<size_t>(blockIdx.x) * (t + 1);
  const int per = (t + T - 1) / T, lo = threadIdx.x * per, hi = min(t, lo + per);
  // a thread's run is read RS_BATCH counts at a time (independent loads in flight): one cloud of 1e5 targets is one CTA
  constexpr int RS_BATCH = 8;
  int s = 0;
  for (int q0 = lo; q0 < hi; q0 += RS_BATCH) {
    int v[RS_BATCH];
#pragma unroll
    for (int u = 0; u < RS_BATCH; ++u) v[u] = q0 + u < hi ? c[q0 + u] : 0;
#pragma unroll
    for (int u = 0; u < RS_BATCH; ++u) s += v[u];
  }
  part[threadIdx.x] = s;
  __syncthreads();
  for (int o = 1; o < T; o <<= 1) {  // Hillis-Steele inclusive scan of the T partial sums
    const int v = threadIdx.x >= o ? part[threadIdx.x - o] : 0;
    __syncthreads();
    part[threadIdx.x] += v;
    __syncthreads();
  }
  int run = threadIdx.x ? part[threadIdx.x - 1] : 0;
  for (int q0 = lo; q0 < hi; q0 += RS_BATCH) {
    int v[RS_BATCH];
#pragma unroll
    for (int u = 0; u < RS_BATCH; ++u) v[u] = q0 + u < hi ? c[q0 + u] : 0;
#pragma unroll
    for (int u = 0; u < RS_BATCH; ++u) {
      if (q0 + u < hi) {
        p[q0 + u] = run;
        c[q0 + u] = 0;
      }
      run += v[u];
    }
  }
  if (threadIdx.x == T - 1) p[t] = part[T - 1];
}

// the scan of long rows (t > REV_SCAN_TILE, e.g. one cloud of 1e5 points) on many CTAs: tile sums, then every tile scans
// itself after adding the sums of the tiles before it (at most t / REV_SCAN_TILE of them); one CTA per row would serialise
// the whole row's load latencies on one SM
constexpr int REV_SCAN_TILE = 4096, REV_SCAN_THREADS = 256, REV_SCAN_PER = REV_SCAN_TILE / REV_SCAN_THREADS;

__global__ void __launch_bounds__(REV_SCAN_THREADS) rev_tile_sum_kernel(const int *__restrict__ cnt, int t, int *__restrict__ tsum) {
  __shared__ int wsum[REV_SCAN_THREADS / 32];
  const int *c = cnt + static_cast<size_t>(blockIdx.y) * t;
  const int base = blockIdx.x * REV_SCAN_TILE;
  int s = 0;
#pragma unroll
  for (int u = 0; u < REV_SCAN_PER; ++u) {
    const int q = base + u * REV_SCAN_THREADS + threadIdx.x;
    s += q < t ? c[q] : 0;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if ((threadIdx.x & 31) == 0) wsum[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    int tot = 0;
    for (int w = 0; w < REV_SCAN_THREADS / 32; ++w) tot += wsum[w];
    tsum[static_cast<size_t>(blockIdx.y) * gridDim.x + blockIdx.x] = tot;
  }
}

__global__ void __launch_bounds__(REV_SCAN_THREADS) rev_tile_scan_kernel(int *__restrict__ cnt, int t, const int *__restrict__ tsum,
                                                                         int *__restrict__ ptr) {
  __shared__ int part[REV_SCAN_THREADS];
  __shared__ int carry;
  int *c = cnt + static_cast<size_t>(blockIdx.y) * t;
  int *p = ptr + static_cast<size_t>(blockIdx.y) * (t + 1);
  const int base = blockIdx.x * REV_SCAN_TILE, lo = base + threadIdx.x * REV_SCAN_PER;
  if (threadIdx.x == 0) {
    int off = 0;
    for (int k = 0; k < static_cast<int>(blockIdx.x); ++k) off += tsum[static_cast<size_t>(blockIdx.y) * gridDim.x + k];
    carry = off;
  }
  int v[REV_SCAN_PER], s = 0;
#pragma unroll
  for (int u = 0; u < REV_SCAN_PER; ++u) {
    v[u] = lo + u < t ? c[lo + u] : 0;
    s += v[u];
  }
  part[threadIdx.x] = s;
  __syncthreads();
  for (int o = 1; o < REV_SCAN_THREADS; o <<= 1) {
    const int x = threadIdx.x >= o ? part[threadIdx.x - o] : 0;
    __syncthreads();
    part[threadIdx.x] += x;
    __syncthreads();
  }
  int run = carry + (threadIdx.x ? part[threadIdx.x - 1] : 0);
#pragma unroll
  for (int u = 0; u < REV_SCAN_PER; ++u) {
    if (lo + u < t) {
      p[lo + u] = run;
      c[lo + u] = 0;
    }
    run += v[u];
  }
  if (blockIdx.x == gridDim.x - 1 && threadIdx.x == REV_SCAN_THREADS - 1) p[t] = run;
}

template <typename I>
__global__ void __launch_bounds__(256) rev_fill_kernel(const I *__restrict__ idx, int s, int t, int div, long long total,
                                                       const int *__restrict__ ptr, int *__restrict__ cursor,
                                                       int *__restrict__ slot) {
  const long long e = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (e >= total) return;
  const long long cloud = e / s;
  const int within = static_cast<int>(e - cloud * s);
  const long long v = static_cast<long long>(__ldg(idx + e));
  if (v < 0 || v >= t) return;
  const int pos = atomicAdd(cursor + cloud * t + v, 1);
  slot[cloud * s + __ldg(ptr + cloud * (t + 1) + v) + pos] = within / div;
}

// ordering pass, part 1: one thread per bucket sorts buckets of up to REV_SHORT slots in place (insertion sort) and
// queues the longer ones in longq[1 ..] (longq[0] = their count)
__global__ void __launch_bounds__(256) rev_sort_short_kernel(const int *__restrict__ ptr, int *__restrict__ slot, int b, int s,
                                                             int t, int *__restrict__ longq) {
  const long long u = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (u >= static_cast<long long>(b) * t) return;
  const long long cloud = u / t;
  const int p = static_cast<int>(u - cloud * t);
  const int lo = __ldg(ptr + cloud * (t + 1) + p), len = __ldg(ptr + cloud * (t + 1) + p + 1) - lo;
  if (len <= 1) return;
  if (len > REV_SHORT) {
    longq[1 + atomicAdd(longq, 1)] = static_cast<int>(u);
    return;
  }
  int *a = slot + cloud * s + lo;
  for (int i = 1; i < len; ++i) {
    const int v = a[i];
    int j = i - 1;
    while (j >= 0 && a[j] > v) {
      a[j + 1] = a[j];
      --j;
    }
    a[j + 1] = v;
  }
}

constexpr int REV_LONG_THREADS = 512;

// ordering pass, part 2: CTAs take the queued buckets in turn.  Up to REV_MID slots: bitonic sort in shared memory (the
// slots of a bucket are distinct, so padding with INT_MAX keeps them in front).  Longer: ordered stream compaction of
// the cloud's sources whose target is this bucket's.
template <typename I>
__global__ void __launch_bounds__(REV_LONG_THREADS) rev_sort_long_kernel(const I *__restrict__ idx, const int *__restrict__ ptr,
                                                                         int *__restrict__ slot, int s, int t,
                                                                         const int *__restrict__ longq) {
  __shared__ int buf[REV_MID];
  __shared__ int wsum[REV_LONG_THREADS / 32];
  const int nlong = longq[0];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (int w = blockIdx.x; w < nlong; w += gridDim.x) {
    const int u = longq[1 + w];
    const long long cloud = u / t;
    const int p = static_cast<int>(u - cloud * t);
    const int lo = ptr[cloud * (t + 1) + p], len = ptr[cloud * (t + 1) + p + 1] - lo;
    int *a = slot + cloud * s + lo;
    if (len <= REV_MID) {
      int P = 1;
      while (P < len) P <<= 1;
      for (int i = tid; i < P; i += REV_LONG_THREADS) buf[i] = i < len ? a[i] : INT_MAX;
      __syncthreads();
      for (int k = 2; k <= P; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
          for (int i = tid; i < P; i += REV_LONG_THREADS) {
            const int ixj = i ^ j;
            if (ixj > i) {
              const int x = buf[i], y = buf[ixj];
              if ((x > y) == ((i & k) == 0)) buf[i] = y, buf[ixj] = x;
            }
          }
          __syncthreads();
        }
      }
      for (int i = tid; i < len; i += REV_LONG_THREADS) a[i] = buf[i];
    } else {
      const I *src = idx + cloud * s;
      int base = 0;
      for (int j0 = 0; j0 < s; j0 += REV_LONG_THREADS) {
        const int j = j0 + tid;
        const bool hit = j < s && static_cast<long long>(__ldg(src + j)) == p;
        const unsigned bal = __ballot_sync(0xffffffffu, hit);
        if (lane == 0) wsum[warp] = __popc(bal);
        __syncthreads();
        int off = 0, tot = 0;
#pragma unroll
        for (int v = 0; v < REV_LONG_THREADS / 32; ++v) {
          const int cw = wsum[v];
          off += v < warp ? cw : 0;
          tot += cw;
        }
        if (hit) a[base + off + __popc(bal & ((1u << lane) - 1u))] = j;
        base += tot;
        __syncthreads();
      }
    }
    __syncthreads();
  }
}

// channel-major gradient gather (reverse.cuh): thread per target, RG_CH channels per thread; the bucket is walked once
constexpr int RG_CH = 8;

__global__ void __launch_bounds__(256) rev_gather_cm_kernel(const float *__restrict__ gout, const float *__restrict__ weight,
                                                            int c, int s, int t, int div, int bpc, const int *__restrict__ ptr,
                                                            const int *__restrict__ slot, float *__restrict__ g) {
  const long long cloud = blockIdx.x / bpc;
  const int p = static_cast<int>(blockIdx.x - cloud * bpc) * 256 + threadIdx.x;
  if (p >= t) return;
  const int l0 = blockIdx.y * RG_CH;
  const int lo = __ldg(ptr + cloud * (t + 1) + p), hi = __ldg(ptr + cloud * (t + 1) + p + 1);
  const int *__restrict__ sl = slot + cloud * s;
  const long long gs = s / div;
  const float *__restrict__ go = gout + (cloud * c + l0) * gs;
  const float *__restrict__ wt = weight ? weight + cloud * s : nullptr;
  const int nch = min(RG_CH, c - l0);
  float acc[RG_CH];
#pragma unroll
  for (int l = 0; l < RG_CH; ++l) acc[l] = 0.f;
  for (int q = lo; q < hi; ++q) {
    const int j = __ldg(sl + q);
    const float w = wt ? __ldg(wt + j) : 1.f;
    const long long src = j / div;
#pragma unroll
    for (int l = 0; l < RG_CH; ++l) {
      if (l < nch) {
        const float v = __ldg(go + l * gs + src);
        acc[l] = __fadd_rn(acc[l], wt ? __fmul_rn(v, w) : v);
      }
    }
  }
#pragma unroll
  for (int l = 0; l < RG_CH; ++l)
    if (l < nch) g[(cloud * c + l0 + l) * t + p] = acc[l];
}


static bool rev_shape_ok(int b, int s, int t) {
  return static_cast<long long>(b) * s <= INT_MAX && static_cast<long long>(b) * (t + 1LL) <= INT_MAX;
}

// tsum: scratch of b * ceil(t / REV_SCAN_TILE) ints for the many-CTA scan of long rows, or null (one CTA per row)
template <typename I>
static int rev_csr(const I *idx, int b, int s, int t, int div, int *cnt, int *ptr, int *slot, cudaStream_t st,
                   int *tsum = nullptr) {
  const long long total = static_cast<long long>(b) * s;
  if (t) PDAE_CUDA_TRY(cudaMemsetAsync(cnt, 0, static_cast<size_t>(b) * t * sizeof(int), st));
  const unsigned grid = static_cast<unsigned>((total + 255) / 256);
  if (total) {
    rev_count_kernel<I><<<grid, 256, 0, st>>>(idx, s, t, total, cnt);
    PDAE_RETURN_IF_LAUNCH_FAILED();
  }
  if (tsum && t > REV_SCAN_TILE && b <= 65535) {
    const dim3 grid(static_cast<unsigned>((t + REV_SCAN_TILE - 1) / REV_SCAN_TILE), static_cast<unsigned>(b));
    rev_tile_sum_kernel<<<grid, REV_SCAN_THREADS, 0, st>>>(cnt, t, tsum);
    PDAE_RETURN_IF_LAUNCH_FAILED();
    rev_tile_scan_kernel<<<grid, REV_SCAN_THREADS, 0, st>>>(cnt, t, tsum, ptr);
    PDAE_RETURN_IF_LAUNCH_FAILED();
  } else {
    int threads = 32;
    while (threads < t && threads < 1024) threads <<= 1;
    rev_scan_kernel<<<b, threads, 0, st>>>(cnt, t, ptr);
    PDAE_RETURN_IF_LAUNCH_FAILED();
  }
  if (total) {
    rev_fill_kernel<I><<<grid, 256, 0, st>>>(idx, s, t, div, total, ptr, cnt, slot);
    PDAE_RETURN_IF_LAUNCH_FAILED();
  }
  return 0;
}

template <typename I>
int rev_csr_unordered(const I *idx, int b, int s, int t, int div, int *cnt, int *ptr, int *slot, cudaStream_t st) {
  if (b == 0) return 0;
  return rev_csr(idx, b, s, t, div, cnt, ptr, slot, st);
}
template int rev_csr_unordered<int64_t>(const int64_t *, int, int, int, int, int *, int *, int *, cudaStream_t);

// scratch of the ordered form: cursor (b, t), then the long-bucket queue (count + up to b * t entries)
static size_t rev_scratch_bytes(int b, int t) { return (2 * static_cast<size_t>(b) * t + 1) * sizeof(int); }

template <typename I>
static int rev_ordered(const I *idx, int b, int s, int t, int *ptr, int *slot, void *scratch, cudaStream_t st) {
  if (b == 0) return 0;
  if (!rev_shape_ok(b, s, t)) return PDAE_E_UNSUPPORTED;
  int *cnt = static_cast<int *>(scratch);
  int *longq = cnt + static_cast<size_t>(b) * t;
  int rc = rev_csr(idx, b, s, t, 1, cnt, ptr, slot, st, longq + 1);  // the queue is free until the ordering pass
  if (rc) return rc;
  PDAE_CUDA_TRY(cudaMemsetAsync(longq, 0, sizeof(int), st));
  if (s <= 1 || t == 0) return 0;
  const long long buckets = static_cast<long long>(b) * t;
  rev_sort_short_kernel<<<static_cast<unsigned>((buckets + 255) / 256), 256, 0, st>>>(ptr, slot, b, s, t, longq);
  PDAE_RETURN_IF_LAUNCH_FAILED();
  if (s > REV_SHORT) {  // a bucket can only be long when a cloud has more than REV_SHORT sources
    const long long most = static_cast<long long>(b) * (s / (REV_SHORT + 1));
    const unsigned grid = static_cast<unsigned>(most < 4LL * sm_count() ? most : 4LL * sm_count());
    rev_sort_long_kernel<I><<<grid, REV_LONG_THREADS, 0, st>>>(idx, ptr, slot, s, t, longq);
    PDAE_RETURN_IF_LAUNCH_FAILED();
  }
  return 0;
}

size_t rev_map_bytes(int b, int s, int t) {
  if (b <= 0 || s < 0 || t < 0) return 0;
  return align256(static_cast<size_t>(b) * (t + 1) * sizeof(int)) + align256(static_cast<size_t>(b) * s * sizeof(int)) +
         align256(rev_scratch_bytes(b, t));
}

template <typename I>
int rev_map_build(const I *idx, int b, int s, int t, void *ws, RevMap *out, cudaStream_t st) {
  unsigned char *w = static_cast<unsigned char *>(ws);
  int *ptr = reinterpret_cast<int *>(w);
  int *slot = reinterpret_cast<int *>(w + align256(static_cast<size_t>(b) * (t + 1) * sizeof(int)));
  void *scratch = w + align256(static_cast<size_t>(b) * (t + 1) * sizeof(int)) + align256(static_cast<size_t>(b) * s * sizeof(int));
  out->ptr = ptr;
  out->slot = slot;
  out->longq = static_cast<int *>(scratch) + static_cast<size_t>(b) * t;
  return rev_ordered(idx, b, s, t, ptr, slot, scratch, st);
}
template int rev_map_build<int32_t>(const int32_t *, int, int, int, void *, RevMap *, cudaStream_t);
template int rev_map_build<int64_t>(const int64_t *, int, int, int, void *, RevMap *, cudaStream_t);

int rev_gather_channel_major(const float *gout, const float *weight, int b, int c, int s, int t, int div, RevMap map,
                             float *g, cudaStream_t st) {
  if (b == 0 || c == 0 || t == 0) return 0;
  const long long bpc = (t + 255LL) / 256, gy = (c + RG_CH - 1LL) / RG_CH;
  if (bpc * b > 0x7fffffffLL || gy > 65535) return PDAE_E_UNSUPPORTED;
  const dim3 grid(static_cast<unsigned>(bpc * b), static_cast<unsigned>(gy));
  rev_gather_cm_kernel<<<grid, 256, 0, st>>>(gout, weight, c, s, t, div, static_cast<int>(bpc), map.ptr, map.slot, g);
  PDAE_RETURN_IF_LAUNCH_FAILED();
  return 0;
}

}  // namespace pdae

using namespace pdae;

extern "C" size_t pdae_reverse_index_workspace_bytes(int b, int s, int t) {
  if (b <= 0 || s < 0 || t < 0) return 0;
  return rev_scratch_bytes(b, t);
}

template <typename I>
static int reverse_index_entry(const I *idx, int b, int s, int t, int *ptr, int *slot, void *workspace, size_t workspace_bytes,
                               pdae_stream_t stream) {
  if (b < 0 || s < 0 || t < 0) return PDAE_E_INVALID;
  if (b == 0) return 0;
  if (!ptr || (s && (!idx || !slot))) return PDAE_E_INVALID;
  if (!workspace || workspace_bytes < pdae_reverse_index_workspace_bytes(b, s, t)) return PDAE_E_WORKSPACE;
  return rev_ordered(idx, b, s, t, ptr, slot, workspace, static_cast<cudaStream_t>(stream));
}

extern "C" int pdae_reverse_index_i32(const int32_t *idx, int b, int s, int t, int *ptr, int *slot, void *workspace,
                                      size_t workspace_bytes, pdae_stream_t stream) {
  return reverse_index_entry(idx, b, s, t, ptr, slot, workspace, workspace_bytes, stream);
}

extern "C" int pdae_reverse_index_i64(const int64_t *idx, int b, int s, int t, int *ptr, int *slot, void *workspace,
                                      size_t workspace_bytes, pdae_stream_t stream) {
  return reverse_index_entry(idx, b, s, t, ptr, slot, workspace, workspace_bytes, stream);
}
