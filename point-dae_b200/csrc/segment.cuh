// segment.cuh -- device helpers shared by the kernels over packed variable-size clouds (pointops.cu, segchamfer.cu, segemd.cu).
#pragma once
#include "common.cuh"

namespace pdae {

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

// Segment ends under the rule the segment kNN applies to its queries: row p belongs to the first segment s with
// p < offset[s], so segment s is [end[s-1], end[s]) with end[s] = max(clamp(offset[0..s])), end[-1] = 0.  For
// non-decreasing offsets that is [offset[s-1], offset[s]) clamped into [0, total]; for any others the segments still
// never overlap, so every row has at most one segment.  One chunk [base, base + 1024) of segments on a 1024-thread CTA:
// this thread's segment gets (end[s-1], end[s]) (empty past b); `carry` enters as end[base - 1] and leaves as the last
// end of the chunk.  incl[1024] is scratch.
__device__ __forceinline__ int2 seg_range_chunk(const int *__restrict__ off, int base, int b, int total, int &carry,
                                                int *warp_tot /*[32]*/, int *incl /*[1024]*/) {
  const int s = base + threadIdx.x;
  const int e = s < b ? min(max(__ldg(off + s), 0), total) : 0;
  int chunk_max;
  const int hi = max(block_scan_incl(e, warp_tot, chunk_max, true), carry);
  incl[threadIdx.x] = hi;
  __syncthreads();
  const int lo = threadIdx.x ? incl[threadIdx.x - 1] : carry;
  __syncthreads();
  carry = max(carry, chunk_max);
  return make_int2(lo, hi);
}

}  // namespace pdae
