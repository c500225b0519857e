// segemd.cu -- approximate Earth Mover's Distance over variable-size clouds packed in one batch: approxmatch, cost and
// gradient.  Layout and semantics: include/pointdae_b200.h (segment EMD).
//
// Every call starts with a one-CTA pre-pass that turns the offsets into a range table (lo1, hi1, lo2, hi2) per
// segment and, for the sums, one unit table per side: units of EMD_CHUNK owned points of one segment, listed only where
// both sides of the segment hold points.  The same pass writes the zeros of every point without an opposite segment or
// past the last segment.  Grids are sized from host-known bounds only and their CTAs past the device-side counts exit.
//
// approxmatch: segment s runs on cluster s of `cs` CTAs, the equal-size body (emd_core.cuh) on the segment's base
// pointers with the packed level strides.  The sums: the equal-size kernel with SEG set, one CTA per unit.  The cost:
// one CTA per segment (grid-stride), the equal-size reduction order relative to the segment's first column.  Every row
// and column sum is one thread's chain and there are no atomics, so a segment's bits are those of the equal-size op at
// b = 1 whatever `cs`, the grid or the stream.
#include "emd_core.cuh"
#include "segment.cuh"

namespace pdae {

// points [lo, hi) of a side: ratios (10, total) and / or gradients (total, 3) set to 0, by the whole 1024-thread CTA
__device__ __forceinline__ void seg_emd_zero(int lo, int hi, int total, float *ratio, float *grad) {
  for (int p = lo + static_cast<int>(threadIdx.x); p < hi; p += 1024) {
    if (ratio) {
#pragma unroll
      for (int j = 0; j < EMD_LEVELS; ++j) ratio[j * total + p] = 0.f;
    }
    if (grad) grad[3 * static_cast<size_t>(p)] = 0.f, grad[3 * static_cast<size_t>(p) + 1] = 0.f, grad[3 * static_cast<size_t>(p) + 2] = 0.f;
  }
}

// one CTA of 1024 threads: ranges (b), units1 / units2 (segment, first owned point relative to the segment start) and
// count = [units1, units2]; zeros as above for whichever of ratio_l / ratio_r / grad1 / grad2 is non-null
__global__ void __launch_bounds__(1024) seg_emd_table_kernel(const int *__restrict__ off1, const int *__restrict__ off2, int b,
                                                             int n_total, int m_total, int4 *__restrict__ ranges,
                                                             int2 *__restrict__ units1, int2 *__restrict__ units2,
                                                             int *__restrict__ count, float *ratio_l, float *ratio_r,
                                                             float *grad1, float *grad2) {
  __shared__ int warp_tot[32];
  __shared__ int incl[1024];
  __shared__ int4 fill[1024];
  const int tid = threadIdx.x;
  int carry1 = 0, carry2 = 0, before1 = 0, before2 = 0;
  for (int base = 0; base < b; base += 1024) {
    const int2 r1 = seg_range_chunk(off1, base, b, n_total, carry1, warp_tot, incl);
    const int2 r2 = seg_range_chunk(off2, base, b, m_total, carry2, warp_tot, incl);
    const int s = base + tid;
    if (s < b) ranges[s] = make_int4(r1.x, r1.y, r2.x, r2.y);
    const int c1 = r1.y - r1.x, c2 = r2.y - r2.x;
    const bool both = c1 > 0 && c2 > 0;
    const int nb1 = both ? (c1 + EMD_CHUNK - 1) / EMD_CHUNK : 0, nb2 = both ? (c2 + EMD_CHUNK - 1) / EMD_CHUNK : 0;
    int tot1, tot2, ftot;
    const int first1 = before1 + block_scan_incl(nb1, warp_tot, tot1, false) - nb1;
    const int first2 = before2 + block_scan_incl(nb2, warp_tot, tot2, false) - nb2;
    for (int t = 0; t < nb1; ++t) units1[first1 + t] = make_int2(s, t * EMD_CHUNK);
    for (int t = 0; t < nb2; ++t) units2[first2 + t] = make_int2(s, t * EMD_CHUNK);
    before1 += tot1;
    before2 += tot2;
    // segments with one empty side: listed, then their points are zeroed by the whole CTA
    const int nf = (!both && (c1 > 0 || c2 > 0)) ? 1 : 0;
    const int pos = block_scan_incl(nf, warp_tot, ftot, false) - nf;
    if (nf) fill[pos] = make_int4(r1.x, r1.y, r2.x, r2.y);
    __syncthreads();
    for (int f = 0; f < ftot; ++f) {
      const int4 r = fill[f];
      seg_emd_zero(r.x, r.y, n_total, ratio_l, grad1);
      seg_emd_zero(r.z, r.w, m_total, ratio_r, grad2);
    }
    __syncthreads();  // `fill` is rewritten by the next chunk
  }
  if (tid == 0) count[0] = before1, count[1] = before2;
  // points past the last segment
  seg_emd_zero(carry1, n_total, n_total, ratio_l, grad1);
  seg_emd_zero(carry2, m_total, m_total, ratio_r, grad2);
}

// grid: b * cs CTAs, clusters of cs; cluster s matches segment s
__global__ void __launch_bounds__(EMD_THREADS) seg_emd_approxmatch_kernel(const EmdMatchArgs a, const EmdSegTables sg) {
  __shared__ float4 tile[EMD_TILE];
  emd_approxmatch_body<true>(a, sg, tile);
}

// cost[s] from the rowcost of segment s's columns; 0 for a segment with an empty side (no rowcost was written there)
__global__ void __launch_bounds__(256) seg_emd_cost_reduce_kernel(const float *__restrict__ rowcost,
                                                                  const int4 *__restrict__ ranges, int b,
                                                                  float *__restrict__ cost) {
  __shared__ float p[256];
  for (int s = blockIdx.x; s < b; s += gridDim.x) {
    const int4 r = __ldg(ranges + s);
    if (r.y == r.x || r.w == r.z) {  // uniform for the CTA
      if (threadIdx.x == 0) cost[s] = 0.f;
      continue;
    }
    emd_cost_reduce_body(rowcost + r.z, r.w - r.z, p);
    if (threadIdx.x == 0) cost[s] = p[0];
    __syncthreads();  // p is rewritten for the next segment
  }
}

static size_t seg_emd_units(int b, int total) { return static_cast<size_t>(total + EMD_CHUNK - 1) / EMD_CHUNK + b; }

// workspace: count (2 ints) | ranges (b) | units1 | units2 | remainL or nothing (n_total) | remainR or rowcost (m_total)
struct SegEmdWs {
  int *count;
  int4 *ranges;
  int2 *units1, *units2;
  float *rem_l, *rem_r;
};

static SegEmdWs seg_emd_carve(void *workspace, int b, int n_total, int m_total) {
  unsigned char *w = static_cast<unsigned char *>(workspace);
  SegEmdWs r;
  r.count = reinterpret_cast<int *>(w);
  w += 256;
  r.ranges = reinterpret_cast<int4 *>(w);
  w += align256(static_cast<size_t>(b) * sizeof(int4));
  r.units1 = reinterpret_cast<int2 *>(w);
  w += align256(seg_emd_units(b, n_total) * sizeof(int2));
  r.units2 = reinterpret_cast<int2 *>(w);
  w += align256(seg_emd_units(b, m_total) * sizeof(int2));
  r.rem_l = reinterpret_cast<float *>(w);
  w += align256(static_cast<size_t>(n_total) * sizeof(float));
  r.rem_r = reinterpret_cast<float *>(w);
  return r;
}

// shared argument checks; > 0: return *rc (an error, or 0 for b = 0), 0: go on
static int seg_emd_prologue(const float *xyz1, int n_total, const float *xyz2, int m_total, const int *offset1,
                            const int *offset2, int b, int *rc) {
  *rc = 0;
  if (b < 0 || n_total < 0 || m_total < 0) return *rc = PDAE_E_INVALID, 1;
  if (b == 0) return 1;
  if (!offset1 || !offset2 || (n_total && !xyz1) || (m_total && !xyz2)) return *rc = PDAE_E_INVALID, 1;
  // ratio offsets j * total + p stay in int; b clusters of up to EMD_MAX_CLUSTER CTAs stay in one grid
  if (n_total > 0x7fffffff / EMD_LEVELS || m_total > 0x7fffffff / EMD_LEVELS || b > 0x7fffffff / EMD_MAX_CLUSTER)
    return *rc = PDAE_E_UNSUPPORTED, 1;
  return 0;
}

static int seg_emd_tables(const int *offset1, const int *offset2, int b, int n_total, int m_total, const SegEmdWs &w,
                          float *ratio_l, float *ratio_r, float *grad1, float *grad2, cudaStream_t st) {
  seg_emd_table_kernel<<<1, 1024, 0, st>>>(offset1, offset2, b, n_total, m_total, w.ranges, w.units1, w.units2, w.count,
                                           ratio_l, ratio_r, grad1, grad2);
  PDAE_RETURN_IF_LAUNCH_FAILED();
  return 0;
}

}  // namespace pdae

using namespace pdae;

extern "C" size_t pdae_seg_emd_workspace_bytes(int b, int n_total, int m_total) {
  if (b <= 0 || n_total < 0 || m_total < 0) return 0;
  return 256 + align256(static_cast<size_t>(b) * sizeof(int4)) + align256(seg_emd_units(b, n_total) * sizeof(int2)) +
         align256(seg_emd_units(b, m_total) * sizeof(int2)) + align256(static_cast<size_t>(n_total) * sizeof(float)) +
         align256(static_cast<size_t>(m_total) * sizeof(float));
}

extern "C" int pdae_seg_emd_match_f32(const float *xyz1, int n_total, const float *xyz2, int m_total, const int *offset1,
                                      const int *offset2, int b, float *ratio_l, float *ratio_r, void *workspace,
                                      size_t workspace_bytes, pdae_stream_t stream) {
  int rc;
  if (seg_emd_prologue(xyz1, n_total, xyz2, m_total, offset1, offset2, b, &rc)) return rc;
  if ((n_total && !ratio_l) || (m_total && !ratio_r)) return PDAE_E_INVALID;
  if (!workspace || workspace_bytes < pdae_seg_emd_workspace_bytes(b, n_total, m_total)) return PDAE_E_WORKSPACE;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const SegEmdWs w = seg_emd_carve(workspace, b, n_total, m_total);
  if ((rc = seg_emd_tables(offset1, offset2, b, n_total, m_total, w, ratio_l, ratio_r, nullptr, nullptr, st))) return rc;
  if (n_total == 0 || m_total == 0) return 0;  // no segment has both sides
  // cluster size from the average segment: host-known values only
  const int avg = static_cast<int>((static_cast<long long>(n_total > m_total ? n_total : m_total) + b - 1) / b);
  const int cs = emd_cluster_size(b, avg, avg);
  const EmdMatchArgs args{xyz1, xyz2, n_total, m_total, cs, ratio_l, ratio_r, w.rem_l, w.rem_r};
  PDAE_CUDA_TRY(emd_launch_clusters(seg_emd_approxmatch_kernel, b, cs, st, args, EmdSegTables{w.ranges, nullptr, nullptr}));
  return 0;
}

extern "C" int pdae_seg_emd_cost_f32(const float *xyz1, int n_total, const float *xyz2, int m_total, const int *offset1,
                                     const int *offset2, int b, const float *ratio_l, const float *ratio_r, float *cost,
                                     void *workspace, size_t workspace_bytes, pdae_stream_t stream) {
  int rc;
  if (seg_emd_prologue(xyz1, n_total, xyz2, m_total, offset1, offset2, b, &rc)) return rc;
  if (!cost || (n_total && !ratio_l) || (m_total && !ratio_r)) return PDAE_E_INVALID;
  if (!workspace || workspace_bytes < pdae_seg_emd_workspace_bytes(b, n_total, m_total)) return PDAE_E_WORKSPACE;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const SegEmdWs w = seg_emd_carve(workspace, b, n_total, m_total);
  if ((rc = seg_emd_tables(offset1, offset2, b, n_total, m_total, w, nullptr, nullptr, nullptr, nullptr, st))) return rc;
  float *rowcost = w.rem_r;
  const EmdSumArgs s{xyz1, xyz2, n_total, m_total, nullptr, ratio_l, ratio_r};
  emd_sum_kernel<true, 0, true><<<static_cast<unsigned>(seg_emd_units(b, m_total)), EMD_THREADS, 0, st>>>(
      s, nullptr, rowcost, EmdSegTables{w.ranges, w.units2, w.count + 1});
  PDAE_RETURN_IF_LAUNCH_FAILED();
  const int grid = b < 8 * sm_count() ? b : 8 * sm_count();
  seg_emd_cost_reduce_kernel<<<grid, 256, 0, st>>>(rowcost, w.ranges, b, cost);
  PDAE_RETURN_IF_LAUNCH_FAILED();
  return 0;
}

extern "C" int pdae_seg_emd_cost_grad_f32(const float *grad_cost, const float *xyz1, int n_total, const float *xyz2,
                                          int m_total, const int *offset1, const int *offset2, int b, const float *ratio_l,
                                          const float *ratio_r, float *grad1, float *grad2, void *workspace,
                                          size_t workspace_bytes, pdae_stream_t stream) {
  int rc;
  if (seg_emd_prologue(xyz1, n_total, xyz2, m_total, offset1, offset2, b, &rc)) return rc;
  if (!grad_cost || (n_total && (!ratio_l || !grad1)) || (m_total && (!ratio_r || !grad2))) return PDAE_E_INVALID;
  if (!workspace || workspace_bytes < pdae_seg_emd_workspace_bytes(b, n_total, m_total)) return PDAE_E_WORKSPACE;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const SegEmdWs w = seg_emd_carve(workspace, b, n_total, m_total);
  if ((rc = seg_emd_tables(offset1, offset2, b, n_total, m_total, w, nullptr, nullptr, grad1, grad2, st))) return rc;
  const EmdSumArgs s{xyz1, xyz2, n_total, m_total, nullptr, ratio_l, ratio_r};
  emd_sum_kernel<false, 1, true><<<static_cast<unsigned>(seg_emd_units(b, n_total)), EMD_THREADS, 0, st>>>(
      s, grad_cost, grad1, EmdSegTables{w.ranges, w.units1, w.count});
  PDAE_RETURN_IF_LAUNCH_FAILED();
  emd_sum_kernel<true, 1, true><<<static_cast<unsigned>(seg_emd_units(b, m_total)), EMD_THREADS, 0, st>>>(
      s, grad_cost, grad2, EmdSegTables{w.ranges, w.units2, w.count + 1});
  PDAE_RETURN_IF_LAUNCH_FAILED();
  return 0;
}
