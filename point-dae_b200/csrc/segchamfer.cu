// segchamfer.cu -- Chamfer distance over variable-size clouds packed in one batch: forward, gradients and the L2 / L1
// mean losses.  Layout and semantics: include/pointdae_b200.h (segment Chamfer).
//
// Forward: a one-CTA pre-pass turns the offsets into a table of units (direction, row block of one segment): no unit
// straddles a segment and units exist only where both sides of the segment hold points; the same pass writes (0, -1)
// for every row without an opposite segment.  The main grid is sized from host-known values only and its CTAs beyond
// the table exit.  Each unit runs the FP32-pipe scan body of the equal-size forward (chamfer_core.cuh,
// chamfer_min_body<..., SYM = false, SEG = true>) over its rows against the opposite segment: exact minimum, lowest
// index on ties, so the results do not depend on the launch shape.  No atomics.
//
// Backward: the indices are global and a point is only ever matched inside its own segment, so the gradient is the
// equal-size backward at b = 1 over the packed arrays (atomic or ordered form), instantiated with the idx < 0 guard.
//
// Loss: per-segment means in float64 (one CTA per segment, fixed order), then one fixed-order pass over the segments.
#include "chamfer_core.cuh"
#include "segment.cuh"

namespace pdae {

constexpr int SEG_LOSS_THREADS = 256;

// one CTA of 1024 threads.  table0 entry (rows [r, e) of xyz1, segment [o0, o1) of xyz2); table1 the converse.
__global__ void __launch_bounds__(1024) seg_chamfer_table_kernel(const int *__restrict__ off1, const int *__restrict__ off2,
                                                                 int b, int n_total, int m_total, int rows,
                                                                 int4 *__restrict__ table0, int4 *__restrict__ table1,
                                                                 int *__restrict__ count, float *__restrict__ dist1,
                                                                 float *__restrict__ dist2, int *__restrict__ idx1,
                                                                 int *__restrict__ idx2) {
  __shared__ int warp_tot[32];
  __shared__ int incl[1024];
  __shared__ int4 fill[1024];
  const int tid = threadIdx.x;
  int carry1 = 0, carry2 = 0, before0 = 0, before1 = 0;
  for (int base = 0; base < b; base += 1024) {
    const int2 r1 = seg_range_chunk(off1, base, b, n_total, carry1, warp_tot, incl);
    const int2 r2 = seg_range_chunk(off2, base, b, m_total, carry2, warp_tot, incl);
    const int c1 = r1.y - r1.x, c2 = r2.y - r2.x;
    const bool both = c1 > 0 && c2 > 0;
    const int nb0 = both ? (c1 + rows - 1) / rows : 0, nb1 = both ? (c2 + rows - 1) / rows : 0;
    int tot0, tot1, ftot;
    const int first0 = before0 + block_scan_incl(nb0, warp_tot, tot0, false) - nb0;
    const int first1 = before1 + block_scan_incl(nb1, warp_tot, tot1, false) - nb1;
    for (int t = 0; t < nb0; ++t) table0[first0 + t] = make_int4(r1.x + t * rows, r1.y, r2.x, r2.y);
    for (int t = 0; t < nb1; ++t) table1[first1 + t] = make_int4(r2.x + t * rows, r2.y, r1.x, r1.y);
    before0 += tot0;
    before1 += tot1;
    // segments with one empty side: listed, then their rows are written by the whole CTA
    const int nf = (!both && (c1 > 0 || c2 > 0)) ? 1 : 0;
    const int pos = block_scan_incl(nf, warp_tot, ftot, false) - nf;
    if (nf) fill[pos] = make_int4(r1.x, r1.y, r2.x, r2.y);
    __syncthreads();
    for (int f = 0; f < ftot; ++f) {
      const int4 r = fill[f];
      for (int p = r.x + tid; p < r.y; p += 1024) dist1[p] = 0.0f, idx1[p] = -1;
      for (int p = r.z + tid; p < r.w; p += 1024) dist2[p] = 0.0f, idx2[p] = -1;
    }
    __syncthreads();  // `fill` is rewritten by the next chunk
  }
  if (tid == 0) count[0] = before0, count[1] = before1;
  // rows past the last segment
  for (int p = carry1 + tid; p < n_total; p += 1024) dist1[p] = 0.0f, idx1[p] = -1;
  for (int p = carry2 + tid; p < m_total; p += 1024) dist2[p] = 0.0f, idx2[p] = -1;
}

template <int QT>
__global__ void __launch_bounds__(CH_THREADS, 1) seg_chamfer_min_kernel(const float *__restrict__ xyz1,
                                                                        const float *__restrict__ xyz2,
                                                                        const int4 *__restrict__ table0,
                                                                        const int4 *__restrict__ table1,
                                                                        const int *__restrict__ count, float *dist1,
                                                                        float *dist2, int *idx1, int *idx2) {
  __shared__ __align__(16) float tile[2][3][CH_TILE];
  __shared__ __align__(16) unsigned colmin[1][CH_THREADS / 32][4];
  const int n0 = __ldg(count), n1 = __ldg(count + 1);
  int u = blockIdx.x;
  const bool second = u >= n0;
  if (second) {
    u -= n0;
    if (u >= n1) return;  // uniform for the CTA
  }
  const int4 e = __ldg((second ? table1 : table0) + u);
  const float *Q = (second ? xyz2 : xyz1) + 3 * static_cast<size_t>(e.x);
  const float *R = (second ? xyz1 : xyz2) + 3 * static_cast<size_t>(e.z);
  float *dist = (second ? dist2 : dist1) + e.x;
  int *idx = (second ? idx2 : idx1) + e.x;
  chamfer_min_body<QT, false, true>(Q, R, e.y - e.x, e.w - e.z, 0, 0, dist, idx, nullptr, e.z, nullptr, tile, colmin);
}

// rows per unit: 128 (one query per thread) when the segments average at most 256 points, as the equal-size forward
// does for small clouds, else 512.  Host-known values only.
static int seg_chamfer_rows(int b, int n_total, int m_total) {
  const long long big = n_total > m_total ? n_total : m_total;
  return big <= 256LL * b ? CH_THREADS : 4 * CH_THREADS;
}
static long long seg_chamfer_units0(int b, int n_total, int rows) { return (static_cast<long long>(n_total) + rows - 1) / rows + b; }

// ---- loss ----------------------------------------------------------------------------------------------------------
// state (4b + 1 words) = [|S|, end1 (b), end2 (b), weight1 (b), weight2 (b)]: the loss writes it, its backward reads it.
// weight = rn(w / (float)(|S| * size)) of each side of each segment of S (0 elsewhere), fp32 bits.
__global__ void __launch_bounds__(1024) seg_ends_kernel(const int *__restrict__ off1, const int *__restrict__ off2, int b,
                                                        int n_total, int m_total, int *__restrict__ state) {
  __shared__ int warp_tot[32];
  __shared__ int incl[1024];
  int carry1 = 0, carry2 = 0;
  for (int base = 0; base < b; base += 1024) {
    const int2 r1 = seg_range_chunk(off1, base, b, n_total, carry1, warp_tot, incl);
    const int2 r2 = seg_range_chunk(off2, base, b, m_total, carry2, warp_tot, incl);
    const int s = base + threadIdx.x;
    if (s < b) state[1 + s] = r1.y, state[1 + b + s] = r2.y;
  }
}

// means (b, 2): mean f(dist) of each side of each segment (0 for an empty side); f = identity or sqrt, summed in float64
__global__ void __launch_bounds__(SEG_LOSS_THREADS) seg_loss_partial_kernel(const float *__restrict__ dist1,
                                                                            const float *__restrict__ dist2,
                                                                            const int *__restrict__ state, int b, int l1,
                                                                            double *__restrict__ means) {
  __shared__ double red[2][SEG_LOSS_THREADS / 32];
  const int tid = threadIdx.x;
  for (int s = blockIdx.x; s < b; s += gridDim.x) {
#pragma unroll
    for (int side = 0; side < 2; ++side) {
      const int *end = state + 1 + side * b;
      const int lo = s ? end[s - 1] : 0, hi = end[s];
      const float *__restrict__ d = side ? dist2 : dist1;
      double acc = 0.0;
      for (int p = lo + tid; p < hi; p += SEG_LOSS_THREADS) {
        acc += static_cast<double>(l1 ? __fsqrt_rn(d[p]) : d[p]);  // the fp32 sqrt of the equal-size loss
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
      if ((tid & 31) == 0) red[side][tid >> 5] = acc;
    }
    __syncthreads();
    if (tid < 2) {
      const int *end = state + 1 + tid * b;
      const int cnt = end[s] - (s ? end[s - 1] : 0);
      double t = 0.0;
#pragma unroll
      for (int w = 0; w < SEG_LOSS_THREADS / 32; ++w) t += red[tid][w];
      means[2 * static_cast<size_t>(s) + tid] = cnt ? t / cnt : 0.0;
    }
    __syncthreads();
  }
}

__global__ void __launch_bounds__(1024) seg_loss_final_kernel(const double *__restrict__ means, int *__restrict__ state,
                                                              int b, int l1, float *__restrict__ loss3) {
  __shared__ double r1[1024], r2[1024];
  __shared__ int rc[1024];
  const int tid = threadIdx.x;
  double t1 = 0.0, t2 = 0.0;
  int c = 0;
  for (int s = tid; s < b; s += 1024) {
    const int n1 = state[1 + s] - (s ? state[s] : 0), n2 = state[1 + b + s] - (s ? state[b + s] : 0);
    if (n1 > 0 && n2 > 0) t1 += means[2 * static_cast<size_t>(s)], t2 += means[2 * static_cast<size_t>(s) + 1], ++c;
  }
  r1[tid] = t1, r2[tid] = t2, rc[tid] = c;
  __syncthreads();
  for (int w = 512; w > 0; w >>= 1) {
    if (tid < w) r1[tid] += r1[tid + w], r2[tid] += r2[tid + w], rc[tid] += rc[tid + w];
    __syncthreads();
  }
  const int ns = rc[0];
  // w is 1 or 1/2, so rn(w / c) = w * rn(1 / c) exactly (c <= 2^62: no subnormal), and rn(1 / c) is __frcp_rn
  const float w = l1 ? 0.5f : 1.0f;
  for (int s = tid; s < b; s += 1024) {
    const int n1 = state[1 + s] - (s ? state[s] : 0), n2 = state[1 + b + s] - (s ? state[b + s] : 0);
    const bool in = n1 > 0 && n2 > 0;
    state[1 + 2 * b + s] = __float_as_int(in ? __fmul_rn(w, __frcp_rn(__ll2float_rn(static_cast<long long>(ns) * n1))) : 0.0f);
    state[1 + 3 * b + s] = __float_as_int(in ? __fmul_rn(w, __frcp_rn(__ll2float_rn(static_cast<long long>(ns) * n2))) : 0.0f);
  }
  if (tid == 0) {
    const double term1 = ns ? r1[0] / ns : 0.0, term2 = ns ? r2[0] / ns : 0.0;
    loss3[0] = static_cast<float>(l1 ? (term1 + term2) * 0.5 : term1 + term2);
    loss3[1] = static_cast<float>(term1);
    loss3[2] = static_cast<float>(term2);
    state[0] = ns;
  }
}

// d(loss)/d(dist) of a point: the upstream scalar times the weight of the point's segment in `state` (rounded as GradMean
// rounds w / (b * n)), with the sqrt derivative for L1.  Called only for points with a match, whose segment therefore
// has both sides non-empty; it is found by binary search over the ends in `state`.
struct GradSegMean {
  const float *gloss;
  const float *dist1, *dist2;
  const int *state;
  int b, l1;
  __device__ __forceinline__ float at(bool second, size_t o) const {
    const int *end = state + 1 + (second ? b : 0);
    const int p = static_cast<int>(o);
    int lo = 0, hi = b - 1;
    while (lo < hi) {
      const int mid = (lo + hi) >> 1;
      if (__ldg(end + mid) > p) hi = mid;
      else lo = mid + 1;
    }
    const float g = __fmul_rn(__ldg(gloss), __int_as_float(__ldg(end + 2 * b + lo)));
    if (!l1) return g;
    return __fdiv_rn(g, __fmul_rn(2.0f, __fsqrt_rn(__ldg((second ? dist2 : dist1) + o))));
  }
};

}  // namespace pdae

using namespace pdae;

extern "C" size_t pdae_seg_chamfer_fwd_workspace_bytes(int b, int n_total, int m_total) {
  if (b <= 0 || n_total < 0 || m_total < 0 || (n_total == 0 && m_total == 0)) return 0;
  const int rows = seg_chamfer_rows(b, n_total, m_total);
  return 256 + align256(static_cast<size_t>(seg_chamfer_units0(b, n_total, rows)) * sizeof(int4)) +
         align256(static_cast<size_t>(seg_chamfer_units0(b, m_total, rows)) * sizeof(int4));
}

extern "C" int pdae_seg_chamfer_fwd_f32(const float *xyz1, int n_total, const float *xyz2, int m_total, const int *offset1,
                                        const int *offset2, int b, float *dist1, float *dist2, int *idx1, int *idx2,
                                        void *workspace, size_t workspace_bytes, pdae_stream_t stream) {
  if (b < 0 || n_total < 0 || m_total < 0) return PDAE_E_INVALID;
  if (b == 0) return 0;
  if (!offset1 || !offset2 || (n_total > 0 && (!xyz1 || !dist1 || !idx1)) || (m_total > 0 && (!xyz2 || !dist2 || !idx2)))
    return PDAE_E_INVALID;
  if (n_total == 0 && m_total == 0) return 0;
  if (n_total > 0x7fffffff / 3 || m_total > 0x7fffffff / 3) return PDAE_E_UNSUPPORTED;  // the scan body's 3 * nr
  if (!workspace || workspace_bytes < pdae_seg_chamfer_fwd_workspace_bytes(b, n_total, m_total)) return PDAE_E_WORKSPACE;
  const int rows = seg_chamfer_rows(b, n_total, m_total);
  const long long u0 = seg_chamfer_units0(b, n_total, rows), u1 = seg_chamfer_units0(b, m_total, rows);
  if (u0 + u1 > 0x7fffffffLL) return PDAE_E_UNSUPPORTED;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  unsigned char *w = static_cast<unsigned char *>(workspace);
  int *count = reinterpret_cast<int *>(w);
  int4 *table0 = reinterpret_cast<int4 *>(w + 256);
  int4 *table1 = reinterpret_cast<int4 *>(w + 256 + align256(static_cast<size_t>(u0) * sizeof(int4)));
  seg_chamfer_table_kernel<<<1, 1024, 0, st>>>(offset1, offset2, b, n_total, m_total, rows, table0, table1, count, dist1,
                                               dist2, idx1, idx2);
  PDAE_RETURN_IF_LAUNCH_FAILED();
  const unsigned grid = static_cast<unsigned>(u0 + u1);
  if (rows == CH_THREADS)
    seg_chamfer_min_kernel<1><<<grid, CH_THREADS, 0, st>>>(xyz1, xyz2, table0, table1, count, dist1, dist2, idx1, idx2);
  else
    seg_chamfer_min_kernel<4><<<grid, CH_THREADS, 0, st>>>(xyz1, xyz2, table0, table1, count, dist1, dist2, idx1, idx2);
  PDAE_RETURN_IF_LAUNCH_FAILED();
  return 0;
}

// shared argument checks of the four gradient entry points; > 0: gradients zeroed (an empty side), 0: go on
static int seg_bwd_prologue(const float *xyz1, int n_total, const float *xyz2, int m_total, float *gx1, float *gx2,
                            cudaStream_t st, int *rc) {
  *rc = 0;
  if (n_total < 0 || m_total < 0) return *rc = PDAE_E_INVALID, 1;
  if ((n_total && (!xyz1 || !gx1)) || (m_total && (!xyz2 || !gx2))) return *rc = PDAE_E_INVALID, 1;
  if (n_total == 0 || m_total == 0) {  // no point has a match
    cudaError_t e = cudaSuccess;
    if (n_total) e = cudaMemsetAsync(gx1, 0, static_cast<size_t>(n_total) * 3 * sizeof(float), st);
    if (e == cudaSuccess && m_total) e = cudaMemsetAsync(gx2, 0, static_cast<size_t>(m_total) * 3 * sizeof(float), st);
    *rc = static_cast<int>(e);
    return 1;
  }
  return 0;
}

extern "C" int pdae_seg_chamfer_bwd_f32(const float *xyz1, int n_total, const float *xyz2, int m_total, const int *idx1,
                                        const int *idx2, const float *gd1, const float *gd2, float *gx1, float *gx2,
                                        pdae_stream_t stream) {
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int rc;
  if (seg_bwd_prologue(xyz1, n_total, xyz2, m_total, gx1, gx2, st, &rc)) return rc;
  if (!idx1 || !idx2 || !gd1 || !gd2) return PDAE_E_INVALID;
  return launch_chamfer_bwd<GradArrays, true>(xyz1, xyz2, idx1, idx2, GradArrays{gd1, gd2}, 1, n_total, m_total, gx1, gx2, st);
}

extern "C" size_t pdae_seg_chamfer_bwd_det_workspace_bytes(int n_total, int m_total) {
  if (n_total <= 0 || m_total <= 0) return 0;
  return chamfer_bwd_det_bytes(1, n_total, m_total);
}

extern "C" int pdae_seg_chamfer_bwd_det_f32(const float *xyz1, int n_total, const float *xyz2, int m_total, const int *idx1,
                                            const int *idx2, const float *gd1, const float *gd2, float *gx1, float *gx2,
                                            void *workspace, size_t workspace_bytes, pdae_stream_t stream) {
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int rc;
  if (seg_bwd_prologue(xyz1, n_total, xyz2, m_total, gx1, gx2, st, &rc)) return rc;
  if (!idx1 || !idx2 || !gd1 || !gd2) return PDAE_E_INVALID;
  if (!workspace || workspace_bytes < pdae_seg_chamfer_bwd_det_workspace_bytes(n_total, m_total)) return PDAE_E_WORKSPACE;
  return launch_chamfer_bwd_det<GradArrays, true>(xyz1, xyz2, idx1, idx2, GradArrays{gd1, gd2}, 1, n_total, m_total, gx1, gx2,
                                                  workspace, st);
}

extern "C" size_t pdae_seg_chamfer_loss_workspace_bytes(int b) {
  if (b <= 0) return 0;
  return align256(2 * static_cast<size_t>(b) * sizeof(double));
}

extern "C" int pdae_seg_chamfer_loss_f32(const float *dist1, int n_total, const float *dist2, int m_total, const int *offset1,
                                         const int *offset2, int b, int l1, float *loss3, int *state, void *workspace,
                                         size_t workspace_bytes, pdae_stream_t stream) {
  if (b < 0 || n_total < 0 || m_total < 0) return PDAE_E_INVALID;
  if (b == 0) return 0;
  if (!offset1 || !offset2 || !loss3 || !state || (n_total && !dist1) || (m_total && !dist2)) return PDAE_E_INVALID;
  if (!workspace || workspace_bytes < pdae_seg_chamfer_loss_workspace_bytes(b)) return PDAE_E_WORKSPACE;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  double *means = static_cast<double *>(workspace);
  seg_ends_kernel<<<1, 1024, 0, st>>>(offset1, offset2, b, n_total, m_total, state);
  PDAE_RETURN_IF_LAUNCH_FAILED();
  const int grid = b < 8 * sm_count() ? b : 8 * sm_count();
  seg_loss_partial_kernel<<<grid, SEG_LOSS_THREADS, 0, st>>>(dist1, dist2, state, b, l1 ? 1 : 0, means);
  PDAE_RETURN_IF_LAUNCH_FAILED();
  seg_loss_final_kernel<<<1, 1024, 0, st>>>(means, state, b, l1 ? 1 : 0, loss3);
  PDAE_RETURN_IF_LAUNCH_FAILED();
  return 0;
}

static int seg_loss_bwd_impl(const float *xyz1, int n_total, const float *xyz2, int m_total, const int *idx1, const int *idx2,
                             const float *dist1, const float *dist2, const int *state, int b, const float *gloss, int l1,
                             float *gx1, float *gx2, void *workspace, size_t workspace_bytes, bool det,
                             pdae_stream_t stream) {
  if (b < 0) return PDAE_E_INVALID;
  if (b == 0) return 0;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int rc;
  if (seg_bwd_prologue(xyz1, n_total, xyz2, m_total, gx1, gx2, st, &rc)) return rc;
  if (!idx1 || !idx2 || !gloss || !state || (l1 && (!dist1 || !dist2))) return PDAE_E_INVALID;
  const GradSegMean gs{gloss, dist1, dist2, state, b, l1 ? 1 : 0};
  if (!det) return launch_chamfer_bwd<GradSegMean, true>(xyz1, xyz2, idx1, idx2, gs, 1, n_total, m_total, gx1, gx2, st);
  if (!workspace || workspace_bytes < pdae_seg_chamfer_bwd_det_workspace_bytes(n_total, m_total)) return PDAE_E_WORKSPACE;
  return launch_chamfer_bwd_det<GradSegMean, true>(xyz1, xyz2, idx1, idx2, gs, 1, n_total, m_total, gx1, gx2, workspace, st);
}

extern "C" int pdae_seg_chamfer_loss_bwd_f32(const float *xyz1, int n_total, const float *xyz2, int m_total, const int *idx1,
                                             const int *idx2, const float *dist1, const float *dist2, const int *state, int b,
                                             const float *gloss, int l1, float *gx1, float *gx2, pdae_stream_t stream) {
  return seg_loss_bwd_impl(xyz1, n_total, xyz2, m_total, idx1, idx2, dist1, dist2, state, b, gloss, l1, gx1, gx2, nullptr, 0,
                           false, stream);
}

extern "C" int pdae_seg_chamfer_loss_bwd_det_f32(const float *xyz1, int n_total, const float *xyz2, int m_total,
                                                 const int *idx1, const int *idx2, const float *dist1, const float *dist2,
                                                 const int *state, int b, const float *gloss, int l1, float *gx1, float *gx2,
                                                 void *workspace, size_t workspace_bytes, pdae_stream_t stream) {
  return seg_loss_bwd_impl(xyz1, n_total, xyz2, m_total, idx1, idx2, dist1, dist2, state, b, gloss, l1, gx1, gx2, workspace,
                           workspace_bytes, true, stream);
}
