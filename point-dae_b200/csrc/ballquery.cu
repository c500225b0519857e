// ballquery.cu -- radius grouping for the 3DETR / PointNet++ configs ("next" rows, SURVEY.md 8f):
// ball_query, group_points and group_points_grad.
//
// Semantics follow extensions/pointnet2/_ext_src/src/ball_query_gpu.cu:12-47 (first `nsample`
// indices, in index order, with d2 < radius^2; unfilled slots repeat the first hit; no hit ->
// zeros) and group_points_gpu.cu:11-31 / :46-67 of the reference.
//
// The reference runs ONE block per cloud with one thread per query scanning all n points
// serially; here a warp owns a query and scans 32 points per step (ballot + prefix popcount keep
// the index order), so a 20 000-point scene uses the whole GPU and stops as soon as a ball is full.
#include "common.cuh"
#include "reverse.cuh"

namespace pdae {

__global__ void __launch_bounds__(256) ball_query_kernel(const float *__restrict__ new_xyz, const float *__restrict__ xyz,
                                                         int n, int m, float radius2, int nsample, long long nquery,
                                                         int *__restrict__ idx) {
  const long long w = (static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  if (w >= nquery) return;
  const int lane = threadIdx.x & 31;
  const long long cloud = w / m;
  const float *__restrict__ P = xyz + cloud * n * 3;
  const float qx = __ldg(new_xyz + w * 3), qy = __ldg(new_xyz + w * 3 + 1), qz = __ldg(new_xyz + w * 3 + 2);
  int *__restrict__ out = idx + w * nsample;
  int cnt = 0, first = 0;
  for (int k0 = 0; k0 < n && cnt < nsample; k0 += 32) {
    const int k = k0 + lane;
    bool hit = false;
    if (k < n) {
      const float d2 = dist_yxz(__fsub_rn(qx, __ldg(P + 3 * k)), __fsub_rn(qy, __ldg(P + 3 * k + 1)),
                                __fsub_rn(qz, __ldg(P + 3 * k + 2)));
      hit = d2 < radius2;
    }
    const unsigned mk = __ballot_sync(0xffffffffu, hit);
    if (mk) {
      if (cnt == 0) first = k0 + __ffs(mk) - 1;
      const int pos = cnt + __popc(mk & ((1u << lane) - 1u));
      if (hit && pos < nsample) out[pos] = k;
      cnt += __popc(mk);
    }
  }
  if (cnt > nsample) cnt = nsample;
  // unfilled slots: the first hit (ball_query_gpu.cu:36-40), or 0 when the ball is empty
  for (int l = cnt + lane; l < nsample; l += 32) out[l] = first;
}

__global__ void __launch_bounds__(256) group_points_kernel(const float *__restrict__ points, const int *__restrict__ idx,
                                                           int c, int n, int ps /*npoints*nsample*/, long long total,
                                                           float *__restrict__ out) {
  const long long e = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (e >= total) return;
  const long long bc = e / ps;  // b*c + l
  const int jk = static_cast<int>(e - bc * ps);
  const long long bi = bc / c;
  out[e] = __ldg(points + bc * n + __ldg(idx + bi * ps + jk));
}

__global__ void __launch_bounds__(256) group_points_grad_kernel(const float *__restrict__ gout, const int *__restrict__ idx,
                                                                int c, int n, int ps, long long total,
                                                                float *__restrict__ gpoints) {
  const long long e = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (e >= total) return;
  const long long bc = e / ps;
  const int jk = static_cast<int>(e - bc * ps);
  const long long bi = bc / c;
  atomicAdd(gpoints + bc * n + __ldg(idx + bi * ps + jk), __ldg(gout + e));
}

}  // namespace pdae

using namespace pdae;

extern "C" int pdae_ball_query_f32(const float *new_xyz, const float *xyz, int b, int n, int m, float radius,
                                   int nsample, int *idx, pdae_stream_t stream) {
  if (b < 0 || n < 0 || m < 0 || nsample < 0) return PDAE_E_INVALID;
  const long long nquery = static_cast<long long>(b) * m;
  if (nquery == 0 || nsample == 0) return 0;
  if (!new_xyz || !idx || (n && !xyz)) return PDAE_E_INVALID;
  const long long grid = (nquery * 32 + 255) / 256;
  if (grid > 0x7fffffffLL) return PDAE_E_UNSUPPORTED;
  ball_query_kernel<<<static_cast<unsigned>(grid), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      new_xyz, xyz, n, m, radius * radius, nsample, nquery, idx);
  PDAE_RETURN_IF_LAUNCH_FAILED();
  return 0;
}

extern "C" int pdae_group_points_f32(const float *points, const int *idx, int b, int c, int n, int npoints,
                                     int nsample, float *out, pdae_stream_t stream) {
  if (b < 0 || c < 0 || n < 0 || npoints < 0 || nsample < 0) return PDAE_E_INVALID;
  const long long ps = static_cast<long long>(npoints) * nsample;
  const long long total = static_cast<long long>(b) * c * ps;
  if (total == 0) return 0;
  if (!points || !idx || !out || n == 0 || ps > 0x7fffffffLL) return PDAE_E_INVALID;
  const long long grid = (total + 255) / 256;
  if (grid > 0x7fffffffLL) return PDAE_E_UNSUPPORTED;
  group_points_kernel<<<static_cast<unsigned>(grid), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      points, idx, c, n, static_cast<int>(ps), total, out);
  PDAE_RETURN_IF_LAUNCH_FAILED();
  return 0;
}

extern "C" int pdae_group_points_grad_f32(const float *gout, const int *idx, int b, int c, int n, int npoints,
                                          int nsample, float *gpoints, pdae_stream_t stream) {
  if (b < 0 || c < 0 || n < 0 || npoints < 0 || nsample < 0) return PDAE_E_INVALID;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const size_t gsz = static_cast<size_t>(b) * c * n;
  if (gsz) {
    if (!gpoints) return PDAE_E_INVALID;
    PDAE_CUDA_TRY(cudaMemsetAsync(gpoints, 0, gsz * sizeof(float), st));
  }
  const long long ps = static_cast<long long>(npoints) * nsample;
  const long long total = static_cast<long long>(b) * c * ps;
  if (total == 0 || gsz == 0) return 0;
  if (!gout || !idx || ps > 0x7fffffffLL) return PDAE_E_INVALID;
  const long long grid = (total + 255) / 256;
  if (grid > 0x7fffffffLL) return PDAE_E_UNSUPPORTED;
  group_points_grad_kernel<<<static_cast<unsigned>(grid), 256, 0, st>>>(gout, idx, c, n, static_cast<int>(ps), total,
                                                                       gpoints);
  PDAE_RETURN_IF_LAUNCH_FAILED();
  return 0;
}

// deterministic form: gpoints[b][l][p] = +0 (+) gout[b][l][j] over the slots j = q * nsample + k with idx == p, ascending
extern "C" size_t pdae_group_points_grad_det_workspace_bytes(int b, int n, int npoints, int nsample) {
  if (b <= 0 || n < 0 || npoints < 0 || nsample < 0) return 0;
  const long long ps = static_cast<long long>(npoints) * nsample;
  if (ps > 0x7fffffffLL) return 0;
  return rev_map_bytes(b, static_cast<int>(ps), n);
}

extern "C" int pdae_group_points_grad_det_f32(const float *gout, const int *idx, int b, int c, int n, int npoints, int nsample,
                                              float *gpoints, void *workspace, size_t workspace_bytes, pdae_stream_t stream) {
  if (b < 0 || c < 0 || n < 0 || npoints < 0 || nsample < 0) return PDAE_E_INVALID;
  const size_t gsz = static_cast<size_t>(b) * c * n;
  if (gsz == 0) return 0;
  const long long ps = static_cast<long long>(npoints) * nsample;
  if (!gpoints || ps > 0x7fffffffLL || (ps && (!gout || !idx))) return PDAE_E_INVALID;
  if (!workspace || workspace_bytes < pdae_group_points_grad_det_workspace_bytes(b, n, npoints, nsample)) return PDAE_E_WORKSPACE;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  RevMap map;
  const int rc = rev_map_build(idx, b, static_cast<int>(ps), n, workspace, &map, st);
  if (rc) return rc;
  return rev_gather_channel_major(gout, nullptr, b, c, static_cast<int>(ps), n, 1, map, gpoints, st);
}
