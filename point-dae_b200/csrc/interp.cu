// interp.cu -- three_nn / three_interpolate (+grad): the feature-propagation ops of the PointNet++ decoder
// exported by the reference's pointnet2._ext (SURVEY.md 8b row 5, bindings.cpp:14-16).
//
// Semantics follow extensions/pointnet2/_ext_src/src/interpolate_gpu.cu:
//   three_nn (:12-62): for every "unknown" point the three smallest squared distances to the "known" set,
//     ascending, ties -> lower index (the reference's strict `<` insertion chain), slots that never fill keep
//     (float)1e40 = +inf and index 0; d = fma(dz,dz, fma(dx,dx, dy*dy)) with dx = u - k (SASS of the rebuilt
//     reference); the reference compares in double, which is exact for fp32 inputs.
//   three_interpolate (:76-104): out[b,l,j] = p[l,i1]*w1 + p[l,i2]*w2 + p[l,i3]*w3, contracted by nvcc to
//     fma(p3,w3, fma(p1,w1, rn(p2*w2))).
//   three_interpolate_grad (:118-144): scatter-add of g*w into zeros (order-free like the reference's atomics).
//
// The reference launches ONE block per cloud (<= 512 threads); here the unknown points of all clouds spread over
// the grid, the known cloud streams through shared memory as planes (one LDS.128 feeds four candidates) and the
// three best stay in registers behind a single "beats the third" test.
#include "common.cuh"
#include "reverse.cuh"

namespace pdae {

constexpr int TN_THREADS = 128;
constexpr int TN_TILE = 1024;  // known points per shared-memory tile (12 KB)

__global__ void __launch_bounds__(TN_THREADS) three_nn_kernel(const float *__restrict__ unknown,
                                                              const float *__restrict__ known, int n, int m,
                                                              int blocks_per_cloud, float *__restrict__ dist2,
                                                              int *__restrict__ idx) {
  __shared__ __align__(16) float sx[TN_TILE], sy[TN_TILE], sz[TN_TILE];
  const int cloud = blockIdx.x / blocks_per_cloud;
  const int j = (blockIdx.x - cloud * blocks_per_cloud) * TN_THREADS + threadIdx.x;
  const float *__restrict__ K = known + static_cast<long long>(cloud) * m * 3;
  const bool live = j < n;
  float ux = 0.f, uy = 0.f, uz = 0.f;
  if (live) {
    const float *u = unknown + (static_cast<long long>(cloud) * n + j) * 3;
    ux = __ldg(u), uy = __ldg(u + 1), uz = __ldg(u + 2);
  }
  const float inf = __int_as_float(0x7f800000);
  float b1 = inf, b2 = inf, b3 = inf;
  int i1 = 0, i2 = 0, i3 = 0;
  for (int t0 = 0; t0 < m; t0 += TN_TILE) {
    const int cnt = min(TN_TILE, m - t0);
    __syncthreads();
    for (int e = threadIdx.x; e < cnt * 3; e += TN_THREADS) {  // coalesced AoS read, planar store
      const float v = __ldg(K + static_cast<long long>(t0) * 3 + e);
      const int p = e / 3, c = e - p * 3;
      (c == 0 ? sx : c == 1 ? sy : sz)[p] = v;
    }
    for (int e = cnt + threadIdx.x; e < ((cnt + 3) & ~3); e += TN_THREADS) sx[e] = sy[e] = sz[e] = inf;  // pad: d = inf
    __syncthreads();
    for (int p = 0; p < cnt; p += 4) {
      const float4 x4 = *reinterpret_cast<const float4 *>(sx + p);
      const float4 y4 = *reinterpret_cast<const float4 *>(sy + p);
      const float4 z4 = *reinterpret_cast<const float4 *>(sz + p);
      const float xs[4] = {x4.x, x4.y, x4.z, x4.w}, ys[4] = {y4.x, y4.y, y4.z, y4.w}, zs[4] = {z4.x, z4.y, z4.z, z4.w};
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const float d = dist_yxz(__fsub_rn(ux, xs[q]), __fsub_rn(uy, ys[q]), __fsub_rn(uz, zs[q]));
        if (d < b3) {  // b1 <= b2 <= b3 always holds, so failing this test fails the whole reference chain
          const int k = t0 + p + q;
          if (d < b1) {
            b3 = b2, i3 = i2, b2 = b1, i2 = i1, b1 = d, i1 = k;
          } else if (d < b2) {
            b3 = b2, i3 = i2, b2 = d, i2 = k;
          } else {
            b3 = d, i3 = k;
          }
        }
      }
    }
  }
  if (live) {
    const long long o = (static_cast<long long>(cloud) * n + j) * 3;
    dist2[o] = b1, dist2[o + 1] = b2, dist2[o + 2] = b3;
    idx[o] = i1, idx[o + 1] = i2, idx[o + 2] = i3;
  }
}

constexpr int TI_CH = 8;  // channels per thread: idx / weight loaded once, reused TI_CH times

__global__ void __launch_bounds__(256) three_interpolate_kernel(const float *__restrict__ points,
                                                                const int *__restrict__ idx,
                                                                const float *__restrict__ weight, int c, int m, int n,
                                                                float *__restrict__ out) {
  const int j = blockIdx.x * 256 + threadIdx.x;
  if (j >= n) return;
  const int cloud = blockIdx.z, l0 = blockIdx.y * TI_CH;
  const long long o = (static_cast<long long>(cloud) * n + j) * 3;
  const int i1 = __ldg(idx + o), i2 = __ldg(idx + o + 1), i3 = __ldg(idx + o + 2);
  const float w1 = __ldg(weight + o), w2 = __ldg(weight + o + 1), w3 = __ldg(weight + o + 2);
#pragma unroll
  for (int dl = 0; dl < TI_CH; ++dl) {
    const int l = l0 + dl;
    if (l >= c) break;
    const float *__restrict__ row = points + (static_cast<long long>(cloud) * c + l) * m;
    const float v = __fmaf_rn(__ldg(row + i3), w3, __fmaf_rn(__ldg(row + i1), w1, __fmul_rn(__ldg(row + i2), w2)));
    out[(static_cast<long long>(cloud) * c + l) * n + j] = v;
  }
}

__global__ void __launch_bounds__(256) three_interpolate_grad_kernel(const float *__restrict__ gout,
                                                                     const int *__restrict__ idx,
                                                                     const float *__restrict__ weight, int c, int m,
                                                                     int n, float *__restrict__ gpoints) {
  const int j = blockIdx.x * 256 + threadIdx.x;
  if (j >= n) return;
  const int cloud = blockIdx.z, l0 = blockIdx.y * TI_CH;
  const long long o = (static_cast<long long>(cloud) * n + j) * 3;
  const int i1 = __ldg(idx + o), i2 = __ldg(idx + o + 1), i3 = __ldg(idx + o + 2);
  const float w1 = __ldg(weight + o), w2 = __ldg(weight + o + 1), w3 = __ldg(weight + o + 2);
#pragma unroll
  for (int dl = 0; dl < TI_CH; ++dl) {
    const int l = l0 + dl;
    if (l >= c) break;
    const float g = __ldg(gout + (static_cast<long long>(cloud) * c + l) * n + j);
    float *__restrict__ row = gpoints + (static_cast<long long>(cloud) * c + l) * m;
    atomicAdd(row + i1, __fmul_rn(g, w1));
    atomicAdd(row + i2, __fmul_rn(g, w2));
    atomicAdd(row + i3, __fmul_rn(g, w3));
  }
}

}  // namespace pdae

using namespace pdae;

extern "C" int pdae_three_nn_f32(const float *unknown, const float *known, int b, int n, int m, float *dist2, int *idx,
                                 pdae_stream_t stream) {
  if (b < 0 || n < 0 || m < 0) return PDAE_E_INVALID;
  if (b == 0 || n == 0) return 0;
  if (!unknown || !dist2 || !idx || (m && !known)) return PDAE_E_INVALID;
  const long long bpc = (static_cast<long long>(n) + TN_THREADS - 1) / TN_THREADS;
  if (bpc * b > 0x7fffffffLL) return PDAE_E_UNSUPPORTED;
  three_nn_kernel<<<static_cast<unsigned>(bpc * b), TN_THREADS, 0, static_cast<cudaStream_t>(stream)>>>(
      unknown, known, n, m, static_cast<int>(bpc), dist2, idx);
  PDAE_RETURN_IF_LAUNCH_FAILED();
  return 0;
}

static int interp_grid(int b, int c, int n, dim3 *grid) {
  const long long gx = (static_cast<long long>(n) + 255) / 256, gy = (c + TI_CH - 1) / TI_CH;
  if (gy > 65535 || b > 65535) return PDAE_E_UNSUPPORTED;
  *grid = dim3(static_cast<unsigned>(gx), static_cast<unsigned>(gy), static_cast<unsigned>(b));
  return 0;
}

extern "C" int pdae_three_interpolate_f32(const float *points, const int *idx, const float *weight, int b, int c, int m,
                                          int n, float *out, pdae_stream_t stream) {
  if (b < 0 || c < 0 || m < 0 || n < 0) return PDAE_E_INVALID;
  if (b == 0 || c == 0 || n == 0) return 0;
  if (!points || !idx || !weight || !out || m == 0) return PDAE_E_INVALID;
  dim3 grid;
  const int rc = interp_grid(b, c, n, &grid);
  if (rc) return rc;
  three_interpolate_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(points, idx, weight, c, m, n, out);
  PDAE_RETURN_IF_LAUNCH_FAILED();
  return 0;
}

extern "C" int pdae_three_interpolate_grad_f32(const float *gout, const int *idx, const float *weight, int b, int c,
                                               int n, int m, float *gpoints, pdae_stream_t stream) {
  if (b < 0 || c < 0 || m < 0 || n < 0) return PDAE_E_INVALID;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const size_t gsz = static_cast<size_t>(b) * c * m;
  if (gsz) {
    if (!gpoints) return PDAE_E_INVALID;
    PDAE_CUDA_TRY(cudaMemsetAsync(gpoints, 0, gsz * sizeof(float), st));
  }
  if (gsz == 0 || n == 0) return 0;
  if (!gout || !idx || !weight) return PDAE_E_INVALID;
  dim3 grid;
  const int rc = interp_grid(b, c, n, &grid);
  if (rc) return rc;
  three_interpolate_grad_kernel<<<grid, 256, 0, st>>>(gout, idx, weight, c, m, n, gpoints);
  PDAE_RETURN_IF_LAUNCH_FAILED();
  return 0;
}

// deterministic form: gpoints[b][l][p] = +0 (+) rn(gout[b][l][i] * weight[b][i][s]) over the slots i * 3 + s with
// idx == p, ascending
extern "C" size_t pdae_three_interpolate_grad_det_workspace_bytes(int b, int n, int m) {
  if (b <= 0 || n < 0 || m < 0 || 3LL * n > 0x7fffffffLL) return 0;
  return rev_map_bytes(b, 3 * n, m);
}

extern "C" int pdae_three_interpolate_grad_det_f32(const float *gout, const int *idx, const float *weight, int b, int c, int n,
                                                   int m, float *gpoints, void *workspace, size_t workspace_bytes,
                                                   pdae_stream_t stream) {
  if (b < 0 || c < 0 || m < 0 || n < 0 || 3LL * n > 0x7fffffffLL) return PDAE_E_INVALID;
  const size_t gsz = static_cast<size_t>(b) * c * m;
  if (gsz == 0) return 0;
  if (!gpoints || (n && (!gout || !idx || !weight))) return PDAE_E_INVALID;
  if (!workspace || workspace_bytes < pdae_three_interpolate_grad_det_workspace_bytes(b, n, m)) return PDAE_E_WORKSPACE;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  RevMap map;
  const int rc = rev_map_build(idx, b, 3 * n, m, workspace, &map, st);
  if (rc) return rc;
  return rev_gather_channel_major(gout, weight, b, c, 3 * n, m, 3, map, gpoints, st);
}
