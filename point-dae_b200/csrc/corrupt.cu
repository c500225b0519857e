// corrupt.cu -- the affine corruptions the model applies between the patchifier and the encoder
// (SURVEY.md 8f row 3): datasets/corrupt_util_tensor.py:59-343 (`corrupt_scale_nonorm`, `corrupt_tranlate`,
// `corrupt_rotate_360`, `corrupt_rotate_z_360`, `corrupt_reflection`, `corrupt_shear`) chained by `corrupt_data`
// (:706-728), call site models/PointCAE_transformer.py:1011-1017.
//
// The reference launches, per selected corruption, one broadcast product or batched matmul over the
// (B,G,M,3) patches and one over the (B,G,3) centres, plus the `+ center` / `- center` passes around them:
// 8-12 kernels over the same 3 MB.  Here the host hands over the per-cloud 3x3 matrices in the order they were
// drawn (b, t, 3, 3) and
//   * pdae_affine_points_f32 applies the whole chain to patches and centres in ONE pass (drop-in for
//     `corrupt_data` on tensors the model already formed), and
//   * pdae_group_affine_f32 produces the clean and the corrupted, re-centred patches straight from the kNN
//     epilogue of the patchifier (knn4.cu), so the absolute-coordinate copies never exist in memory.
// Bound: HBM/L2 streaming, 24 B per point (12 in, 12 out); the arithmetic is 9*t FMA-pipe ops per point.
#include "common.cuh"

namespace pdae {

// one thread per point of `points` (b, p, 3) followed by the points of `center` (b, g, 3)
__global__ void __launch_bounds__(256) affine_points_kernel(const float *__restrict__ points, const float *__restrict__ center,
                                                            const float *__restrict__ mats, int p, int g, int t,
                                                            long long total, float *__restrict__ out_points,
                                                            float *__restrict__ out_center) {
  const int per = p + g;
  for (long long i = blockIdx.x * 256LL + threadIdx.x; i < total; i += gridDim.x * 256LL) {
    const int cloud = static_cast<int>(i / per);
    const int j = static_cast<int>(i - static_cast<long long>(cloud) * per);
    const bool is_center = j >= p;
    const size_t o = is_center ? (static_cast<size_t>(cloud) * g + (j - p)) * 3 : (static_cast<size_t>(cloud) * p + j) * 3;
    const float *src = is_center ? center : points;
    float *dst = is_center ? out_center : out_points;
    float x = src[o], y = src[o + 1], z = src[o + 2];
    affine_seq(mats + static_cast<size_t>(cloud) * t * 9, t, x, y, z);
    dst[o] = x, dst[o + 1] = y, dst[o + 2] = z;
  }
}

// wide patches (m > 64, served by the streaming kNN of knn.cu): second pass over the centred patches
__global__ void __launch_bounds__(256) group_affine_post_kernel(float *__restrict__ nb /*in: x - c, out: ((x-c)+c)-c*/,
                                                                const float *__restrict__ center, const float *__restrict__ mats,
                                                                int g, int m, int t, long long total,
                                                                float *__restrict__ tgroup, float *__restrict__ tcenter) {
  for (long long i = blockIdx.x * 256LL + threadIdx.x; i < total; i += gridDim.x * 256LL) {
    const long long bq = i / m;
    const int pidx = static_cast<int>(i - bq * m);
    const int cloud = static_cast<int>(bq / g);
    const float *M = mats + static_cast<size_t>(cloud) * t * 9;
    const float q0 = __ldg(center + bq * 3), q1 = __ldg(center + bq * 3 + 1), q2 = __ldg(center + bq * 3 + 2);
    float ax = __fadd_rn(nb[i * 3], q0), ay = __fadd_rn(nb[i * 3 + 1], q1), az = __fadd_rn(nb[i * 3 + 2], q2);
    nb[i * 3] = __fsub_rn(ax, q0), nb[i * 3 + 1] = __fsub_rn(ay, q1), nb[i * 3 + 2] = __fsub_rn(az, q2);
    float cx = q0, cy = q1, cz = q2;
    affine_seq(M, t, ax, ay, az);
    affine_seq(M, t, cx, cy, cz);
    tgroup[i * 3] = __fsub_rn(ax, cx), tgroup[i * 3 + 1] = __fsub_rn(ay, cy), tgroup[i * 3 + 2] = __fsub_rn(az, cz);
    if (pidx == 0) tcenter[bq * 3] = cx, tcenter[bq * 3 + 1] = cy, tcenter[bq * 3 + 2] = cz;
  }
}

static unsigned stream_grid(long long total) {
  const long long want = (total + 255) / 256, cap = 148LL * 8 * 4;  // grid-stride beyond four waves of 8 CTAs per SM
  return static_cast<unsigned>(want < cap ? want : cap);
}

}  // namespace pdae

using namespace pdae;

extern "C" int pdae_affine_points_f32(const float *points, const float *center, const float *mats, int b, int p, int g, int t,
                                      float *out_points, float *out_center, pdae_stream_t stream) {
  if (b < 0 || p < 0 || g < 0 || t < 0 || t > PDAE_AFFINE_MAX_CHAIN) return PDAE_E_INVALID;
  const long long total = static_cast<long long>(b) * (static_cast<long long>(p) + g);
  if (total == 0) return 0;
  if (static_cast<long long>(p) + g > 0x7fffffffLL) return PDAE_E_UNSUPPORTED;
  if ((p > 0 && (!points || !out_points)) || (g > 0 && (!center || !out_center)) || (t > 0 && !mats)) return PDAE_E_INVALID;
  affine_points_kernel<<<stream_grid(total), 256, 0, static_cast<cudaStream_t>(stream)>>>(points, center, mats, p, g, t, total,
                                                                                         out_points, out_center);
  PDAE_RETURN_IF_LAUNCH_FAILED();
  return 0;
}

extern "C" int pdae_group_affine_f32(const float *xyz, const float *center, const float *mats, int b, int n, int g, int m, int t,
                                     int64_t *idx, float *neighborhood, float *t_neighborhood, float *t_center,
                                     pdae_stream_t stream) {
  if (b < 0 || n < 0 || g < 0 || m <= 0 || t < 0 || t > PDAE_AFFINE_MAX_CHAIN) return PDAE_E_INVALID;
  if (b == 0 || g == 0) return 0;
  if (m > n) return PDAE_E_INVALID;
  if (!xyz || !center || !neighborhood || !t_neighborhood || !t_center || (t > 0 && !mats)) return PDAE_E_INVALID;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (m <= 64) {
    // t == 0 still takes the fused branch (identity chain): point at any valid address, never dereferenced
    const GroupAffine aff{mats ? mats : xyz, t, t_neighborhood, t_center};
    return knn4_points(xyz, center, b, n, g, m, 0, nullptr, idx, neighborhood, st, nullptr, 0u, 0, &aff);
  }
  const int rc = pdae_group_f32(xyz, center, b, n, g, m, idx, neighborhood, stream);
  if (rc) return rc;
  const long long total = static_cast<long long>(b) * g * m;
  group_affine_post_kernel<<<stream_grid(total), 256, 0, st>>>(neighborhood, center, mats, g, m, t, total, t_neighborhood,
                                                              t_center);
  PDAE_RETURN_IF_LAUNCH_FAILED();
  return 0;
}
