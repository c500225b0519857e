// common.cuh -- shared device helpers for the sm_100a geometry kernels.
//
// Rounding contract: every distance is formed with explicitly rounded single operations in
// the order nvcc emits for the reference kernels (chamfer.cu:42-45, sampling_gpu.cu:106-107:
// fma(dz,dz, fma(dx,dx, rn(dy*dy)))), so results are bit-identical with the reference on any
// input.  Blackwell's packed fp32 ops (FADD2/FMUL2/FFMA2, PTX *.f32x2) are IEEE-exact per half
// and are used to halve the issue slots of the FMA-pipe-bound inner loops.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "pointdae_b200.h"

namespace pdae {

__device__ __forceinline__ uint64_t f2_as_u64(float2 v) { return *reinterpret_cast<uint64_t *>(&v); }
__device__ __forceinline__ float2 u64_as_f2(uint64_t v) { return *reinterpret_cast<float2 *>(&v); }

// packed fp32x2 (sm_100+): one issue slot, two IEEE fp32 results.
__device__ __forceinline__ float2 sub2(float2 a, float2 b) {
  uint64_t r;
  asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(f2_as_u64(a)), "l"(f2_as_u64(b)));
  return u64_as_f2(r);
}
__device__ __forceinline__ float2 mul2(float2 a, float2 b) {
  uint64_t r;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(f2_as_u64(a)), "l"(f2_as_u64(b)));
  return u64_as_f2(r);
}
__device__ __forceinline__ float2 fma2(float2 a, float2 b, float2 c) {
  uint64_t r;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(f2_as_u64(a)), "l"(f2_as_u64(b)), "l"(f2_as_u64(c)));
  return u64_as_f2(r);
}
// 3-input min (FMNMX3, sm_100+); NaN operands are ignored like fminf.
__device__ __forceinline__ float min3(float a, float b, float c) {
  float r;
  asm("min.f32 %0, %1, %2, %3;" : "=f"(r) : "f"(a), "f"(b), "f"(c));
  return r;
}

// squared distance, chamfer / FPS / ball-query rounding order (y product first, then x, then z).
__device__ __forceinline__ float dist_yxz(float dx, float dy, float dz) {
  return __fmaf_rn(dz, dz, __fmaf_rn(dx, dx, __fmul_rn(dy, dy)));
}
__device__ __forceinline__ float2 dist_yxz2(float2 dx, float2 dy, float2 dz) {
  return fma2(dz, dz, fma2(dx, dx, mul2(dy, dy)));
}
// squared distance, kNN rounding order (sequential fma over dims 0,1,2 from +0).
__device__ __forceinline__ float dist_seq3(float dx, float dy, float dz) {
  return __fmaf_rn(dz, dz, __fmaf_rn(dy, dy, __fmul_rn(dx, dx)));
}

__device__ __forceinline__ int lane_id() { return threadIdx.x & 31; }

// Row vector times a stack of t row-major 3x3 matrices, one after the other (the reference applies its affine
// corruptions sequentially with torch.matmul(points, R), datasets/corrupt_util_tensor.py:59-343): every step is
// out_j = fma(z, R[2][j], fma(y, R[1][j], rn(x * R[0][j]))), which for the diagonal matrices of scale / translate /
// reflection is exactly the reference's elementwise product.
__device__ __forceinline__ void affine_seq(const float *__restrict__ mats, int t, float &x, float &y, float &z) {
  for (int s = 0; s < t; ++s, mats += 9) {
    const float nx = __fmaf_rn(z, __ldg(mats + 6), __fmaf_rn(y, __ldg(mats + 3), __fmul_rn(x, __ldg(mats + 0))));
    const float ny = __fmaf_rn(z, __ldg(mats + 7), __fmaf_rn(y, __ldg(mats + 4), __fmul_rn(x, __ldg(mats + 1))));
    const float nz = __fmaf_rn(z, __ldg(mats + 8), __fmaf_rn(y, __ldg(mats + 5), __fmul_rn(x, __ldg(mats + 2))));
    x = nx, y = ny, z = nz;
  }
}

// optional second output of the fused Group epilogue (knn4.cu, patchify.cu): the corrupted copy of every patch.
struct GroupAffine {
  const float *mats;  // (b, t, 3, 3)
  int t;
  float *tgroup;      // (b, q, k, 3): affine(((x - c) + c)) - affine(c)
  float *tcenter;     // (b, q, 3):    affine(c)
};

// ascending-order key of a (non-negative distance, index) pair: a plain unsigned compare orders
// by distance first and by index on ties.
__device__ __forceinline__ uint64_t pack_key(float d, uint32_t i) {
  return (static_cast<uint64_t>(__float_as_uint(d)) << 32) | i;
}

static inline int ceil_div(long long a, long long b) { return static_cast<int>((a + b - 1) / b); }
static inline size_t align256(size_t v) { return (v + 255) & ~static_cast<size_t>(255); }

// SMs of the current device (cached per device index; 148 if the query fails)
inline int sm_count() {
  static int cached[64];
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
  if (cached[dev] == 0) {
    int n = 0;
    cached[dev] = (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && n > 0) ? n : 148;
  }
  return cached[dev];
}

// cross-file internals
// knn.cu: planar-input, any-channel-count DGCNN kNN (warp-select kernel); used directly for small c.
int feat_knn_generic(const float *x, int b, int c, int n, int k, int64_t *idx, cudaStream_t st);
// knn4.cu: 3-D fast path, k <= 64 (multi-query warps, segment-minima threshold, TMA tile prefetch, chunks along the
// reference cloud through an optional caller-owned workspace): row-major points with optional fused Group output, and
// planar (b,3,n) self-kNN; same results as knn.cu.  PDAE_E_UNSUPPORTED when one chunk exceeds its 16-bit step numbers.
int knn4_points(const float *ref, const float *query, int b, int r, int q, int k, int out_kq, float *dist, int64_t *idx,
                float *group, cudaStream_t st, uint64_t *keys = nullptr, uint32_t ref_offset = 0u, int raw_group = 0,
                const GroupAffine *affine = nullptr, void *ws = nullptr, size_t ws_bytes = 0);
int knn4_planar(const float *x, int b, int n, int k, int64_t *idx, cudaStream_t st, void *ws = nullptr, size_t ws_bytes = 0);
size_t knn4_workspace_bytes(int b, int r, int q, int k);
// chamfer_tc.cu: Chamfer forward with the tensor cores as an exact filter (both clouds >= 512 points; clouds above 2048
// points are searched in column chunks and need the forward's workspace for the merged keys)
bool chamfer_tc_applies(int b, int n, int m, size_t workspace_bytes);
int chamfer_tc_forward(const float *xyz1, const float *xyz2, int b, int n, int m, float *dist1, float *dist2, int *idx1,
                       int *idx2, void *workspace, size_t workspace_bytes, cudaStream_t st, unsigned long long *stats = nullptr,
                       long long *trace = nullptr);
bool chamfer_tc_sharded_applies(int b, int n, int m_local);
int chamfer_tc_sharded(const float *xyz1, const float *xyz2_local, int b, int n, int m_local, int ref_offset, uint64_t *keys1,
                       float *dist2_local, int *idx2_local, void *workspace, size_t workspace_bytes, cudaStream_t st);

}  // namespace pdae

// host-side launch check: returns the cudaError_t (positive) to the caller, never prints/exits.
#define PDAE_RETURN_IF_LAUNCH_FAILED()          \
  do {                                          \
    cudaError_t e__ = cudaPeekAtLastError();    \
    if (e__ != cudaSuccess) {                   \
      (void)cudaGetLastError();                 \
      return static_cast<int>(e__);             \
    }                                           \
  } while (0)

#define PDAE_CUDA_TRY(expr)                                  \
  do {                                                       \
    cudaError_t e__ = (expr);                                \
    if (e__ != cudaSuccess) return static_cast<int>(e__);    \
  } while (0)
