// fps_rank.cuh -- value / tie-rank encodings of the furthest-point-sampling arg-max, shared by fps.cu, the fused
// patchifier (patchify.cu) and the segment FPS (pointops.cu).  Reference rule: extensions/pointnet2/_ext_src/src/sampling_gpu.cu:72-176.
#pragma once
#include "common.cuh"

namespace pdae {

// value -> monotone unsigned: -1 ("no valid point", the reference's initial best) -> 0,
// v >= 0 -> bits + 1.  Values are never NaN (fminf drops NaN distances) and never exceed 1e10.
__device__ __forceinline__ unsigned fps_val_bits(float v) { return v < 0.0f ? 0u : __float_as_uint(v) + 1u; }

// tie rank of point k: smaller wins.  (bit-reversed slot, k / bs) lexicographic.
__device__ __forceinline__ unsigned fps_rank(int k, int lg_bs) {
  const unsigned slot = static_cast<unsigned>(k) & ((1u << lg_bs) - 1u);
  const unsigned rev = lg_bs ? (__brev(slot) >> (32 - lg_bs)) : 0u;
  return (rev << 22) | (static_cast<unsigned>(k) >> lg_bs);
}
__device__ __forceinline__ int fps_unrank(unsigned r, int lg_bs) {
  const unsigned rev = r >> 22, hi = r & 0x3fffffu;
  const unsigned slot = lg_bs ? (__brev(rev) >> (32 - lg_bs)) : 0u;
  return static_cast<int>((hi << lg_bs) | slot);
}

// block-wide arg-max of (value bits, rank): returns the winning rank in every thread.
template <int T>
__device__ __forceinline__ unsigned fps_block_argmax(unsigned vb, unsigned rank, uint2 *slots /*[2][32]*/, int it) {
  constexpr int W = T / 32;
  const unsigned full = 0xffffffffu;
  unsigned m = __reduce_max_sync(full, vb);
  unsigned r = __reduce_min_sync(full, vb == m ? rank : 0xffffffffu);
  if (W == 1) return r;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint2 *buf = slots + (it & 1) * 32;
  if (lane == 0) buf[warp] = make_uint2(m, r);
  __syncthreads();
  const uint2 v = lane < W ? buf[lane] : make_uint2(0u, 0xffffffffu);
  m = __reduce_max_sync(full, v.x);
  r = __reduce_min_sync(full, v.x == m ? v.y : 0xffffffffu);
  return r;
}

// register i of a thread  ->  which of the thread's points (k = tid + p*T) it holds
template <int S, int PG>
__host__ __device__ constexpr int fps_point_of_reg(int i) {
  int sub = i / PG, rev = 0;
  for (int b = 0; b < S; ++b) rev |= ((sub >> b) & 1) << (S - 1 - b);
  return rev + ((i % PG) << S);
}
template <int S, int PG>
__device__ __forceinline__ int fps_point_of_reg_rt(int i) {
  if (S == 0) return i;
  const int sub = i / PG;
  const int rev = static_cast<int>(__brev(static_cast<unsigned>(sub)) >> (32 - S));
  return rev + ((i % PG) << S);
}

// inverse: which register holds the thread's point number v (k = tid + v*T)
template <int S, int PG>
__device__ __forceinline__ int fps_reg_of_point_rt(int v) {
  if (S == 0) return v;
  const int rev = v & ((1 << S) - 1);
  const int sub = static_cast<int>(__brev(static_cast<unsigned>(rev)) >> (32 - S));
  return sub * PG + (v >> S);
}

}  // namespace pdae
