// knn_select.cuh -- warp-level exact top-k selection primitives shared by knn.cu (streaming
// warp-select, any dimension), knn4.cu (3-D fast path with a segment-minima threshold pre-pass), featknn.cu,
// patchify.cu and pointops.cu.
// Keys are (float bits << 32 | index): the unsigned order is the (distance, lower index) order.
#pragma once
#include "common.cuh"

namespace pdae {

constexpr int KNN_WARPS = 8;
constexpr int KNN_THREADS = KNN_WARPS * 32;
constexpr int KNN_MAX_K = 128;
constexpr uint64_t KEY_INF = 0xffffffffffffffffull;

__device__ __forceinline__ uint64_t shfl_xor64(uint64_t v, int m) {
  const unsigned lo = __shfl_xor_sync(0xffffffffu, static_cast<unsigned>(v), m);
  const unsigned hi = __shfl_xor_sync(0xffffffffu, static_cast<unsigned>(v >> 32), m);
  return (static_cast<uint64_t>(hi) << 32) | lo;
}
__device__ __forceinline__ uint64_t shfl64(uint64_t v, int src) {
  const unsigned lo = __shfl_sync(0xffffffffu, static_cast<unsigned>(v), src);
  const unsigned hi = __shfl_sync(0xffffffffu, static_cast<unsigned>(v >> 32), src);
  return (static_cast<uint64_t>(hi) << 32) | lo;
}
__device__ __forceinline__ uint64_t shfl_up64(uint64_t v, int d) {
  const unsigned lo = __shfl_up_sync(0xffffffffu, static_cast<unsigned>(v), d);
  const unsigned hi = __shfl_up_sync(0xffffffffu, static_cast<unsigned>(v >> 32), d);
  return (static_cast<uint64_t>(hi) << 32) | lo;
}
__device__ __forceinline__ uint64_t umin64(uint64_t a, uint64_t b) { return a < b ? a : b; }
__device__ __forceinline__ uint64_t umax64(uint64_t a, uint64_t b) { return a < b ? b : a; }

// ascending bitonic sort of one key per lane
__device__ __forceinline__ uint64_t warp_sort32(uint64_t v, int lane) {
#pragma unroll
  for (int k = 2; k <= 32; k <<= 1) {
#pragma unroll
    for (int j = k >> 1; j > 0; j >>= 1) {
      const uint64_t o = shfl_xor64(v, j);
      const bool keep_min = ((lane & j) == 0) == ((lane & k) == 0);
      v = keep_min ? umin64(v, o) : umax64(v, o);
    }
  }
  return v;
}
// lanes hold a bitonic sequence -> ascending
__device__ __forceinline__ uint64_t warp_bitonic_merge32(uint64_t v, int lane) {
#pragma unroll
  for (int j = 16; j > 0; j >>= 1) {
    const uint64_t o = shfl_xor64(v, j);
    v = (lane & j) == 0 ? umin64(v, o) : umax64(v, o);
  }
  return v;
}

// merge 32 ascending candidates `c` into the ascending list L[0..NS) (32 keys per slot),
// keeping the 32*NS smallest.
template <int NS>
__device__ __forceinline__ void warp_merge(uint64_t (&L)[NS], uint64_t c, int lane) {
  uint64_t mcur = warp_bitonic_merge32(umin64(L[NS - 1], shfl64(c, 31 - lane)), lane);
#pragma unroll
  for (int s = NS - 2; s >= 0; --s) {
    const uint64_t r = shfl64(mcur, 31 - lane);
    const uint64_t lo = umin64(L[s], r), hi = umax64(L[s], r);
    L[s + 1] = warp_bitonic_merge32(hi, lane);
    mcur = warp_bitonic_merge32(lo, lane);
  }
  L[0] = mcur;
}


// bitonic sort of E keys per lane (E a power of two), global position g = e*32 + lane, ascending.
template <int E>
__device__ __forceinline__ void warp_sort_multi(uint64_t (&v)[E], int lane) {
#pragma unroll
  for (int k = 2; k <= 32 * E; k <<= 1) {
#pragma unroll
    for (int j = k >> 1; j > 0; j >>= 1) {
      if (j >= 32) {
#pragma unroll
        for (int e = 0; e < E; ++e) {
          const int pe = e ^ (j >> 5);
          if (pe > e) {
            const bool up = ((e * 32) & k) == 0;
            const uint64_t lo = umin64(v[e], v[pe]), hi = umax64(v[e], v[pe]);
            v[e] = up ? lo : hi;
            v[pe] = up ? hi : lo;
          }
        }
      } else {
#pragma unroll
        for (int e = 0; e < E; ++e) {
          const uint64_t o = shfl_xor64(v[e], j);
          const bool up = ((e * 32 + lane) & k) == 0;
          const bool keep_min = ((lane & j) == 0) == up;
          v[e] = keep_min ? umin64(v[e], o) : umax64(v[e], o);
        }
      }
    }
  }
}

// ---- 32-bit network (knn4.cu) -------------------------------------------------------------------------------------------
// Directions of the ten compare-exchange stages with k < 32 (k = 2,4,8,16; j = k/2..1) as one bit per stage: they depend
// on the lane only, so a kernel computes the mask once and every stage costs one bit test instead of three logic ops.
__device__ __forceinline__ uint32_t warp_sort_dir_mask(int lane) {
  uint32_t m = 0;
  int s = 0;
#pragma unroll
  for (int k = 2; k <= 16; k <<= 1)
#pragma unroll
    for (int j = k >> 1; j > 0; j >>= 1, ++s) m |= ((((lane & j) == 0) == ((lane & k) == 0)) ? 1u : 0u) << s;
  return m;
}
// ascending bitonic sort of E unsigned keys per lane (position e*32 + lane): SHFL + one predicated min/max pair per
// element and stage.  Non-negative floats sort correctly through their bit patterns.
template <int E>
__device__ __forceinline__ void warp_sort_u32(uint32_t (&v)[E], int lane, uint32_t dir_mask) {
  int s = 0;
#pragma unroll
  for (int k = 2; k <= 32 * E; k <<= 1) {
#pragma unroll
    for (int j = k >> 1; j > 0; j >>= 1) {
      if (j >= 32) {
#pragma unroll
        for (int e = 0; e < E; ++e) {
          const int pe = e ^ (j >> 5);
          if (pe > e) {
            const bool up = ((e * 32) & k) == 0;
            const uint32_t lo = min(v[e], v[pe]), hi = max(v[e], v[pe]);
            v[e] = up ? lo : hi;
            v[pe] = up ? hi : lo;
          }
        }
      } else {
        const bool low_lane = (lane & j) == 0;
        const bool keep_small = k < 32 ? ((dir_mask >> s) & 1u) != 0 : low_lane;  // k >= 32: flipped per element below
        if (k < 32) ++s;
#pragma unroll
        for (int e = 0; e < E; ++e) {
          const uint32_t o = __shfl_xor_sync(0xffffffffu, v[e], j);
          const bool up = k < 32 ? true : ((e * 32) & k) == 0;  // compile time (k < 32: already folded into the mask)
          const bool take_min = up ? keep_small : !keep_small;
          v[e] = take_min ? min(v[e], o) : max(v[e], o);
        }
      }
    }
  }
}

// NQ independent arrays through the same network in lockstep: the compare-exchange chains of one array are strictly
// dependent (SHFL -> min/max -> SHFL ...), so interleaving the arrays of a warp's queries hides the shuffle latency.
template <int NQ, int E>
__device__ __forceinline__ void warp_sort_u32_multi(uint32_t (&v)[NQ][E], int lane, uint32_t dir_mask) {
  int s = 0;
#pragma unroll
  for (int k = 2; k <= 32 * E; k <<= 1) {
#pragma unroll
    for (int j = k >> 1; j > 0; j >>= 1) {
      if (j >= 32) {
#pragma unroll
        for (int a = 0; a < NQ; ++a)
#pragma unroll
          for (int e = 0; e < E; ++e) {
            const int pe = e ^ (j >> 5);
            if (pe > e) {
              const bool up = ((e * 32) & k) == 0;
              const uint32_t lo = min(v[a][e], v[a][pe]), hi = max(v[a][e], v[a][pe]);
              v[a][e] = up ? lo : hi;
              v[a][pe] = up ? hi : lo;
            }
          }
      } else {
        const bool low_lane = (lane & j) == 0;
        const bool keep_small = k < 32 ? ((dir_mask >> s) & 1u) != 0 : low_lane;
        if (k < 32) ++s;
#pragma unroll
        for (int a = 0; a < NQ; ++a)
#pragma unroll
          for (int e = 0; e < E; ++e) {
            const uint32_t o = __shfl_xor_sync(0xffffffffu, v[a][e], j);
            const bool up = k < 32 ? true : ((e * 32) & k) == 0;
            const bool take_min = up ? keep_small : !keep_small;
            v[a][e] = take_min ? min(v[a][e], o) : max(v[a][e], o);
          }
      }
    }
  }
}

// streaming warp-select state: ascending list of 32*NS keys (one per lane per slot), the running
// k-th key `tau`, and the fill level of the warp's candidate queue (64 entries in shared memory).
template <int NS>
struct WarpSelect {
  uint64_t L[NS];
  uint64_t tau;
  int qn;
  __device__ __forceinline__ void init() {
#pragma unroll
    for (int s = 0; s < NS; ++s) L[s] = KEY_INF;
    tau = KEY_INF;
    qn = 0;
  }
  // offer one candidate per lane (`pass` lanes only); flushes the queue when it holds >= 32 keys
  __device__ __forceinline__ void offer(bool pass, uint64_t key, uint64_t *queue, int lane, int kslot, int klane) {
    const unsigned mk = __ballot_sync(0xffffffffu, pass);
    if (mk) {
      if (pass) queue[qn + __popc(mk & ((1u << lane) - 1u))] = key;
      qn += __popc(mk);
      __syncwarp();
      if (qn >= 32) {
        qn -= 32;
        uint64_t c = queue[qn + lane];
        __syncwarp();
        c = warp_sort32(c, lane);
        warp_merge<NS>(L, c, lane);
        uint64_t lk = L[0];
#pragma unroll
        for (int s = 1; s < NS; ++s) lk = (s == kslot) ? L[s] : lk;
        tau = shfl64(lk, klane);
      }
    }
  }
  __device__ __forceinline__ void finish(uint64_t *queue, int lane) {
    if (qn > 0) {
      uint64_t c = lane < qn ? queue[lane] : KEY_INF;
      __syncwarp();
      c = warp_sort32(c, lane);
      warp_merge<NS>(L, c, lane);
      qn = 0;
    }
  }
};

}  // namespace pdae
