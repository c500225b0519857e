// knn4.cu -- 3-D k nearest neighbours, second-generation fast path (knn_cuda.KNN with dim 3, the fused Group tail,
// the first DGCNN EdgeConv layer).  Same results as knn.cu bit for bit (ascending by (squared distance,
// index), distance = fma(dz,dz, fma(dy,dy, dx*dx)) like KNN_CUDA's `ssd += tmp*tmp` loop); the schedule is built around
// the FP32 FMA pipe instead of the selection logic:
//
//   * a warp owns QW queries AT ONCE: every lane loads four adjacent reference points per step (one LDS.128 per plane)
//     and evaluates them against all QW queries, so the shared-memory traffic and the address arithmetic are paid once
//     per QW x 128 pair evaluations;
//   * pass 1 keeps, per lane and query, E running minima over disjoint subsets of the lane's points ("segments":
//     32*E per query, one FMNMX3 per two pair evaluations).  The minima are distances of distinct points, so their k-th
//     smallest (one fp32 bitonic sort across the warp) is an upper bound tau of the true k-th distance, and a tight one
//     (~1.4 k points pass it);
//   * pass 2 re-evaluates the stream and records only WHICH 4-point steps of a lane contain a distance <= tau (one
//     predicated byte store); the few recorded steps (~k per query) are re-evaluated per tile, their qualifying points
//     compacted into a per-query key queue with ballots, and one 64-bit bitonic sort yields the exact ascending
//     (distance, lower index first) order.  A query whose lists or queue overflow (mass ties) or whose tau is not
//     finite is redone with the exact streaming warp-select of knn.cu, so the result is exact for every input;
//   * reference tiles (2048 points) are prefetched with the TMA unit -- cp.async.bulk global -> shared, completion on
//     an mbarrier -- while the previous tile is being scanned, then transposed shared -> shared into planes
//     (UBLKCP in SASS); clouds whose rows are not 16-byte aligned fall back to register staging;
//   * shapes with few queries and a long reference cloud (scene scale: 2048 queries x 100 000 points) are cut along
//     the reference cloud into grid.z chunks; each chunk emits its k best keys and a warp-per-query merge kernel
//     finishes (the key order makes the merge exact), so every SM has work.
#include "knn_select.cuh"

namespace pdae {

struct Knn4Args {
  const float *ref;     // PLANAR ? (b, 3, r) : (b, r, 3)
  const float *query;   // PLANAR ? unused : (b, q, 3)
  float *dist;          // optional, Euclidean
  int64_t *idx;         // optional
  float *group;         // optional (b, q, k, 3): ref[idx] - query
  uint64_t *keys;       // optional (b, q, k): (squared-distance bits << 32 | ref_offset + index) for sharded merges
  uint64_t *chunk_keys; // (nz, b, q, k) when the reference cloud is cut into nz > 1 chunks (caller-owned workspace)
  uint32_t ref_offset;
  int raw_group;
  GroupAffine aff;
  int r, q, k;
  int tile;             // reference points per shared-memory tile (multiple of 256)
  int tiles_per_chunk;
  int out_kq;
  int tma;              // 1: tiles arrive through cp.async.bulk + mbarrier
  int dense_in_stage;   // 1: the rescan's dense lists live in the landing zone (it is idle by then)
};

// ---- TMA (bulk copy) + mbarrier, PTX ----------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ bool mbar_try_wait(uint64_t *bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}

// ---- shared epilogue: ascending keys -> idx / dist / keys / Group outputs ------------------------------------------------
template <bool PLANAR, int E, bool AFF>
__device__ __forceinline__ void knn4_emit(const Knn4Args &a, const float *__restrict__ R, int cloud, int qidx, float q0,
                                          float q1, float q2, const uint64_t (&keys)[E], int lane) {
  const int q = a.q, k = a.k;
  const size_t bq = static_cast<size_t>(cloud) * q + qidx;
#pragma unroll
  for (int e = 0; e < E; ++e) {
    const int p = e * 32 + lane;
    if (p < k) {
      const uint64_t key = keys[e];
      const uint32_t ji = static_cast<uint32_t>(key);
      const size_t o = a.out_kq ? (static_cast<size_t>(cloud) * k + p) * q + qidx : bq * k + p;
      if (a.idx) a.idx[o] = static_cast<int64_t>(ji);
      if (a.dist) a.dist[o] = __fsqrt_rn(__uint_as_float(static_cast<uint32_t>(key >> 32)));
      if (a.keys) a.keys[bq * k + p] = key == KEY_INF ? KEY_INF : key + a.ref_offset;  // fewer than k points: +inf keys
      if (!PLANAR && a.group) {
        // Group: neighbours relative to the centre (models/PointCAE_transformer.py:84-85); dropout_patch_random: the
        // neighbours themselves
        const bool raw = a.raw_group != 0;
        float *g = a.group + (bq * k + p) * 3;
        const float x = __ldg(R + 3 * static_cast<size_t>(ji)), y = __ldg(R + 3 * static_cast<size_t>(ji) + 1);
        const float z = __ldg(R + 3 * static_cast<size_t>(ji) + 2);
        if constexpr (!AFF) {
          g[0] = raw ? x : __fsub_rn(x, q0);
          g[1] = raw ? y : __fsub_rn(y, q1);
          g[2] = raw ? z : __fsub_rn(z, q2);
        } else {
          // fused corrupt_data: the reference re-adds the centre to the centred patch, transforms patch and centre
          // with the same matrices, and subtracts the centres again (models/PointCAE_transformer.py:1011-1017)
          const float *mats = a.aff.mats + static_cast<size_t>(cloud) * a.aff.t * 9;
          float ax = __fadd_rn(__fsub_rn(x, q0), q0), ay = __fadd_rn(__fsub_rn(y, q1), q1);
          float az = __fadd_rn(__fsub_rn(z, q2), q2);
          g[0] = __fsub_rn(ax, q0), g[1] = __fsub_rn(ay, q1), g[2] = __fsub_rn(az, q2);
          float cx = q0, cy = q1, cz = q2;
          affine_seq(mats, a.aff.t, ax, ay, az);
          affine_seq(mats, a.aff.t, cx, cy, cz);
          float *tg = a.aff.tgroup + (bq * k + p) * 3;
          tg[0] = __fsub_rn(ax, cx), tg[1] = __fsub_rn(ay, cy), tg[2] = __fsub_rn(az, cz);
          if (p == 0) {
            float *tc = a.aff.tcenter + bq * 3;
            tc[0] = cx, tc[1] = cy, tc[2] = cz;
          }
        }
      }
    }
  }
}

template <int E>
struct Knn4Smem {
  static constexpr int CAP = 32 * E;  // keys per query queue
  static constexpr int LC = 5 * E;    // lane-private step slots per query (+1 slot that absorbs overflow)
  // a query's step lists ([LC + 1][32] u16) are dead once its dense list is built, and only then is its key queue
  // ([CAP] u64) written: both live in one region
  static constexpr size_t lists_bytes = static_cast<size_t>(LC + 1) * 64, queue_bytes = static_cast<size_t>(CAP) * 8;
  static constexpr size_t per_query = lists_bytes > queue_bytes ? lists_bytes : queue_bytes;
  static constexpr size_t dense_bytes = static_cast<size_t>(LC) * 32 * 4;  // per warp: (step, lane) entries of one query
  // with TMA the dense lists sit in the landing zone (no copy is in flight while the rescan runs)
  __host__ __device__ static constexpr size_t per_warp(int qw, int tma) { return qw * per_query + (tma ? 0 : dense_bytes); }
};

// SPEC (streamed clouds): the CTA's last warp is a PRODUCER -- it waits for the TMA copy of the next tile, transposes it
// into the free one of two plane buffers and hands it to the NW-1 compute warps through mbarriers (full / empty per
// buffer); the compute warps never meet at a CTA barrier and never touch the staging, so the FMA pipe keeps running while
// tiles are converted.  !SPEC (single-tile clouds): all warps stage the tile together, once.
template <bool PLANAR, int E /*keys per lane in the final sort: 2 (k<=32) or 4 (k<=64)*/, int QW /*queries per warp*/,
          int NW /*warps per CTA*/, bool AFF, bool SPEC>
__global__ void __launch_bounds__(NW * 32, NW == 8 ? 3 : 5) knn4_kernel(const Knn4Args a) {
  constexpr int CW = SPEC ? NW - 1 : NW;   // compute warps
  constexpr int NT = SPEC ? 32 : NW * 32;  // threads that stage a tile
  constexpr int CAP = Knn4Smem<E>::CAP, LC = Knn4Smem<E>::LC;
  constexpr int NS = E / 2;  // fallback warp-select slots
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int T = a.tile;
  uint64_t *bar = reinterpret_cast<uint64_t *>(smem_raw);  // [0] landing zone full, [1..2] planes full, [3..4] planes empty
  float *planes0 = reinterpret_cast<float *>(smem_raw + 128);                       // [SPEC ? 2 : 1][3][T]
  float *stage = planes0 + (SPEC ? 6 : 3) * T;                                      // [3*T] landing zone (tma only)
  unsigned char *warp_area = reinterpret_cast<unsigned char *>(a.tma ? stage + 3 * T : stage);
  const int tid = SPEC ? (threadIdx.x & 31) : threadIdx.x, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  constexpr size_t PQ = Knn4Smem<E>::per_query;
  unsigned char *my_area = warp_area + static_cast<size_t>(warp) * Knn4Smem<E>::per_warp(QW, a.dense_in_stage);
  // query qi: step lists = [LC + 1][32] u16 at my_area + qi * PQ, later overwritten by its key queue [CAP] u64
  uint32_t *dense = a.dense_in_stage ? reinterpret_cast<uint32_t *>(stage) + warp * (32 * LC)
                                     : reinterpret_cast<uint32_t *>(my_area + static_cast<size_t>(QW) * PQ);  // [32 * LC]
  float *planes = planes0;  // the buffer being filled (producer) / scanned (compute warps)
  const int cloud = blockIdx.y;
  const int r = a.r, q = a.q, k = a.k;
  const float *__restrict__ R = a.ref + static_cast<size_t>(cloud) * r * 3;
  const float *__restrict__ Qp = PLANAR ? R : a.query + static_cast<size_t>(cloud) * q * 3;
  const int ntiles_all = (r + T - 1) / T;
  const int t_begin = blockIdx.z * a.tiles_per_chunk;
  const int t_end = min(ntiles_all, t_begin + a.tiles_per_chunk);
  const int nt = t_end - t_begin;
  const int kslot = (k - 1) >> 5, klane = (k - 1) & 31;
  const float INF = __int_as_float(0x7f800000);
  const unsigned FULL = 0xffffffffu;
  const unsigned lt_mask = (1u << lane) - 1u;
  uint32_t parity = 0;

  if (threadIdx.x == 0) {
    mbar_init(bar, 1);
    if (SPEC) {
      mbar_init(bar + 1, 1), mbar_init(bar + 2, 1);
      mbar_init(bar + 3, CW), mbar_init(bar + 4, CW);
    }
  }
  __syncthreads();

  auto tile_n = [&](int tl) { return min(T, r - tl * T); };
  auto issue_tile = [&](int tl) {  // one thread
    const int tbase = tl * T, tn = tile_n(tl);
    if (PLANAR) {
      mbar_expect_tx(bar, static_cast<uint32_t>(tn) * 12u);
#pragma unroll
      for (int c = 0; c < 3; ++c) bulk_g2s(stage + c * T, R + static_cast<size_t>(c) * r + tbase, static_cast<uint32_t>(tn) * 4u, bar);
    } else {
      mbar_expect_tx(bar, static_cast<uint32_t>(tn) * 12u);
      bulk_g2s(stage, R + static_cast<size_t>(tbase) * 3, static_cast<uint32_t>(tn) * 12u, bar);
    }
  };
  // planes <- tile tl (from the landing zone, or from global memory), padded to a multiple of 256 points with x = +inf
  auto fill_planes = [&](int tl) {
    const int tbase = tl * T, tn = tile_n(tl);
    const int tnp = (tn + 255) & ~255;
    const float4 PX = make_float4(INF, INF, INF, INF), P0 = make_float4(0.f, 0.f, 0.f, 0.f);
    float4 *pl4 = reinterpret_cast<float4 *>(planes);
    const int T4 = T >> 2;
    if (a.tma) {
      const float4 *st4 = reinterpret_cast<const float4 *>(stage);
      const int nquad = tn >> 2;  // tn % 4 == 0 on this path
      for (int g = tid; g < (tnp >> 2); g += NT) {
        float4 X = PX, Y = P0, Z = P0;
        if (g < nquad) {
          if (PLANAR) {
            X = st4[g], Y = st4[T4 + g], Z = st4[2 * T4 + g];
          } else {
            const float4 a0 = st4[3 * g], a1 = st4[3 * g + 1], a2 = st4[3 * g + 2];
            X = make_float4(a0.x, a0.w, a1.z, a2.y);
            Y = make_float4(a0.y, a1.x, a1.w, a2.z);
            Z = make_float4(a0.z, a1.y, a2.x, a2.w);
          }
        }
        pl4[g] = X, pl4[T4 + g] = Y, pl4[2 * T4 + g] = Z;
      }
    } else if (PLANAR) {
      for (int c = 0; c < 3; ++c)
        for (int p = tid; p < tnp; p += NT)
          planes[c * T + p] = p < tn ? __ldg(R + static_cast<size_t>(c) * r + tbase + p) : (c == 0 ? INF : 0.f);
    } else if ((r & 3) == 0 && (reinterpret_cast<uintptr_t>(a.ref) & 15) == 0) {
      const float4 *src4 = reinterpret_cast<const float4 *>(R + static_cast<size_t>(tbase) * 3);
      const int nquad = tn >> 2;
      for (int g = tid; g < (tnp >> 2); g += NT) {
        float4 X = PX, Y = P0, Z = P0;
        if (g < nquad) {
          const float4 a0 = __ldg(src4 + 3 * g), a1 = __ldg(src4 + 3 * g + 1), a2 = __ldg(src4 + 3 * g + 2);
          X = make_float4(a0.x, a0.w, a1.z, a2.y);
          Y = make_float4(a0.y, a1.x, a1.w, a2.z);
          Z = make_float4(a0.z, a1.y, a2.x, a2.w);
        }
        pl4[g] = X, pl4[T4 + g] = Y, pl4[2 * T4 + g] = Z;
      }
    } else {
      const float *src = R + static_cast<size_t>(tbase) * 3;
      for (int f = tid; f < tnp * 3; f += NT) {
        const int p = f / 3, c = f - p * 3;
        planes[c * T + p] = p < tn ? __ldg(src + f) : (c == 0 ? INF : 0.f);
      }
    }
  };
  // make tile tl current; (tma) start the copy of tile `next` (-1: none) as soon as the landing zone is free
  auto acquire = [&](int tl, int next) {
    if (a.tma) {
      while (!mbar_try_wait(bar, parity)) {}
      parity ^= 1u;
    }
    __syncthreads();  // the previous tile's planes are fully consumed
    fill_planes(tl);
    __syncthreads();
    if (a.tma && next >= 0 && tid == 0) issue_tile(next);
  };

  // SPEC, compute warps: wait for / give back the plane buffer of position cseq in the CTA's tile sequence
  uint32_t cseq = 0;
  auto tile_begin = [&](int tl, int next) {
    if constexpr (SPEC) {
      const uint32_t buf = cseq & 1u;
      while (!mbar_try_wait(bar + 1 + buf, (cseq >> 1) & 1u)) {}
      planes = planes0 + buf * 3 * T;
    } else {
      acquire(tl, next);
    }
  };
  auto tile_end = [&]() {
    if constexpr (SPEC) {
      __syncwarp();
      if (lane == 0) mbar_arrive(bar + 3 + (cseq & 1u));
      ++cseq;
    }
  };
  if constexpr (SPEC) {
    if (warp == CW) {
      // ---- producer warp --------------------------------------------------------------------------------------------
      uint32_t pseq = 0;
      auto produce = [&](int npass) {
        const int total = npass * nt;
        if (a.tma && lane == 0 && total > 0) issue_tile(t_begin);
        int ti = 0;
        for (int p = 0; p < total; ++p, ++pseq) {
          const uint32_t buf = pseq & 1u;
          if (a.tma) {
            while (!mbar_try_wait(bar, parity)) {}
            parity ^= 1u;
          }
          while (!mbar_try_wait(bar + 3 + buf, ((pseq >> 1) & 1u) ^ 1u)) {}  // the buffer's previous tile is consumed
          planes = planes0 + buf * 3 * T;
          fill_planes(t_begin + ti);
          ti = ti + 1 == nt ? 0 : ti + 1;
          __syncwarp();
          if (lane == 0) {
            mbar_arrive(bar + 1 + buf);
            if (a.tma && p + 1 < total) {
              fence_proxy_async();
              issue_tile(t_begin + ti);
            }
          }
          __syncwarp();
        }
      };
      produce(2);  // pass 1 and pass 2 stream the chunk's tiles
      for (int qi = 0; qi < QW; ++qi)
        if (__syncthreads_or(0)) produce(1);  // exact fallback of some warp's query: one more sweep
      return;
    }
  }

  // ---- this warp's queries ------------------------------------------------------------------------------------------
  const int qbase = (blockIdx.x * CW + warp) * QW;
  float q0[QW], q1[QW], q2[QW];
  float2 qx2[QW], qy2[QW], qz2[QW];
#pragma unroll
  for (int qi = 0; qi < QW; ++qi) {
    const int qidx = qbase + qi;
    q0[qi] = q1[qi] = q2[qi] = 0.f;
    if (qidx < q) {
      if (PLANAR) {
        q0[qi] = __ldg(Qp + qidx), q1[qi] = __ldg(Qp + r + qidx), q2[qi] = __ldg(Qp + 2 * r + qidx);
      } else {
        q0[qi] = __ldg(Qp + 3 * qidx), q1[qi] = __ldg(Qp + 3 * qidx + 1), q2[qi] = __ldg(Qp + 3 * qidx + 2);
      }
    }
    qx2[qi] = make_float2(q0[qi], q0[qi]), qy2[qi] = make_float2(q1[qi], q1[qi]), qz2[qi] = make_float2(q2[qi], q2[qi]);
  }
  const float4 *px, *py, *pz;
  auto set_planes = [&]() {
    px = reinterpret_cast<const float4 *>(planes) + lane;
    py = px + (T >> 2), pz = px + (T >> 1);
  };
  set_planes();
  auto pair2 = [&](float2 X, float2 Y, float2 Z, int qi) {
    const float2 dx = sub2(X, qx2[qi]), dy = sub2(Y, qy2[qi]), dz = sub2(Z, qz2[qi]);
    return fma2(dz, dz, fma2(dy, dy, mul2(dx, dx)));
  };

  if (!SPEC && a.tma && tid == 0 && nt > 0) issue_tile(t_begin);

  // ---- pass 1: segment minima -> tau -------------------------------------------------------------------------------------
  float m[QW][E];
#pragma unroll
  for (int qi = 0; qi < QW; ++qi)
#pragma unroll
    for (int e = 0; e < E; ++e) m[qi][e] = INF;
  for (int i = 0; i < nt; ++i) {
    const int tl = t_begin + i;
    tile_begin(tl, nt > 1 ? (i + 1 < nt ? tl + 1 : t_begin) : -1);
    set_planes();
    const int nsteps = ((tile_n(tl) + 255) & ~255) >> 7;  // even
    for (int s = 0; s < nsteps; s += 2) {
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const float4 X = px[(s + h) * 32], Y = py[(s + h) * 32], Z = pz[(s + h) * 32];
#pragma unroll
        for (int qi = 0; qi < QW; ++qi) {
          const float2 dA = pair2(make_float2(X.x, X.y), make_float2(Y.x, Y.y), make_float2(Z.x, Z.y), qi);
          const float2 dB = pair2(make_float2(X.z, X.w), make_float2(Y.z, Y.w), make_float2(Z.z, Z.w), qi);
          const int sa = E == 2 ? 0 : 2 * h, sb = sa + 1;
          m[qi][sa] = min3(m[qi][sa], dA.x, dA.y);
          m[qi][sb] = min3(m[qi][sb], dB.x, dB.y);
        }
      }
    }
    tile_end();
  }
  // The per-query phases below run as ROLLED loops over the warp's queries (values picked out of the register arrays
  // with select chains): the sorting networks appear once in the code instead of QW times, which keeps the kernel
  // inside the instruction cache.
  const uint32_t dir_mask = warp_sort_dir_mask(lane);
  float tau[QW];
  {
    uint32_t sv[QW][E];  // non-negative floats order like their bit patterns
#pragma unroll
    for (int qi = 0; qi < QW; ++qi)
#pragma unroll
      for (int e = 0; e < E; ++e) sv[qi][e] = __float_as_uint(m[qi][e]);
    warp_sort_u32_multi<QW, E>(sv, lane, dir_mask);
#pragma unroll
    for (int qi = 0; qi < QW; ++qi) {
      uint32_t kth = sv[qi][0];
#pragma unroll
      for (int e = 1; e < E; ++e) kth = (e == kslot) ? sv[qi][e] : kth;
      tau[qi] = __uint_as_float(__shfl_sync(FULL, kth, klane));
    }
  }

  // ---- pass 2: which 4-point steps hold a distance <= tau ------------------------------------------------------------------
  // lp = shared-window address of the lane's next free slot.  The running step number is stored unconditionally; the
  // address only advances when the step holds a candidate, so a miss is overwritten by the next step (no predicated
  // store, no branch).  The lists span all tiles of the chunk: tau is final, so they stay ~k entries per query.
  const uint32_t lbase_s = smem_u32(my_area) + 2 * lane;  // slot LC of a list only absorbs the stores of a full list
  uint32_t lp[QW], lend[QW];
#pragma unroll
  for (int qi = 0; qi < QW; ++qi) lp[qi] = lbase_s + qi * static_cast<uint32_t>(PQ), lend[qi] = lp[qi] + LC * 64;
  for (int i = 0; i < nt; ++i) {
    const int tl = t_begin + i;
    if (SPEC || nt > 1) {
      tile_begin(tl, i + 1 < nt ? tl + 1 : -1);
      set_planes();
    }
    const int nsteps = ((tile_n(tl) + 255) & ~255) >> 7;
    const int gs0 = i * (T >> 7);  // step number inside the chunk
#pragma unroll 2
    for (int s = 0; s < nsteps; ++s) {
      const float4 X = px[s * 32], Y = py[s * 32], Z = pz[s * 32];
      const int gs = gs0 + s;
#pragma unroll
      for (int qi = 0; qi < QW; ++qi) {
        const float2 dA = pair2(make_float2(X.x, X.y), make_float2(Y.x, Y.y), make_float2(Z.x, Z.y), qi);
        const float2 dB = pair2(make_float2(X.z, X.w), make_float2(Y.z, Y.w), make_float2(Z.z, Z.w), qi);
        const float mm = min3(dA.x, dA.y, fminf(dB.x, dB.y));
        asm volatile("st.shared.u16 [%0], %1;" ::"r"(lp[qi]), "r"(gs) : "memory");
        if (mm <= tau[qi]) lp[qi] = min(lp[qi] + 64u, lend[qi]);
      }
    }
    tile_end();
  }
  __syncwarp();

  // ---- rescan: the recorded quads, compacted across the warp, re-evaluated from global memory -------------------------------
  // (one quad per lane and round; ~k quads per query, L2 hits).  Qualifying points go to the query's key queue.
  int qn[QW];
  bool ovf[QW];
  const uint32_t chunk_quad0 = static_cast<uint32_t>(t_begin) * static_cast<uint32_t>(T >> 2);
  const bool vec_ok = (r & 3) == 0 && (reinterpret_cast<uintptr_t>(a.ref) & 15) == 0;
#pragma unroll 1
  for (int qi = 0; qi < QW; ++qi) {
    uint32_t lpq = lp[0];
    float tq = tau[0], f0 = q0[0], f1 = q1[0], f2 = q2[0];
#pragma unroll
    for (int j = 1; j < QW; ++j)
      if (j == qi) lpq = lp[j], tq = tau[j], f0 = q0[j], f1 = q1[j], f2 = q2[j];
    int n = 0;
    bool over = !(tq < INF);
    const int c = static_cast<int>(lpq - lbase_s - qi * static_cast<uint32_t>(PQ)) >> 6;
    over = over || __any_sync(FULL, c >= LC);  // a lane filled its list: it may have dropped steps
    int incl = c;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int t = __shfl_up_sync(FULL, incl, o);
      if (lane >= o) incl += t;
    }
    const int total = __shfl_sync(FULL, incl, 31);
    if (!over && total > 32 * LC) over = true;
    if (!over && total > 0) {
      const int maxc = __reduce_max_sync(FULL, c);
      const int off = incl - c;
      for (int it = 0; it < maxc; ++it)
        if (it < c)
          dense[off + it] = (static_cast<uint32_t>(reinterpret_cast<const unsigned short *>(my_area + qi * PQ)[it * 32 + lane]) << 5) | lane;
      __syncwarp();
      uint64_t *qq = reinterpret_cast<uint64_t *>(my_area + qi * PQ);
      for (int e0 = 0; e0 < total; e0 += 32) {
        const bool act = e0 + lane < total;
        const uint32_t quad = chunk_quad0 + (act ? dense[e0 + lane] : 0u);  // quad index inside the cloud
        const uint32_t jg = 4u * quad;
        float4 X, Y, Z;
        if (PLANAR) {
          if (vec_ok) {
            const float4 *P = reinterpret_cast<const float4 *>(R);
            X = __ldg(P + quad), Y = __ldg(P + (r >> 2) + quad), Z = __ldg(P + 2 * (r >> 2) + quad);
          } else {
            float *xs = &X.x, *ys = &Y.x, *zs = &Z.x;
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const bool in = jg + e < static_cast<uint32_t>(r);
              xs[e] = in ? __ldg(R + jg + e) : INF, ys[e] = in ? __ldg(R + r + jg + e) : 0.f;
              zs[e] = in ? __ldg(R + 2 * static_cast<size_t>(r) + jg + e) : 0.f;
            }
          }
        } else if (vec_ok) {
          const float4 *P = reinterpret_cast<const float4 *>(R) + 3 * static_cast<size_t>(quad);
          const float4 a0 = __ldg(P), a1 = __ldg(P + 1), a2 = __ldg(P + 2);
          X = make_float4(a0.x, a0.w, a1.z, a2.y);
          Y = make_float4(a0.y, a1.x, a1.w, a2.z);
          Z = make_float4(a0.z, a1.y, a2.x, a2.w);
        } else {
          float *xs = &X.x, *ys = &Y.x, *zs = &Z.x;
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const bool in = jg + e < static_cast<uint32_t>(r);
            const float *pt = R + 3 * static_cast<size_t>(in ? jg + e : 0u);
            xs[e] = in ? __ldg(pt) : INF, ys[e] = in ? __ldg(pt + 1) : 0.f, zs[e] = in ? __ldg(pt + 2) : 0.f;
          }
        }
        const float2 g0 = make_float2(f0, f0), g1 = make_float2(f1, f1), g2 = make_float2(f2, f2);
        const float2 dxa = sub2(make_float2(X.x, X.y), g0), dxb = sub2(make_float2(X.z, X.w), g0);
        const float2 dya = sub2(make_float2(Y.x, Y.y), g1), dyb = sub2(make_float2(Y.z, Y.w), g1);
        const float2 dza = sub2(make_float2(Z.x, Z.y), g2), dzb = sub2(make_float2(Z.z, Z.w), g2);
        const float2 dA = fma2(dza, dza, fma2(dya, dya, mul2(dxa, dxa)));
        const float2 dB = fma2(dzb, dzb, fma2(dyb, dyb, mul2(dxb, dxb)));
        const float dv[4] = {dA.x, dA.y, dB.x, dB.y};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const bool hit = act && dv[e] <= tq;
          const unsigned mk = __ballot_sync(FULL, hit);
          const int pos = n + __popc(mk & lt_mask);
          if (hit && pos < CAP) qq[pos] = pack_key(dv[e], jg + e);
          n += __popc(mk);
        }
      }
      __syncwarp();
      over = n > CAP;
    }
#pragma unroll
    for (int j = 0; j < QW; ++j)
      if (j == qi) qn[j] = n, ovf[j] = over;
  }
  __syncwarp();

  // ---- exact order of the candidates; queries that overflowed go to the streaming warp-select --------------------------------
  uint64_t *chunk_out = a.chunk_keys ? a.chunk_keys + (static_cast<size_t>(blockIdx.z) * gridDim.y + cloud) * q * k : nullptr;
  auto finish_query = [&](int qidx, float f0, float f1, float f2, const uint64_t (&keys)[E]) {
    if (chunk_out) {
#pragma unroll
      for (int e = 0; e < E; ++e) {
        const int p = e * 32 + lane;
        if (p < k) chunk_out[static_cast<size_t>(qidx) * k + p] = keys[e];
      }
    } else {
      knn4_emit<PLANAR, E, AFF>(a, R, cloud, qidx, f0, f1, f2, keys, lane);
    }
  };
  constexpr int TB = E == 2 ? 6 : 7;  // tag bits: position of the candidate in its queue (CAP = 64 or 128)
  // Fast order: sort 32-bit words (distance bits with the low TB bits replaced by the queue position), all queries of
  // the warp in lockstep.  That order is the exact (distance, index) order unless two of the first k+1 words agree above
  // the tag -- then, and only then, the full 64-bit keys are sorted.
  {
    uint32_t w[QW][E];
#pragma unroll
    for (int qi = 0; qi < QW; ++qi) {
      const uint64_t *qq = reinterpret_cast<const uint64_t *>(my_area + qi * PQ);
      const int n = ovf[qi] ? 0 : qn[qi];
#pragma unroll
      for (int e = 0; e < E; ++e) {
        const int p = e * 32 + lane;
        w[qi][e] = p < n ? ((static_cast<uint32_t>(qq[p] >> 32) & ~((1u << TB) - 1u)) | static_cast<uint32_t>(p)) : 0xffffffffu;
      }
    }
    warp_sort_u32_multi<QW, E>(w, lane, dir_mask);
#pragma unroll
    for (int qi = 0; qi < QW; ++qi) {
      const int qidx = qbase + qi;
      if (ovf[qi] || qidx >= q) continue;  // warp-uniform
      const uint64_t *qq = reinterpret_cast<const uint64_t *>(my_area + qi * PQ);
      bool amb = false;
#pragma unroll
      for (int e = 0; e < E; ++e) {
        uint32_t nxt = __shfl_down_sync(FULL, w[qi][e], 1);
        const uint32_t head = __shfl_sync(FULL, w[qi][e + 1 < E ? e + 1 : e], 0);
        if (lane == 31) nxt = e + 1 < E ? head : 0xffffffffu;
        amb |= (e * 32 + lane < k) && (w[qi][e] >> TB) == (nxt >> TB);
      }
      uint64_t keys[E];
      if (!__any_sync(FULL, amb)) {
#pragma unroll
        for (int e = 0; e < E; ++e) keys[e] = w[qi][e] == 0xffffffffu ? KEY_INF : qq[w[qi][e] & ((1u << TB) - 1u)];
      } else {
#pragma unroll
        for (int e = 0; e < E; ++e) keys[e] = (e * 32 + lane) < qn[qi] ? qq[e * 32 + lane] : KEY_INF;
        warp_sort_multi<E>(keys, lane);
      }
      finish_query(qidx, q0[qi], q1[qi], q2[qi], keys);
    }
  }
#pragma unroll 1
  for (int qi = 0; qi < QW; ++qi) {
    bool flagged = ovf[0];
    float f0 = q0[0], f1 = q1[0], f2 = q2[0];
#pragma unroll
    for (int j = 1; j < QW; ++j)
      if (j == qi) flagged = ovf[j], f0 = q0[j], f1 = q1[j], f2 = q2[j];
    const bool mine = flagged && qbase + qi < q;
    if (!__syncthreads_or(mine)) continue;  // the tiles are re-streamed by the whole CTA
    WarpSelect<NS> sel;
    sel.init();
    uint64_t *wq = reinterpret_cast<uint64_t *>(my_area);  // 64 entries: the region of the warp's first query (CAP >= 64)
    if (!SPEC && a.tma && nt > 1 && tid == 0) issue_tile(t_begin);
    for (int i = 0; i < nt; ++i) {
      const int tl = t_begin + i;
      if (SPEC || nt > 1) tile_begin(tl, i + 1 < nt ? tl + 1 : -1);
      if (mine) {
        const int tn = tile_n(tl);
        const float *sx = planes, *sy = planes + T, *sz = planes + 2 * T;
        for (int j0 = 0; j0 < tn; j0 += 32) {
          const int j = j0 + lane;
          const bool in = j < tn;
          const float d = dist_seq3(__fsub_rn(sx[in ? j : 0], f0), __fsub_rn(sy[in ? j : 0], f1), __fsub_rn(sz[in ? j : 0], f2));
          const uint64_t key = pack_key(d, static_cast<uint32_t>(tl * T + j));
          sel.offer(in && key < sel.tau, key, wq, lane, kslot, klane);
        }
      }
      if (SPEC || nt > 1) tile_end();
    }
    if (mine) {
      sel.finish(wq, lane);
      uint64_t keys[E];
#pragma unroll
      for (int e = 0; e < E; ++e) keys[e] = e < NS ? sel.L[e < NS ? e : 0] : KEY_INF;
      finish_query(qbase + qi, f0, f1, f2, keys);
    }
  }
}

// warp per query: merge the chunks' ascending key lists (chunk z holds reference points [z*len, (z+1)*len), keys carry
// cloud-wide indices) and run the common epilogue
template <bool PLANAR, int E, bool AFF>
__global__ void __launch_bounds__(128) knn4_merge_kernel(const Knn4Args a, int nz, int b) {
  const int lane = threadIdx.x & 31;
  const long long w = (static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  if (w >= static_cast<long long>(b) * a.q) return;
  const int cloud = static_cast<int>(w / a.q), qidx = static_cast<int>(w - static_cast<long long>(cloud) * a.q);
  const int k = a.k, r = a.r;
  uint64_t L[E];
#pragma unroll
  for (int e = 0; e < E; ++e) L[e] = KEY_INF;
  for (int z = 0; z < nz; ++z) {
    const uint64_t *src = a.chunk_keys + ((static_cast<size_t>(z) * b + cloud) * a.q + qidx) * k;
    for (int p0 = 0; p0 < k; p0 += 32) {
      const uint64_t c = (p0 + lane) < k ? src[p0 + lane] : KEY_INF;
      warp_merge<E>(L, c, lane);
    }
  }
  const float *__restrict__ R = a.ref + static_cast<size_t>(cloud) * r * 3;
  float q0, q1, q2;
  if (PLANAR) {
    q0 = __ldg(R + qidx), q1 = __ldg(R + r + qidx), q2 = __ldg(R + 2 * r + qidx);
  } else {
    const float *Q = a.query + (static_cast<size_t>(cloud) * a.q + qidx) * 3;
    q0 = __ldg(Q), q1 = __ldg(Q + 1), q2 = __ldg(Q + 2);
  }
  knn4_emit<PLANAR, E, AFF>(a, R, cloud, qidx, q0, q1, q2, L, lane);
}

// ---- host side ---------------------------------------------------------------------------------------------------------
struct Knn4Plan {
  int qw, nw, tile, nz, tma, spec, dense_in_stage;
};

// The (queries per warp, warps per CTA, warp-specialised) forms the plan chooses from, numbered as pdae_tune_knn takes them.
struct Knn4Form {
  int qw, nw, spec;
};
constexpr int KNN4_NFORMS = 4;
static constexpr Knn4Form KNN4_FORMS[KNN4_NFORMS] = {{4, 8, 1}, {4, 8, 0}, {4, 4, 0}, {2, 4, 0}};

// Tuning hook (profiles/tune_knn.py, tests/test_gpu_knn4.py): pdae_tune_knn overrides the plan; -1 = automatic.
struct Knn4Tune {
  int form, tile, nz, tma;
};
static Knn4Tune knn4_tune{-1, -1, -1, -1};

static size_t knn4_smem_bytes(int e, const Knn4Plan &p) {
  const size_t per_warp = e == 2 ? Knn4Smem<2>::per_warp(p.qw, p.dense_in_stage) : Knn4Smem<4>::per_warp(p.qw, p.dense_in_stage);
  const int cw = p.spec ? p.nw - 1 : p.nw;
  return 128 + static_cast<size_t>((p.spec ? 24 : 12) + (p.tma ? 12 : 0)) * p.tile + static_cast<size_t>(cw) * per_warp;
}

static Knn4Plan knn4_plan(int b, int r, int q, int k, bool aligned, bool have_ws) {
  Knn4Plan p;
  const int e = k <= 32 ? 2 : 4;
  const Knn4Tune &tn = knn4_tune;
  // streamed clouds that cannot fill the GPU with CTAs (scene scale: few queries, long cloud): warp-specialised CTAs
  // (7 compute warps + 1 producer, two plane buffers) keep the lone CTA of an SM computing while tiles are converted;
  // with several CTAs per SM the conversions already overlap with other CTAs' scans and the eighth compute warp wins
  // (measured, profiles/r02/tune_knn_v5.json: C4 611 vs 690 us, C5 161 vs 142 us)
  const bool streamed = r > 2048;
  const long long ctas_plain = static_cast<long long>(b) * ((q + 31) / 32);
  p.spec = streamed && ctas_plain < 148 * 3 ? 1 : 0;
  p.tile = tn.tile > 0 ? tn.tile : 2048;
  if (p.tile < 256) p.tile = 256;
  p.tile = (p.tile + 255) & ~255;
  const int r256 = (r + 255) & ~255;
  if (r256 < p.tile) p.tile = r256;
  const int ntiles = (r + p.tile - 1) / p.tile;
  // queries per warp / warps per CTA: a CTA stages the tile once for qw*nw queries; keep a few CTAs per SM in flight
  const long long nq = static_cast<long long>(b) * q;
  p.qw = nq >= 148LL * 4 * 8 ? 4 : 2;
  p.nw = 4;
  if (q >= 256 && nq >= 148LL * 8 * 4 * 2) p.nw = 8;
  if (streamed) p.qw = 4, p.nw = 8;
  if (tn.form >= 0) p.qw = KNN4_FORMS[tn.form].qw, p.nw = KNN4_FORMS[tn.form].nw, p.spec = KNN4_FORMS[tn.form].spec;
  // the TMA landing zone costs a tile of shared memory: worth it only when tiles are streamed
  p.tma = aligned && (r & 3) == 0 && ntiles > 1;
  if (tn.tma >= 0) p.tma = tn.tma;
  if (!aligned || (r & 3) != 0) p.tma = 0;
  // the idle landing zone holds the rescan's dense lists when they fit
  const int cw = p.spec ? p.nw - 1 : p.nw;
  p.dense_in_stage = p.tma && 12 * p.tile >= cw * 32 * (5 * e) * 4;
  // chunks along the reference cloud: waves x (two passes over the chunk's tiles + the per-chunk selection work)
  p.nz = 1;
  const int qpc = cw * p.qw;  // queries per CTA
  if (have_ws && ntiles > 1) {
    // CTAs that share an SM share its issue slots: count waves against the SMs, not against the resident slots
    const long long slots = 148;
    const long long ctas1 = static_cast<long long>(b) * ((q + qpc - 1) / qpc);
    const double tiles2k = p.tile / 2048.0;  // cost unit: one pass over 2048 points
    double best = 1e30;
    for (int nz = 1; nz <= 16 && nz <= ntiles; ++nz) {
      const int tpc = (ntiles + nz - 1) / nz;
      const int nz_eff = (ntiles + tpc - 1) / tpc;
      if (nz_eff != nz) continue;
      const long long waves = (ctas1 * nz + slots - 1) / slots;
      const double cost = static_cast<double>(waves) * (2.0 * tpc * tiles2k + (e == 2 ? 3.0 : 6.0)) + (nz > 1 ? 0.5 : 0.0);
      if (cost < best * 0.97) best = cost, p.nz = nz;
    }
  }
  if (tn.nz > 0 && have_ws) {
    const int tpc = (ntiles + tn.nz - 1) / tn.nz;
    p.nz = (ntiles + tpc - 1) / tpc;
    if (p.nz > 16) p.nz = 16;
  }
  return p;
}

template <bool PLANAR, int E, int QW, int NW, bool AFF, bool SPEC>
static int knn4_launch_cfg(Knn4Args a, int b, const Knn4Plan &p, cudaStream_t st) {
  const size_t smem = knn4_smem_bytes(E, p);
  static int configured = 0;  // per instantiation; the attribute is sticky per device function
  if (smem > 48 * 1024 && static_cast<int>(smem) > configured) {
    PDAE_CUDA_TRY(cudaFuncSetAttribute(knn4_kernel<PLANAR, E, QW, NW, AFF, SPEC>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       static_cast<int>(smem)));
    configured = static_cast<int>(smem);
  }
  const dim3 grid(ceil_div(a.q, (SPEC ? NW - 1 : NW) * QW), b, p.nz);
  knn4_kernel<PLANAR, E, QW, NW, AFF, SPEC><<<grid, NW * 32, smem, st>>>(a);
  PDAE_RETURN_IF_LAUNCH_FAILED();
  if (p.nz > 1) {
    const long long warps = static_cast<long long>(b) * a.q;
    knn4_merge_kernel<PLANAR, E, AFF><<<static_cast<unsigned>((warps + 3) / 4), 128, 0, st>>>(a, p.nz, b);
    PDAE_RETURN_IF_LAUNCH_FAILED();
  }
  return 0;
}

template <bool PLANAR, int E, bool AFF>
static int knn4_launch_e(const Knn4Args &a, int b, const Knn4Plan &p, cudaStream_t st) {
  // the plan yields one of KNN4_FORMS
  if (p.spec) return knn4_launch_cfg<PLANAR, E, 4, 8, AFF, true>(a, b, p, st);
  if (p.nw == 8) return knn4_launch_cfg<PLANAR, E, 4, 8, AFF, false>(a, b, p, st);
  if (p.qw == 4) return knn4_launch_cfg<PLANAR, E, 4, 4, AFF, false>(a, b, p, st);
  return knn4_launch_cfg<PLANAR, E, 2, 4, AFF, false>(a, b, p, st);
}

size_t knn4_workspace_bytes(int b, int r, int q, int k) {
  if (b <= 0 || q <= 0 || k <= 0 || k > 64 || r <= 2048) return 0;
  // up to 16 chunks of k keys per query; only shapes that cannot fill the GPU otherwise ever use it
  const long long ctas = static_cast<long long>(b) * ((q + 15) / 16);
  if (ctas >= 148LL * 8) return 0;
  return static_cast<size_t>(16) * b * q * k * sizeof(uint64_t);
}

template <bool PLANAR>
static int knn4_dispatch(Knn4Args a, int b, void *ws, size_t ws_bytes, cudaStream_t st) {
  if (b > 65535) return PDAE_E_UNSUPPORTED;
  const bool aligned = (reinterpret_cast<uintptr_t>(a.ref) & 15) == 0;
  const size_t need1 = static_cast<size_t>(b) * a.q * a.k * sizeof(uint64_t);
  Knn4Plan p = knn4_plan(b, a.r, a.q, a.k, aligned, ws != nullptr && ws_bytes >= 2 * need1);
  if (p.nz > 1 && static_cast<size_t>(p.nz) * need1 > ws_bytes) {
    int nz = static_cast<int>(ws_bytes / need1);
    const int ntiles = (a.r + p.tile - 1) / p.tile;
    const int tpc = (ntiles + nz - 1) / nz;
    p.nz = (ntiles + tpc - 1) / tpc;
  }
  a.tile = p.tile;
  a.tma = p.tma;
  a.dense_in_stage = p.dense_in_stage;
  const int ntiles = (a.r + p.tile - 1) / p.tile;
  a.tiles_per_chunk = (ntiles + p.nz - 1) / p.nz;
  if (static_cast<long long>(a.tiles_per_chunk) * (p.tile >> 7) > 65535) return PDAE_E_UNSUPPORTED;  // 16-bit step numbers
  a.chunk_keys = p.nz > 1 ? static_cast<uint64_t *>(ws) : nullptr;
  if constexpr (!PLANAR) {
    if (a.aff.mats != nullptr)
      return a.k <= 32 ? knn4_launch_e<false, 2, true>(a, b, p, st) : knn4_launch_e<false, 4, true>(a, b, p, st);
  }
  return a.k <= 32 ? knn4_launch_e<PLANAR, 2, false>(a, b, p, st) : knn4_launch_e<PLANAR, 4, false>(a, b, p, st);
}

int knn4_points(const float *ref, const float *query, int b, int r, int q, int k, int out_kq, float *dist, int64_t *idx,
                float *group, cudaStream_t st, uint64_t *keys, uint32_t ref_offset, int raw_group, const GroupAffine *affine,
                void *ws, size_t ws_bytes) {
  Knn4Args a{ref, query, dist, idx, group, keys, nullptr, ref_offset, raw_group,
             affine ? *affine : GroupAffine{nullptr, 0, nullptr, nullptr}, r, q, k, 0, 0, out_kq, 0, 0};
  return knn4_dispatch<false>(a, b, ws, ws_bytes, st);
}
int knn4_planar(const float *x, int b, int n, int k, int64_t *idx, cudaStream_t st, void *ws, size_t ws_bytes) {
  Knn4Args a{x, nullptr, nullptr, idx, nullptr, nullptr, nullptr, 0u, 0, GroupAffine{nullptr, 0, nullptr, nullptr}, n, n, k,
             0, 0, 0, 0, 0};
  return knn4_dispatch<true>(a, b, ws, ws_bytes, st);
}

}  // namespace pdae

extern "C" int pdae_tune_knn(int form, int tile, int nz, int tma) {
  if (form < -1 || form >= pdae::KNN4_NFORMS) return PDAE_E_INVALID;
  pdae::knn4_tune = pdae::Knn4Tune{form, tile, nz, tma};
  return 0;
}
