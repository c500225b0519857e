// edgeconv.cu -- SURVEY.md 8f row 4, first stage: the gather half of an eval-mode EdgeConv layer of the DGCNN encoder
// (models/dgcnn_util.py:114-126: get_graph_feature -> Conv2d(2C, Co, 1, bias=False) -> BatchNorm2d -> LeakyReLU(0.2) ->
// max over the k neighbours).  With the convolution weight split as W = [W1 | W2],
//     W [x_j - x_i; x_i] = W1 x_j + (W2 - W1) x_i = P[j] + Q[i],
// and BatchNorm (running statistics) + LeakyReLU is monotone per channel, increasing where the folded scale s_o >= 0
// and decreasing where s_o < 0, so
//     max_j act(s_o (P[j][o] + Q[i][o]) + t_o) = act(s_o (ext_j P[j][o] + Q[i][o]) + t_o),  ext = max (s_o >= 0) / min.
// P and Q are two small GEMMs (library calls on the host side, N x C x Co per cloud); this kernel does the rest: per
// point it gathers the k neighbour rows of P (row-major (b, n, co): one coalesced row read per neighbour, L2-resident),
// keeps the per-channel extremum, applies the affine + activation and writes the reference's (b, co, n) layout through
// a shared-memory transpose.  The (b, 2C, n, k) graph feature and the (b, Co, n, k) convolution output never exist:
// traffic is b*n*k*co*4 bytes of gathered reads instead of writing and re-reading both tensors.
// Bound: L2 gather bandwidth.  STATUS: bit-exact with its oracle on B200 (tests/test_row4_edgeconv.py); not yet timed.
#include "common.cuh"
#include "reverse.cuh"

namespace pdae {

constexpr int EC_POINTS = 32;   // points per CTA (one output row segment of 128 bytes per channel)
constexpr int EC_WARPS = 8;     // each warp owns EC_POINTS / EC_WARPS points
constexpr int EC_CHUNK = 256;   // channels handled per pass: 8 per lane

__global__ void __launch_bounds__(EC_WARPS * 32) edge_gather_extremum_kernel(const float *__restrict__ P, const float *__restrict__ Q,
                                                                             const int64_t *__restrict__ idx,
                                                                             const float *__restrict__ scale,
                                                                             const float *__restrict__ shift, float slope, int n,
                                                                             int k, int co, float *__restrict__ out) {
  __shared__ float tile[EC_CHUNK][EC_POINTS + 1];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const size_t cloud = blockIdx.y;
  const int i0 = blockIdx.x * EC_POINTS;
  const float *__restrict__ Pc = P + cloud * n * co;
  const float *__restrict__ Qc = Q + cloud * n * co;
  const int64_t *__restrict__ Ic = idx + cloud * n * k;
  constexpr int PER_LANE = EC_CHUNK / 32;
  constexpr int PER_WARP = EC_POINTS / EC_WARPS;

  for (int c0 = 0; c0 < co; c0 += EC_CHUNK) {
    float s[PER_LANE], t[PER_LANE], sgn[PER_LANE];
#pragma unroll
    for (int u = 0; u < PER_LANE; ++u) {
      const int o = c0 + u * 32 + lane;
      s[u] = o < co ? __ldg(scale + o) : 0.0f;
      t[u] = o < co ? __ldg(shift + o) : 0.0f;
      sgn[u] = s[u] >= 0.0f ? 1.0f : -1.0f;  // ext = sgn * max_j(sgn * P): max for s >= 0, min for s < 0 (exact)
    }
    for (int pw = 0; pw < PER_WARP; ++pw) {
      const int pl = warp * PER_WARP + pw;  // point inside the CTA's segment
      const int i = i0 + pl;
      if (i < n) {  // uniform for the warp
        float acc[PER_LANE];
#pragma unroll
        for (int u = 0; u < PER_LANE; ++u) acc[u] = -__int_as_float(0x7f800000);
        for (int j = 0; j < k; ++j) {
          const size_t row = static_cast<size_t>(__ldg(Ic + static_cast<size_t>(i) * k + j)) * co;
#pragma unroll
          for (int u = 0; u < PER_LANE; ++u) {
            const int o = c0 + u * 32 + lane;
            if (o < co) acc[u] = fmaxf(acc[u], __fmul_rn(sgn[u], __ldg(Pc + row + o)));
          }
        }
#pragma unroll
        for (int u = 0; u < PER_LANE; ++u) {
          const int o = c0 + u * 32 + lane;
          if (o < co) {
            const float v = __fadd_rn(__fmul_rn(sgn[u], acc[u]), __ldg(Qc + static_cast<size_t>(i) * co + o));
            float y = __fmaf_rn(s[u], v, t[u]);
            y = y >= 0.0f ? y : __fmul_rn(y, slope);
            tile[u * 32 + lane][pl] = y;
          }
        }
      }
    }
    __syncthreads();
    // (b, co, n) layout: for every channel of the chunk, the CTA's points are contiguous
    for (int e = threadIdx.x; e < EC_CHUNK * EC_POINTS; e += EC_WARPS * 32) {
      const int ol = e / EC_POINTS, pl = e - ol * EC_POINTS;
      const int o = c0 + ol, i = i0 + pl;
      if (o < co && i < n) out[(cloud * co + o) * n + i] = tile[ol][pl];
    }
    __syncthreads();
  }
}

}  // namespace pdae

using namespace pdae;

extern "C" int pdae_edge_gather_extremum_f32(const float *p, const float *q, const int64_t *idx, const float *scale,
                                             const float *shift, float slope, int b, int n, int k, int co, float *out,
                                             pdae_stream_t stream) {
  if (b < 0 || n < 0 || k <= 0 || co <= 0) return PDAE_E_INVALID;
  if (b == 0 || n == 0) return 0;
  if (!p || !q || !idx || !scale || !shift || !out) return PDAE_E_INVALID;
  if (b > 65535) return PDAE_E_UNSUPPORTED;
  const dim3 grid(static_cast<unsigned>((n + EC_POINTS - 1) / EC_POINTS), static_cast<unsigned>(b));
  edge_gather_extremum_kernel<<<grid, EC_WARPS * 32, 0, static_cast<cudaStream_t>(stream)>>>(p, q, idx, scale, shift, slope, n, k,
                                                                                          co, out);
  PDAE_RETURN_IF_LAUNCH_FAILED();
  return 0;
}

// ======================================================================================================================
// Second stage (training mode + backward): the same layer on a point-major product Z = [P | Q] (b, n, 2*co) that
// pdae_conv1x1_tf32x3_f32 writes (tensor cores), with BatchNorm batch statistics from gather sums and the backward pass
// through the maximum, LeakyReLU, BatchNorm and the gather.  With y[i][j][o] = P[idx(i,j)][o] + Q[i][o]:
//   statistics   sum_j y = s1 + k q,   sum_j y^2 = s2 + 2 q s1 + k q^2     (s1 = sum_j p_j, s2 = sum_j p_j^2)
//   forward      out[o][i] = act(scale_o (ext_j p_j + q) + shift_o), jstar = first slot attaining the extremum
//   backward     dbn = g * act'(bn*) on the selected edge;  dbeta = sum dbn,  dgamma = sum dbn * yhat*;
//                training-mode BatchNorm spreads two per-channel terms over EVERY edge:
//                  dy[i][j] = invstd (gamma dbn [j = jstar] - A - Bc yhat[i][j]),  A = gamma dbeta / M, Bc = gamma dgamma / M
//                (eval-mode BatchNorm: A = Bc = 0, only the selected edges carry gradient);
//                dP[idx(i,j)] += dy[i][j] (RED.ADD rows, coalesced over the channels), dQ[i] = sum_j dy[i][j].
// All kernels: one warp per point, lanes over the channels (8 per lane and 256-channel pass), neighbour rows read as
// coalesced row segments (L2 resident).
namespace pdae {

struct EdgeArgs {
  const float *z;        // (b, n, ld): P = z[..., 0:co], Q = z[..., co:2co]
  const int64_t *idx;    // (b, n, k) per-cloud neighbour indices
  int ld, n, k, co;
};

__device__ __forceinline__ void edge_block_sums_to_global(double (&a)[EC_CHUNK / 32], double (&c)[EC_CHUNK / 32], double *sm, int c0,
                                                          int co, double *__restrict__ partial) {
  // sm: [2][EC_CHUNK] doubles, zeroed by the caller before the warps add their lanes' sums
  const int lane = threadIdx.x & 31;
#pragma unroll
  for (int u = 0; u < EC_CHUNK / 32; ++u) {
    atomicAdd(sm + u * 32 + lane, a[u]);
    atomicAdd(sm + EC_CHUNK + u * 32 + lane, c[u]);
  }
  __syncthreads();
  for (int e = threadIdx.x; e < EC_CHUNK; e += EC_WARPS * 32) {
    const int o = c0 + e;
    if (o < co) {
      double *dst = partial + (static_cast<size_t>(blockIdx.y) * gridDim.x + blockIdx.x) * co * 2 + static_cast<size_t>(o) * 2;
      dst[0] = sm[e], dst[1] = sm[EC_CHUNK + e];
    }
  }
  __syncthreads();
}

// SHIFTED: the sums are of v = y - c_o instead of y, c_o = P[0][o] + Q[0][o] of cloud 0 (fp32, one sample of the
// channel).  sum y^2 / M - mean^2 cancels most significant digits when a channel's mean is large against its spread
// (5.4e-5 relative error of invstd for a unit cloud shifted by 20, measured on B200); the shifted sums keep that error
// at the rounding of P and Q themselves.  Per point the kernel forms q_i - c_o once; sum_j v = s1 + k (q_i - c_o),
// sum_j v^2 costs one more FADD per edge and channel.
template <bool SHIFTED>
__global__ void __launch_bounds__(EC_WARPS * 32) edge_stats_kernel(const EdgeArgs a, double *__restrict__ partial,
                                                                   float *__restrict__ s1_out /*(b, n, co) or NULL*/) {
  __shared__ double sm[2 * EC_CHUNK];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const size_t cloud = blockIdx.y;
  const int i0 = blockIdx.x * EC_POINTS, n = a.n, k = a.k, co = a.co, ld = a.ld;
  const float *__restrict__ Z = a.z + cloud * n * ld;
  const int64_t *__restrict__ Ic = a.idx + cloud * n * k;
  constexpr int PER_LANE = EC_CHUNK / 32, PER_WARP = EC_POINTS / EC_WARPS;
  const float kf = static_cast<float>(k);
  for (int c0 = 0; c0 < co; c0 += EC_CHUNK) {
    for (int e = threadIdx.x; e < 2 * EC_CHUNK; e += EC_WARPS * 32) sm[e] = 0.0;
    __syncthreads();
    double t1[PER_LANE], t2[PER_LANE];
    float cz[PER_LANE];  // c_o of the shifted form, read once per channel pass
#pragma unroll
    for (int u = 0; u < PER_LANE; ++u) {
      t1[u] = 0.0, t2[u] = 0.0;
      const int o = c0 + u * 32 + lane, oc = o < co ? o : co - 1;
      cz[u] = SHIFTED ? __fadd_rn(__ldg(a.z + oc), __ldg(a.z + co + oc)) : 0.f;
    }
    for (int pw = 0; pw < PER_WARP; ++pw) {
      const int i = i0 + warp * PER_WARP + pw;
      if (i >= n) continue;  // warp-uniform
      float s1[PER_LANE], s2[PER_LANE];
      int oc[PER_LANE];
      float qs[PER_LANE];  // q_i - c_o (shifted) or 0: v = p + qs
#pragma unroll
      for (int u = 0; u < PER_LANE; ++u) {
        s1[u] = 0.f, s2[u] = 0.f;
        const int o = c0 + u * 32 + lane;
        oc[u] = o < co ? o : co - 1;
        qs[u] = SHIFTED ? __fsub_rn(__ldg(Z + static_cast<size_t>(i) * ld + co + oc[u]), cz[u]) : 0.f;
      }
      const int64_t *ip = Ic + static_cast<size_t>(i) * k;
      int j = 0;
      for (; j + 4 <= k; j += 4) {
        size_t row[4];
#pragma unroll
        for (int t = 0; t < 4; ++t) row[t] = static_cast<size_t>(__ldg(ip + j + t)) * ld;
        float pv[4][PER_LANE];
#pragma unroll
        for (int t = 0; t < 4; ++t)
#pragma unroll
          for (int u = 0; u < PER_LANE; ++u) pv[t][u] = __ldg(Z + row[t] + oc[u]);
#pragma unroll
        for (int t = 0; t < 4; ++t)
#pragma unroll
          for (int u = 0; u < PER_LANE; ++u) {
            s1[u] += pv[t][u];
            const float v = SHIFTED ? __fadd_rn(pv[t][u], qs[u]) : pv[t][u];
            s2[u] = fmaf(v, v, s2[u]);
          }
      }
      for (; j < k; ++j) {
        const size_t row = static_cast<size_t>(__ldg(ip + j)) * ld;
#pragma unroll
        for (int u = 0; u < PER_LANE; ++u) {
          const float p = __ldg(Z + row + oc[u]);
          s1[u] += p;
          const float v = SHIFTED ? __fadd_rn(p, qs[u]) : p;
          s2[u] = fmaf(v, v, s2[u]);
        }
      }
#pragma unroll
      for (int u = 0; u < PER_LANE; ++u) {
        const int o = c0 + u * 32 + lane;
        if (o < co) {
          if (s1_out) s1_out[(cloud * n + i) * co + o] = s1[u];  // sum_j P[idx(i,j)]: the backward's dQ needs it
          if (SHIFTED) {
            t1[u] += static_cast<double>(s1[u]) + kf * static_cast<double>(qs[u]);
            t2[u] += static_cast<double>(s2[u]);
          } else {
            const double q = static_cast<double>(__ldg(Z + static_cast<size_t>(i) * ld + co + o));
            t1[u] += static_cast<double>(s1[u]) + kf * q;
            t2[u] += static_cast<double>(s2[u]) + 2.0 * q * static_cast<double>(s1[u]) + kf * q * q;
          }
        }
      }
    }
    edge_block_sums_to_global(t1, t2, sm, c0, co, partial);
  }
}

// forward on point-major Z: out (b, co, n) like the reference, jstar (b, n, co) = neighbour slot of the extremum
__global__ void __launch_bounds__(EC_WARPS * 32) edge_forward_kernel(const EdgeArgs a, const float *__restrict__ scale,
                                                                     const float *__restrict__ shift, float slope,
                                                                     float *__restrict__ out, unsigned char *__restrict__ jstar) {
  __shared__ float tile[EC_CHUNK][EC_POINTS + 1];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const size_t cloud = blockIdx.y;
  const int i0 = blockIdx.x * EC_POINTS, n = a.n, k = a.k, co = a.co, ld = a.ld;
  const float *__restrict__ Z = a.z + cloud * n * ld;
  const int64_t *__restrict__ Ic = a.idx + cloud * n * k;
  constexpr int PER_LANE = EC_CHUNK / 32, PER_WARP = EC_POINTS / EC_WARPS;
  for (int c0 = 0; c0 < co; c0 += EC_CHUNK) {
    float s[PER_LANE], t[PER_LANE], sgn[PER_LANE];
#pragma unroll
    for (int u = 0; u < PER_LANE; ++u) {
      const int o = c0 + u * 32 + lane;
      s[u] = o < co ? __ldg(scale + o) : 0.0f;
      t[u] = o < co ? __ldg(shift + o) : 0.0f;
      sgn[u] = s[u] >= 0.0f ? 1.0f : -1.0f;
    }
    for (int pw = 0; pw < PER_WARP; ++pw) {
      const int pl = warp * PER_WARP + pw, i = i0 + pl;
      if (i >= n) continue;
      float acc[PER_LANE];
      int js[PER_LANE];
      int oc[PER_LANE];  // channel, clamped into the row: lanes past co read a valid element and drop the result
#pragma unroll
      for (int u = 0; u < PER_LANE; ++u) {
        acc[u] = -__int_as_float(0x7f800000), js[u] = 0;
        const int o = c0 + u * 32 + lane;
        oc[u] = o < co ? o : co - 1;
      }
      const int64_t *ip = Ic + static_cast<size_t>(i) * k;
      int j = 0;
      for (; j + 4 <= k; j += 4) {  // four neighbour rows in flight
        size_t row[4];
#pragma unroll
        for (int t = 0; t < 4; ++t) row[t] = static_cast<size_t>(__ldg(ip + j + t)) * ld;
        float pv[4][PER_LANE];
#pragma unroll
        for (int t = 0; t < 4; ++t)
#pragma unroll
          for (int u = 0; u < PER_LANE; ++u) pv[t][u] = __ldg(Z + row[t] + oc[u]);
#pragma unroll
        for (int t = 0; t < 4; ++t)
#pragma unroll
          for (int u = 0; u < PER_LANE; ++u) {
            const float v = __fmul_rn(sgn[u], pv[t][u]);
            const bool gt = v > acc[u];  // strict: the first slot attaining the extremum
            acc[u] = gt ? v : acc[u];
            js[u] = gt ? j + t : js[u];
          }
      }
      for (; j < k; ++j) {
        const size_t row = static_cast<size_t>(__ldg(ip + j)) * ld;
#pragma unroll
        for (int u = 0; u < PER_LANE; ++u) {
          const float v = __fmul_rn(sgn[u], __ldg(Z + row + oc[u]));
          const bool gt = v > acc[u];
          acc[u] = gt ? v : acc[u];
          js[u] = gt ? j : js[u];
        }
      }
#pragma unroll
      for (int u = 0; u < PER_LANE; ++u) {
        const int o = c0 + u * 32 + lane;
        if (o < co) {
          const float v = __fadd_rn(__fmul_rn(sgn[u], acc[u]), __ldg(Z + static_cast<size_t>(i) * ld + co + o));
          float y = __fmaf_rn(s[u], v, t[u]);
          y = y >= 0.0f ? y : __fmul_rn(y, slope);
          tile[u * 32 + lane][pl] = y;
          if (jstar) jstar[(cloud * n + i) * co + o] = static_cast<unsigned char>(js[u]);
        }
      }
    }
    __syncthreads();
    for (int e = threadIdx.x; e < EC_CHUNK * EC_POINTS; e += EC_WARPS * 32) {
      const int ol = e / EC_POINTS, pl = e - ol * EC_POINTS;
      const int o = c0 + ol, i = i0 + pl;
      if (o < co && i < n) out[(cloud * co + o) * n + i] = tile[ol][pl];
    }
    __syncthreads();
  }
}

struct EdgeBwdArgs {
  const unsigned char *jstar;  // (b, n, co)
  const float *g;              // (b, n, co): upstream gradient, point-major
  const float *scale, *shift;  // folded BatchNorm used in the forward
  const float *mean, *invstd;  // statistics used in the forward
  const float *gamma;          // BatchNorm weight
  const float *ca, *cb;        // A, Bc per channel (zeros for eval-mode BatchNorm)
  float slope;
  int train;
};

// per-channel sums of dbn and dbn * yhat* (-> dbeta, dgamma)
// dz != NULL (zero-filled by the caller): the selected edges' term gamma * dbn is also stored into the Q half (point i) and
// scatter-added into the P half (point idx(i, jstar)) -- b*n*co atomics; eval-mode BatchNorm (train = 0) scales by invstd
// and is then complete, training mode is finished by edge_backward_dense_kernel.
__global__ void __launch_bounds__(EC_WARPS * 32) edge_backward_reduce_kernel(const EdgeArgs a, const EdgeBwdArgs w,
                                                                             double *__restrict__ partial, float *__restrict__ dz) {
  __shared__ double sm[2 * EC_CHUNK];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const size_t cloud = blockIdx.y;
  const int i0 = blockIdx.x * EC_POINTS, n = a.n, k = a.k, co = a.co, ld = a.ld;
  const float *__restrict__ Z = a.z + cloud * n * ld;
  const int64_t *__restrict__ Ic = a.idx + cloud * n * k;
  constexpr int PER_LANE = EC_CHUNK / 32, PER_WARP = EC_POINTS / EC_WARPS;
  for (int c0 = 0; c0 < co; c0 += EC_CHUNK) {
    for (int e = threadIdx.x; e < 2 * EC_CHUNK; e += EC_WARPS * 32) sm[e] = 0.0;
    __syncthreads();
    double t1[PER_LANE], t2[PER_LANE];
#pragma unroll
    for (int u = 0; u < PER_LANE; ++u) t1[u] = 0.0, t2[u] = 0.0;
    for (int pw = 0; pw < PER_WARP; ++pw) {
      const int i = i0 + warp * PER_WARP + pw;
      if (i >= n) continue;
#pragma unroll
      for (int u = 0; u < PER_LANE; ++u) {
        const int o = c0 + u * 32 + lane;
        if (o < co) {
          const size_t e = (cloud * n + i) * co + o;
          const int js = w.jstar[e];
          const size_t row = static_cast<size_t>(__ldg(Ic + static_cast<size_t>(i) * k + js)) * ld;
          const float y = __fadd_rn(__ldg(Z + row + o), __ldg(Z + static_cast<size_t>(i) * ld + co + o));
          const float bn = __fmaf_rn(__ldg(w.scale + o), y, __ldg(w.shift + o));
          const float dbn = __ldg(w.g + e) * (bn > 0.0f ? 1.0f : w.slope);
          const float yhat = (y - __ldg(w.mean + o)) * __ldg(w.invstd + o);
          t1[u] += static_cast<double>(dbn);
          t2[u] += static_cast<double>(dbn) * static_cast<double>(yhat);
          if (dz) {
            const float dsel = __ldg(w.gamma + o) * dbn * (w.train ? 1.0f : __ldg(w.invstd + o));
            float *DZ = dz + cloud * n * ld;
            DZ[static_cast<size_t>(i) * ld + co + o] = dsel;
            atomicAdd(DZ + row + o, dsel);
          }
        }
      }
    }
    edge_block_sums_to_global(t1, t2, sm, c0, co, partial);
  }
}

// dZ = [dP | dQ] (b, n, 2*co), zero-filled by the caller
__global__ void __launch_bounds__(EC_WARPS * 32) edge_backward_kernel(const EdgeArgs a, const EdgeBwdArgs w, float *__restrict__ dz) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const size_t cloud = blockIdx.y;
  const int i0 = blockIdx.x * EC_POINTS, n = a.n, k = a.k, co = a.co, ld = a.ld;
  const float *__restrict__ Z = a.z + cloud * n * ld;
  float *__restrict__ DZ = dz + cloud * n * ld;
  const int64_t *__restrict__ Ic = a.idx + cloud * n * k;
  constexpr int PER_LANE = EC_CHUNK / 32, PER_WARP = EC_POINTS / EC_WARPS;
  for (int c0 = 0; c0 < co; c0 += EC_CHUNK) {
    float sc[PER_LANE], sh[PER_LANE], mu[PER_LANE], is[PER_LANE], ga[PER_LANE], ca[PER_LANE], cb[PER_LANE];
#pragma unroll
    for (int u = 0; u < PER_LANE; ++u) {
      const int o = c0 + u * 32 + lane;
      const bool in = o < co;
      sc[u] = in ? __ldg(w.scale + o) : 0.f, sh[u] = in ? __ldg(w.shift + o) : 0.f;
      mu[u] = in ? __ldg(w.mean + o) : 0.f, is[u] = in ? __ldg(w.invstd + o) : 0.f;
      ga[u] = in ? __ldg(w.gamma + o) : 0.f, ca[u] = in ? __ldg(w.ca + o) : 0.f, cb[u] = in ? __ldg(w.cb + o) : 0.f;
    }
    for (int pw = 0; pw < PER_WARP; ++pw) {
      const int i = i0 + warp * PER_WARP + pw;
      if (i >= n) continue;
      float q[PER_LANE], dsel[PER_LANE], accq[PER_LANE];
      int js[PER_LANE];
#pragma unroll
      for (int u = 0; u < PER_LANE; ++u) {
        const int o = c0 + u * 32 + lane;
        q[u] = 0.f, dsel[u] = 0.f, accq[u] = 0.f, js[u] = 0;
        if (o < co) {
          const size_t e = (cloud * n + i) * co + o;
          js[u] = w.jstar[e];
          q[u] = __ldg(Z + static_cast<size_t>(i) * ld + co + o);
          const size_t row = static_cast<size_t>(__ldg(Ic + static_cast<size_t>(i) * k + js[u])) * ld;
          const float y = __fadd_rn(__ldg(Z + row + o), q[u]);
          const float bn = __fmaf_rn(sc[u], y, sh[u]);
          dsel[u] = ga[u] * (__ldg(w.g + e) * (bn > 0.0f ? 1.0f : w.slope));  // gamma * dbn on the selected edge
        }
      }
      if (w.train) {
        for (int j = 0; j < k; ++j) {
          const size_t row = static_cast<size_t>(__ldg(Ic + static_cast<size_t>(i) * k + j)) * ld;
#pragma unroll
          for (int u = 0; u < PER_LANE; ++u) {
            const int o = c0 + u * 32 + lane;
            if (o < co) {
              const float yhat = (__fadd_rn(__ldg(Z + row + o), q[u]) - mu[u]) * is[u];
              const float val = is[u] * ((j == js[u] ? dsel[u] : 0.f) - ca[u] - cb[u] * yhat);
              atomicAdd(DZ + row + o, val);
              accq[u] += val;
            }
          }
        }
      } else {
#pragma unroll
        for (int u = 0; u < PER_LANE; ++u) {
          const int o = c0 + u * 32 + lane;
          if (o < co) {
            const size_t row = static_cast<size_t>(__ldg(Ic + static_cast<size_t>(i) * k + js[u])) * ld;
            accq[u] = is[u] * dsel[u];
            atomicAdd(DZ + row + o, accq[u]);
          }
        }
      }
#pragma unroll
      for (int u = 0; u < PER_LANE; ++u) {
        const int o = c0 + u * 32 + lane;
        if (o < co) DZ[static_cast<size_t>(i) * ld + co + o] = accq[u];
      }
    }
  }
}

}  // namespace pdae

static int edge_check(const float *z, const int64_t *idx, int b, int n, int k, int co, int ld) {
  if (b < 0 || n < 0 || k <= 0 || co <= 0 || ld < 2 * co || k > 255) return PDAE_E_INVALID;
  if (b > 65535) return PDAE_E_UNSUPPORTED;
  if (b && n && (!z || !idx)) return PDAE_E_INVALID;
  return 0;
}

extern "C" size_t pdae_edge_partial_count(int b, int n) {
  return b <= 0 || n <= 0 ? 0 : static_cast<size_t>(b) * ((n + EC_POINTS - 1) / EC_POINTS);
}

static int edge_stats_launch(const float *z, int ld, const int64_t *idx, int b, int n, int k, int co, int shifted,
                             double *partial, float *s1, pdae_stream_t stream) {
  const int rc = edge_check(z, idx, b, n, k, co, ld);
  if (rc) return rc;
  if (b == 0 || n == 0) return 0;
  if (!partial) return PDAE_E_INVALID;
  const dim3 grid(static_cast<unsigned>((n + EC_POINTS - 1) / EC_POINTS), static_cast<unsigned>(b));
  const EdgeArgs a{z, idx, ld, n, k, co};
  if (shifted)
    edge_stats_kernel<true><<<grid, EC_WARPS * 32, 0, static_cast<cudaStream_t>(stream)>>>(a, partial, s1);
  else
    edge_stats_kernel<false><<<grid, EC_WARPS * 32, 0, static_cast<cudaStream_t>(stream)>>>(a, partial, s1);
  PDAE_RETURN_IF_LAUNCH_FAILED();
  return 0;
}

extern "C" int pdae_edge_stats_f64(const float *z, int ld, const int64_t *idx, int b, int n, int k, int co, double *partial,
                                   float *s1, pdae_stream_t stream) {
  return edge_stats_launch(z, ld, idx, b, n, k, co, 0, partial, s1, stream);
}

extern "C" int pdae_edge_stats_shifted_f64(const float *z, int ld, const int64_t *idx, int b, int n, int k, int co,
                                           double *partial, float *s1, pdae_stream_t stream) {
  return edge_stats_launch(z, ld, idx, b, n, k, co, 1, partial, s1, stream);
}

extern "C" int pdae_edge_forward_f32(const float *z, int ld, const int64_t *idx, const float *scale, const float *shift,
                                     float slope, int b, int n, int k, int co, float *out, unsigned char *jstar,
                                     pdae_stream_t stream) {
  const int rc = edge_check(z, idx, b, n, k, co, ld);
  if (rc) return rc;
  if (b == 0 || n == 0) return 0;
  if (!scale || !shift || !out) return PDAE_E_INVALID;
  const dim3 grid(static_cast<unsigned>((n + EC_POINTS - 1) / EC_POINTS), static_cast<unsigned>(b));
  edge_forward_kernel<<<grid, EC_WARPS * 32, 0, static_cast<cudaStream_t>(stream)>>>(EdgeArgs{z, idx, ld, n, k, co}, scale, shift,
                                                                                  slope, out, jstar);
  PDAE_RETURN_IF_LAUNCH_FAILED();
  return 0;
}

extern "C" int pdae_edge_backward_f32(const float *z, int ld, const int64_t *idx, const unsigned char *jstar, const float *g,
                                      const float *scale, const float *shift, const float *mean, const float *invstd,
                                      const float *gamma, const float *ca, const float *cb, float slope, int train, int b, int n,
                                      int k, int co, double *partial, float *dz, pdae_stream_t stream) {
  const int rc = edge_check(z, idx, b, n, k, co, ld);
  if (rc) return rc;
  if (b == 0 || n == 0) return 0;
  if (!jstar || !g || !scale || !shift || !mean || !invstd || !gamma) return PDAE_E_INVALID;
  if ((partial == nullptr) == (dz == nullptr)) return PDAE_E_INVALID;  // one phase per call
  const dim3 grid(static_cast<unsigned>((n + EC_POINTS - 1) / EC_POINTS), static_cast<unsigned>(b));
  const EdgeArgs a{z, idx, ld, n, k, co};
  const EdgeBwdArgs w{jstar, g, scale, shift, mean, invstd, gamma, ca, cb, slope, train};
  if (partial) {
    edge_backward_reduce_kernel<<<grid, EC_WARPS * 32, 0, static_cast<cudaStream_t>(stream)>>>(a, w, partial, nullptr);
  } else {
    if (!ca || !cb) return PDAE_E_INVALID;
    edge_backward_kernel<<<grid, EC_WARPS * 32, 0, static_cast<cudaStream_t>(stream)>>>(a, w, dz);
  }
  PDAE_RETURN_IF_LAUNCH_FAILED();
  return 0;
}

// ---- training-mode backward without one atomic per edge and channel -----------------------------------------------------------
// dy[i][j] = invstd (gamma dbn [j = jstar] - A - Bc yhat[i][j]) sums, per TARGET point p = idx(i,j), to
//   dP[p] = invstd (selected[p] - deg(p) A - Bc invstd (deg(p) (P[p] - mean) + sum_{(i,j) -> p} Q[i]))
// and per source point to  dQ[i] = invstd (gamma dbn[i] - k A - Bc invstd (s1[i] + k Q[i] - k mean)).
// `selected` is the b*n*co-atomic scatter of the reduce kernel above; the only edge-wise work left is the GATHER of Q rows
// along the reversed graph (CSR by target, built per call by three small kernels) -- coalesced row reads, no atomics on
// floats: 0.66 ms -> ~0.15 ms at 16 x 2048, k = 20, co = 256.
namespace pdae {

__global__ void __launch_bounds__(EC_WARPS * 32) edge_backward_dense_kernel(const EdgeArgs a, const float *__restrict__ s1,
                                                                            const int *__restrict__ ptr, const int *__restrict__ src,
                                                                            const float *__restrict__ mean,
                                                                            const float *__restrict__ invstd,
                                                                            const float *__restrict__ ca, const float *__restrict__ cb,
                                                                            float *__restrict__ dz) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const size_t cloud = blockIdx.y;
  const int i0 = blockIdx.x * EC_POINTS, n = a.n, k = a.k, co = a.co, ld = a.ld;
  const float *__restrict__ Z = a.z + cloud * n * ld;
  float *__restrict__ DZ = dz + cloud * n * ld;
  const int *__restrict__ P = ptr + cloud * (n + 1);
  const int *__restrict__ S = src + cloud * n * k;
  constexpr int PER_LANE = EC_CHUNK / 32, PER_WARP = EC_POINTS / EC_WARPS;
  const float kf = static_cast<float>(k);
  for (int c0 = 0; c0 < co; c0 += EC_CHUNK) {
    float mu[PER_LANE], is[PER_LANE], va[PER_LANE], vb[PER_LANE];
    int oc[PER_LANE];
#pragma unroll
    for (int u = 0; u < PER_LANE; ++u) {
      const int o = c0 + u * 32 + lane;
      oc[u] = o < co ? o : co - 1;
      mu[u] = __ldg(mean + oc[u]), is[u] = __ldg(invstd + oc[u]), va[u] = __ldg(ca + oc[u]), vb[u] = __ldg(cb + oc[u]);
    }
    for (int pw = 0; pw < PER_WARP; ++pw) {
      const int p = i0 + warp * PER_WARP + pw;
      if (p >= n) continue;
      const int e0 = __ldg(P + p), e1 = __ldg(P + p + 1);
      float rq[PER_LANE];
#pragma unroll
      for (int u = 0; u < PER_LANE; ++u) rq[u] = 0.f;
      int e = e0;
      for (; e + 4 <= e1; e += 4) {  // four source rows in flight
        size_t row[4];
#pragma unroll
        for (int t = 0; t < 4; ++t) row[t] = static_cast<size_t>(__ldg(S + e + t)) * ld + co;
#pragma unroll
        for (int t = 0; t < 4; ++t)
#pragma unroll
          for (int u = 0; u < PER_LANE; ++u) rq[u] += __ldg(Z + row[t] + oc[u]);
      }
      for (; e < e1; ++e) {
        const size_t row = static_cast<size_t>(__ldg(S + e)) * ld + co;
#pragma unroll
        for (int u = 0; u < PER_LANE; ++u) rq[u] += __ldg(Z + row + oc[u]);
      }
      const float deg = static_cast<float>(e1 - e0);
#pragma unroll
      for (int u = 0; u < PER_LANE; ++u) {
        const int o = c0 + u * 32 + lane;
        if (o < co) {
          const size_t rp = static_cast<size_t>(p) * ld;
          const float pv = __ldg(Z + rp + o), qv = __ldg(Z + rp + co + o);
          const float sel = DZ[rp + o], dsel = DZ[rp + co + o];
          const float s1v = __ldg(s1 + (cloud * n + p) * co + o);
          DZ[rp + o] = is[u] * (sel - deg * va[u] - vb[u] * is[u] * (deg * (pv - mu[u]) + rq[u]));
          DZ[rp + co + o] = is[u] * (dsel - kf * va[u] - vb[u] * is[u] * (s1v + kf * (qv - mu[u])));
        }
      }
    }
  }
}

}  // namespace pdae

extern "C" size_t pdae_edge_reverse_workspace_ints(int b, int n, int k) {
  if (b <= 0 || n <= 0 || k <= 0) return 0;
  return static_cast<size_t>(b) * (2 * static_cast<size_t>(n) + 1 + static_cast<size_t>(n) * k);
}

// phase 1 of the fused backward: partial sums of dbeta / dgamma AND the selected edges' term into dz (zero-filled)
extern "C" int pdae_edge_backward_select_f32(const float *z, int ld, const int64_t *idx, const unsigned char *jstar, const float *g,
                                             const float *scale, const float *shift, const float *mean, const float *invstd,
                                             const float *gamma, float slope, int train, int b, int n, int k, int co,
                                             double *partial, float *dz, pdae_stream_t stream) {
  const int rc = edge_check(z, idx, b, n, k, co, ld);
  if (rc) return rc;
  if (b == 0 || n == 0) return 0;
  if (!jstar || !g || !scale || !shift || !mean || !invstd || !gamma || !partial || !dz) return PDAE_E_INVALID;
  const dim3 grid(static_cast<unsigned>((n + EC_POINTS - 1) / EC_POINTS), static_cast<unsigned>(b));
  const EdgeBwdArgs w{jstar, g, scale, shift, mean, invstd, gamma, nullptr, nullptr, slope, train};
  edge_backward_reduce_kernel<<<grid, EC_WARPS * 32, 0, static_cast<cudaStream_t>(stream)>>>(EdgeArgs{z, idx, ld, n, k, co}, w, partial,
                                                                                          dz);
  PDAE_RETURN_IF_LAUNCH_FAILED();
  return 0;
}

// phase 2 (training-mode BatchNorm only): reversed graph + dense terms, dz finished in place
extern "C" int pdae_edge_backward_dense_f32(const float *z, int ld, const int64_t *idx, const float *s1, const float *mean,
                                            const float *invstd, const float *ca, const float *cb, int b, int n, int k, int co,
                                            int *workspace, size_t workspace_ints, float *dz, pdae_stream_t stream) {
  const int rc = edge_check(z, idx, b, n, k, co, ld);
  if (rc) return rc;
  if (b == 0 || n == 0) return 0;
  if (!s1 || !mean || !invstd || !ca || !cb || !dz || !workspace) return PDAE_E_INVALID;
  if (workspace_ints < pdae_edge_reverse_workspace_ints(b, n, k)) return PDAE_E_WORKSPACE;
  if (n > (1 << 24)) return PDAE_E_UNSUPPORTED;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int *cnt = workspace;                                  // (b, n): counts, then cursors
  int *ptr = cnt + static_cast<size_t>(b) * n;           // (b, n + 1)
  int *src = ptr + static_cast<size_t>(b) * (n + 1);     // (b, n * k)
  const long long total = static_cast<long long>(b) * n * k;
  if ((total + 255) / 256 > 0x7fffffffLL) return PDAE_E_UNSUPPORTED;
  if (static_cast<long long>(n) * k > 0x7fffffffLL) return PDAE_E_UNSUPPORTED;
  const int rrc = rev_csr_unordered(idx, b, n * k, n, k, cnt, ptr, src, st);  // src = the source POINT of each edge
  if (rrc) return rrc;
  const dim3 grid(static_cast<unsigned>((n + EC_POINTS - 1) / EC_POINTS), static_cast<unsigned>(b));
  edge_backward_dense_kernel<<<grid, EC_WARPS * 32, 0, st>>>(EdgeArgs{z, idx, ld, n, k, co}, s1, ptr, src, mean, invstd, ca, cb, dz);
  PDAE_RETURN_IF_LAUNCH_FAILED();
  return 0;
}

// ---- per-channel BatchNorm arithmetic in one launch each (instead of ~15 / ~8 torch micro-ops on (co)-sized tensors) -------
namespace pdae {

// partial (np, co, 2) fp64 -> batch mean / biased variance -> invstd, folded scale / shift; running buffers updated like
// nn.BatchNorm2d (momentum, unbiased variance).  train = 0: the statistics are the running buffers.
// zc != NULL: the partial sums are of y - c_o (pdae_edge_stats_shifted_f64), c_o = zc[o] + zc[co + o] in fp32.
__global__ void __launch_bounds__(128) edge_bn_prepare_kernel(const double *__restrict__ partial, int np, int co, double m,
                                                              const float *__restrict__ zc,
                                                              const float *__restrict__ gamma, const float *__restrict__ beta,
                                                              float *running_mean, float *running_var, float momentum, float eps,
                                                              int train, float *__restrict__ mean, float *__restrict__ invstd,
                                                              float *__restrict__ scale, float *__restrict__ shift) {
  const int o = blockIdx.x * blockDim.x + threadIdx.x;
  if (o >= co) return;
  float mu, var;
  if (train) {
    double s1 = 0.0, s2 = 0.0;
    for (int p = 0; p < np; ++p) {  // fixed order: deterministic
      s1 += partial[(static_cast<size_t>(p) * co + o) * 2];
      s2 += partial[(static_cast<size_t>(p) * co + o) * 2 + 1];
    }
    const double d64 = s1 / m;  // mean of the summed values
    double var64 = s2 / m - d64 * d64;
    var64 = var64 > 0.0 ? var64 : 0.0;
    const double mean64 = zc ? static_cast<double>(__fadd_rn(zc[o], zc[co + o])) + d64 : d64;
    if (running_mean) {
      running_mean[o] = (1.0f - momentum) * running_mean[o] + momentum * static_cast<float>(mean64);
      running_var[o] = (1.0f - momentum) * running_var[o] + momentum * static_cast<float>(var64 * (m / (m > 1.0 ? m - 1.0 : 1.0)));
    }
    mu = static_cast<float>(mean64), var = static_cast<float>(var64);
  } else {
    mu = running_mean[o], var = running_var[o];
  }
  const float is = rsqrtf(var + eps);
  const float g = gamma ? gamma[o] : 1.0f, bta = beta ? beta[o] : 0.0f;
  const float sc = g * is;
  mean[o] = mu, invstd[o] = is, scale[o] = sc, shift[o] = bta - sc * mu;
}

// partial (np, co, 2) fp64 of the backward's reduce phase -> dbeta, dgamma and the two per-channel terms of training-mode
// BatchNorm's backward
__global__ void __launch_bounds__(128) edge_bn_backward_kernel(const double *__restrict__ partial, int np, int co, double m,
                                                               const float *__restrict__ gamma, float *__restrict__ dgamma,
                                                               float *__restrict__ dbeta, float *__restrict__ ca,
                                                               float *__restrict__ cb) {
  const int o = blockIdx.x * blockDim.x + threadIdx.x;
  if (o >= co) return;
  double s1 = 0.0, s2 = 0.0;
  for (int p = 0; p < np; ++p) {
    s1 += partial[(static_cast<size_t>(p) * co + o) * 2];
    s2 += partial[(static_cast<size_t>(p) * co + o) * 2 + 1];
  }
  dbeta[o] = static_cast<float>(s1), dgamma[o] = static_cast<float>(s2);
  const double g = gamma[o];
  ca[o] = static_cast<float>(g * s1 / m), cb[o] = static_cast<float>(g * s2 / m);
}

}  // namespace pdae

static int edge_bn_prepare_launch(const double *partial, int np, int co, double m, const float *zc, const float *gamma,
                                  const float *beta, float *running_mean, float *running_var, float momentum, float eps, int train,
                                  float *mean, float *invstd, float *scale, float *shift, pdae_stream_t stream) {
  if (co <= 0 || np < 0 || !mean || !invstd || !scale || !shift) return PDAE_E_INVALID;
  if (train && (!partial || np == 0 || m <= 0)) return PDAE_E_INVALID;
  if (!train && (!running_mean || !running_var)) return PDAE_E_INVALID;
  edge_bn_prepare_kernel<<<(co + 127) / 128, 128, 0, static_cast<cudaStream_t>(stream)>>>(partial, np, co, m, train ? zc : nullptr,
                                                                                        gamma, beta, running_mean, running_var,
                                                                                        momentum, eps, train, mean, invstd,
                                                                                        scale, shift);
  PDAE_RETURN_IF_LAUNCH_FAILED();
  return 0;
}

extern "C" int pdae_edge_bn_prepare_f32(const double *partial, int np, int co, double m, const float *gamma, const float *beta,
                                        float *running_mean, float *running_var, float momentum, float eps, int train,
                                        float *mean, float *invstd, float *scale, float *shift, pdae_stream_t stream) {
  return edge_bn_prepare_launch(partial, np, co, m, nullptr, gamma, beta, running_mean, running_var, momentum, eps, train, mean,
                                invstd, scale, shift, stream);
}

extern "C" int pdae_edge_bn_prepare_shifted_f32(const double *partial, int np, int co, double m, const float *z, int ld,
                                                const float *gamma, const float *beta, float *running_mean, float *running_var,
                                                float momentum, float eps, int train, float *mean, float *invstd, float *scale,
                                                float *shift, pdae_stream_t stream) {
  if (train && (!z || ld < 2 * co)) return PDAE_E_INVALID;
  return edge_bn_prepare_launch(partial, np, co, m, z, gamma, beta, running_mean, running_var, momentum, eps, train, mean, invstd,
                                scale, shift, stream);
}

extern "C" int pdae_edge_bn_backward_f32(const double *partial, int np, int co, double m, const float *gamma, float *dgamma,
                                         float *dbeta, float *ca, float *cb, pdae_stream_t stream) {
  if (co <= 0 || np <= 0 || m <= 0 || !partial || !gamma || !dgamma || !dbeta || !ca || !cb) return PDAE_E_INVALID;
  edge_bn_backward_kernel<<<(co + 127) / 128, 128, 0, static_cast<cudaStream_t>(stream)>>>(partial, np, co, m, gamma, dgamma, dbeta, ca,
                                                                                         cb);
  PDAE_RETURN_IF_LAUNCH_FAILED();
  return 0;
}
