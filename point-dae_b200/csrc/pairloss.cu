// pairloss.cu -- SURVEY.md 8f row 2: the index consumers of the Chamfer match.  The reference's normal / curvature /
// position terms (extensions/chamfer_dist/__init__.py:95-120, 143-165 and the other _withnormal* classes) gather the
// matched rows with torch.gather, normalise, form differences and reduce -- about ten elementwise kernels and their
// autograd twins per term.  Here one term
//     mean_j metric(a_j, b[idx1[j]]) + mean_j metric(b_j, a[idx2[j]])
// is one forward launch (per-CTA fp64 partial sums, summed in a fixed order by the caller) and two backward launches
// (own terms stored -- which also initialises the buffers -- then the matched rows' terms scatter-added), for
//     metric 0  dis_l2                    sum (p - t)^2
//     metric 1  dis_normalized_l2         min(|u - w|^2, |u + w|^2),  u = p / max(|p|, 1e-12), w likewise
//     metric 2  dis_normalized_l1         min(sum |u - w|, sum |u + w|)
//     metric 3  dis_normalized_l2_strict  |u - w|^2
// (torch semantics: F.normalize's eps clamp, torch.min's tie splitting the gradient, sign(0) = 0 for |.|).
#include "common.cuh"
#include "reverse.cuh"

namespace pdae {

constexpr int PL_MAXD = 8;

struct PairVal {
  float v;
  float gp[PL_MAXD];  // d v / d p
  float gt[PL_MAXD];  // d v / d t
};

__device__ __forceinline__ void pl_normalize(const float *x, int d, float *u, float &inv) {
  float s = 0.f;
  for (int e = 0; e < d; ++e) s = fmaf(x[e], x[e], s);
  const float den = fmaxf(sqrtf(s), 1e-12f);
  inv = 1.0f / den;
  // true division like torch's x / norm.clamp_min(eps): a one-channel row normalises to exactly +-1 whenever sqrt(x*x) == |x|
  for (int e = 0; e < d; ++e) u[e] = __fdiv_rn(x[e], den);
}

// gradient of f(u(x)) w.r.t. x given g = df/du, u = x * inv (inv = 1 / max(|x|, eps)); below eps the map is linear
__device__ __forceinline__ void pl_normalize_bwd(const float *u, const float *g, float inv, int d, float *gx) {
  float dot = 0.f;
  for (int e = 0; e < d; ++e) dot = fmaf(u[e], g[e], dot);
  const bool clamped = inv >= 1e12f;  // |x| <= eps: u = x / eps
  for (int e = 0; e < d; ++e) gx[e] = clamped ? g[e] * inv : (g[e] - u[e] * dot) * inv;
}

template <bool GRAD>
__device__ __forceinline__ void pair_metric(const float *p, const float *t, int d, int metric, PairVal &o) {
  if (metric == 0) {
    float s = 0.f;
    for (int e = 0; e < d; ++e) {
      const float df = p[e] - t[e];
      s = fmaf(df, df, s);
      if (GRAD) o.gp[e] = 2.f * df, o.gt[e] = -2.f * df;
    }
    o.v = s;
    return;
  }
  float u[PL_MAXD], w[PL_MAXD], iu, iw;
  pl_normalize(p, d, u, iu);
  pl_normalize(t, d, w, iw);
  float vm = 0.f, vp = 0.f;  // value with w and with -w
  for (int e = 0; e < d; ++e) {
    const float a = u[e] - w[e], b = u[e] + w[e];
    if (metric == 2) vm += fabsf(a), vp += fabsf(b);
    else vm = fmaf(a, a, vm), vp = fmaf(b, b, vp);
  }
  // weights of the two branches: strict -> (1, 0); torch.min -> the smaller one, a tie splits the gradient
  float cm = 1.f, cp = 0.f;
  if (metric != 3) {
    cm = vm < vp ? 1.f : (vm == vp ? 0.5f : 0.f);
    cp = 1.f - cm;
    o.v = fminf(vm, vp);
  } else {
    o.v = vm;
  }
  if (GRAD) {
    float gu[PL_MAXD], gw[PL_MAXD];
    for (int e = 0; e < d; ++e) {
      const float a = u[e] - w[e], b = u[e] + w[e];
      float da, db;  // d(branch value) / d(a or b)
      if (metric == 2) {
        da = a > 0.f ? 1.f : (a < 0.f ? -1.f : 0.f);
        db = b > 0.f ? 1.f : (b < 0.f ? -1.f : 0.f);
      } else {
        da = 2.f * a, db = 2.f * b;
      }
      gu[e] = cm * da + cp * db;
      gw[e] = -cm * da + cp * db;
    }
    pl_normalize_bwd(u, gu, iu, d, o.gp);
    pl_normalize_bwd(w, gw, iw, d, o.gt);
  }
}

struct PairArgs {
  const float *a, *b;       // (B,N,D), (B,M,D)
  const int *idx1, *idx2;   // (B,N) into b, (B,M) into a
  int n, m, d, metric;
};

__global__ void __launch_bounds__(256) pair_loss_fwd_kernel(const PairArgs x, double *__restrict__ partial) {
  __shared__ double sm[2][8];
  const int cloud = blockIdx.y, t = blockIdx.x * 256 + threadIdx.x;
  const int n = x.n, m = x.m, d = x.d;
  float v1 = 0.f, v2 = 0.f;
  if (t < n + m) {
    const bool side1 = t < n;
    const int j = side1 ? t : t - n;
    const float *own = (side1 ? x.a + (static_cast<size_t>(cloud) * n + j) * d : x.b + (static_cast<size_t>(cloud) * m + j) * d);
    const int k = side1 ? __ldg(x.idx1 + static_cast<size_t>(cloud) * n + j) : __ldg(x.idx2 + static_cast<size_t>(cloud) * m + j);
    const float *oth = side1 ? x.b + (static_cast<size_t>(cloud) * m + k) * d : x.a + (static_cast<size_t>(cloud) * n + k) * d;
    float p[PL_MAXD], q[PL_MAXD];
    for (int e = 0; e < d; ++e) p[e] = __ldg(own + e), q[e] = __ldg(oth + e);
    PairVal o;
    pair_metric<false>(p, q, d, x.metric, o);
    (side1 ? v1 : v2) = o.v;
  }
  double s1 = v1, s2 = v2;
  for (int o = 16; o > 0; o >>= 1) {
    s1 += __shfl_xor_sync(0xffffffffu, s1, o);
    s2 += __shfl_xor_sync(0xffffffffu, s2, o);
  }
  if ((threadIdx.x & 31) == 0) sm[0][threadIdx.x >> 5] = s1, sm[1][threadIdx.x >> 5] = s2;
  __syncthreads();
  if (threadIdx.x == 0) {
    double a1 = 0.0, a2 = 0.0;
    for (int w = 0; w < 8; ++w) a1 += sm[0][w], a2 += sm[1][w];
    double *dst = partial + (static_cast<size_t>(blockIdx.y) * gridDim.x + blockIdx.x) * 2;
    dst[0] = a1, dst[1] = a2;
  }
}

// SCATTER = false: every point's own term (plain store: initialises ga / gb);  true: the matched rows' terms (RED.ADD)
template <bool SCATTER>
__global__ void __launch_bounds__(256) pair_loss_bwd_kernel(const PairArgs x, const float *__restrict__ gloss, float w1, float w2,
                                                            float *__restrict__ ga, float *__restrict__ gb) {
  const int cloud = blockIdx.y, t = blockIdx.x * 256 + threadIdx.x;
  const int n = x.n, m = x.m, d = x.d;
  if (t >= n + m) return;
  const bool side1 = t < n;
  const int j = side1 ? t : t - n;
  const size_t own_o = side1 ? (static_cast<size_t>(cloud) * n + j) * d : (static_cast<size_t>(cloud) * m + j) * d;
  const int k = side1 ? __ldg(x.idx1 + static_cast<size_t>(cloud) * n + j) : __ldg(x.idx2 + static_cast<size_t>(cloud) * m + j);
  const size_t oth_o = side1 ? (static_cast<size_t>(cloud) * m + k) * d : (static_cast<size_t>(cloud) * n + k) * d;
  const float *own = (side1 ? x.a : x.b) + own_o, *oth = (side1 ? x.b : x.a) + oth_o;
  float p[PL_MAXD], q[PL_MAXD];
  for (int e = 0; e < d; ++e) p[e] = __ldg(own + e), q[e] = __ldg(oth + e);
  PairVal o;
  pair_metric<true>(p, q, d, x.metric, o);
  const float g = __ldg(gloss) * (side1 ? w1 : w2);
  float *gown = (side1 ? ga : gb) + own_o, *goth = (side1 ? gb : ga) + oth_o;
  for (int e = 0; e < d; ++e) {
    if (SCATTER) atomicAdd(goth + e, g * o.gt[e]);
    else gown[e] = g * o.gp[e];
  }
}

// deterministic form: a point's own term, then the matched rows' terms (the points of the other cloud that chose it,
// ascending), rounded fp32 products and adds.  rev1 lists per point of a the points of b with idx2 == it, rev2 the converse.
__global__ void __launch_bounds__(256) pair_loss_bwd_det_kernel(const PairArgs x, const float *__restrict__ gloss, float w1,
                                                                float w2, RevMap rev1, RevMap rev2, float *__restrict__ ga,
                                                                float *__restrict__ gb) {
  const int cloud = blockIdx.y, t = blockIdx.x * 256 + threadIdx.x;
  const int n = x.n, m = x.m, d = x.d;
  if (t >= n + m) return;
  const bool side1 = t < n;
  const int j = side1 ? t : t - n;
  const size_t own_o = side1 ? (static_cast<size_t>(cloud) * n + j) * d : (static_cast<size_t>(cloud) * m + j) * d;
  const int k = side1 ? __ldg(x.idx1 + static_cast<size_t>(cloud) * n + j) : __ldg(x.idx2 + static_cast<size_t>(cloud) * m + j);
  const size_t oth_o = side1 ? (static_cast<size_t>(cloud) * m + k) * d : (static_cast<size_t>(cloud) * n + k) * d;
  const float *own = (side1 ? x.a : x.b) + own_o, *oth = (side1 ? x.b : x.a) + oth_o;
  float p[PL_MAXD], q[PL_MAXD], acc[PL_MAXD];
  for (int e = 0; e < d; ++e) p[e] = __ldg(own + e), q[e] = __ldg(oth + e);
  PairVal o;
  pair_metric<true>(p, q, d, x.metric, o);
  const float g = __ldg(gloss) * (side1 ? w1 : w2), gs = __ldg(gloss) * (side1 ? w2 : w1);
  for (int e = 0; e < d; ++e) acc[e] = __fmul_rn(g, o.gp[e]);
  // sources: points of the other cloud (rows `src`) whose match is this point (row p)
  const int ns = side1 ? m : n, nt = side1 ? n : m;
  const int *rp = (side1 ? rev1.ptr : rev2.ptr) + static_cast<size_t>(cloud) * (nt + 1);
  const int *rs = (side1 ? rev1.slot : rev2.slot) + static_cast<size_t>(cloud) * ns;
  const float *src = (side1 ? x.b : x.a) + static_cast<size_t>(cloud) * ns * d;
  const int lo = __ldg(rp + j), hi = __ldg(rp + j + 1);
  for (int qq = lo; qq < hi; ++qq) {
    const int i = __ldg(rs + qq);
    for (int e = 0; e < d; ++e) q[e] = __ldg(src + static_cast<size_t>(i) * d + e);
    pair_metric<true>(q, p, d, x.metric, o);
    for (int e = 0; e < d; ++e) acc[e] = __fadd_rn(acc[e], __fmul_rn(gs, o.gt[e]));
  }
  float *gown = (side1 ? ga : gb) + own_o;
  for (int e = 0; e < d; ++e) gown[e] = acc[e];
}

}  // namespace pdae

using namespace pdae;

static int pair_check(const float *a, const float *b, const int *idx1, const int *idx2, int bs, int n, int m, int d, int metric) {
  if (bs < 0 || n < 0 || m < 0 || d <= 0 || d > PL_MAXD || metric < 0 || metric > 3) return PDAE_E_INVALID;
  if (bs > 65535) return PDAE_E_UNSUPPORTED;
  if (bs && (n + m) && (!a || !b || !idx1 || !idx2)) return PDAE_E_INVALID;
  return 0;
}

extern "C" size_t pdae_pair_loss_partial_count(int bs, int n, int m) {
  return bs <= 0 || n + m <= 0 ? 0 : static_cast<size_t>(bs) * ((n + m + 255) / 256);
}

extern "C" int pdae_pair_loss_fwd_f64(const float *a, const float *b, const int *idx1, const int *idx2, int bs, int n, int m,
                                      int d, int metric, double *partial, pdae_stream_t stream) {
  const int rc = pair_check(a, b, idx1, idx2, bs, n, m, d, metric);
  if (rc) return rc;
  if (bs == 0 || n + m == 0) return 0;
  if (!partial || n == 0 || m == 0) return PDAE_E_INVALID;
  const dim3 grid((n + m + 255) / 256, bs);
  pair_loss_fwd_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(PairArgs{a, b, idx1, idx2, n, m, d, metric}, partial);
  PDAE_RETURN_IF_LAUNCH_FAILED();
  return 0;
}

extern "C" int pdae_pair_loss_bwd_f32(const float *a, const float *b, const int *idx1, const int *idx2, const float *gloss,
                                      float w1, float w2, int bs, int n, int m, int d, int metric, float *ga, float *gb,
                                      pdae_stream_t stream) {
  const int rc = pair_check(a, b, idx1, idx2, bs, n, m, d, metric);
  if (rc) return rc;
  if (bs == 0 || n + m == 0) return 0;
  if (!gloss || !ga || !gb || n == 0 || m == 0) return PDAE_E_INVALID;
  const dim3 grid((n + m + 255) / 256, bs);
  const PairArgs x{a, b, idx1, idx2, n, m, d, metric};
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  pair_loss_bwd_kernel<false><<<grid, 256, 0, st>>>(x, gloss, w1, w2, ga, gb);
  PDAE_RETURN_IF_LAUNCH_FAILED();
  pair_loss_bwd_kernel<true><<<grid, 256, 0, st>>>(x, gloss, w1, w2, ga, gb);
  PDAE_RETURN_IF_LAUNCH_FAILED();
  return 0;
}

static size_t pair_det_bytes(int bs, int n, int m) {
  return (rev_map_bytes(bs, m, n) + 255) / 256 * 256 + rev_map_bytes(bs, n, m);
}

extern "C" size_t pdae_pair_loss_bwd_det_workspace_bytes(int bs, int n, int m) {
  if (bs <= 0 || n <= 0 || m <= 0) return 0;
  return pair_det_bytes(bs, n, m);
}

extern "C" int pdae_pair_loss_bwd_det_f32(const float *a, const float *b, const int *idx1, const int *idx2, const float *gloss,
                                          float w1, float w2, int bs, int n, int m, int d, int metric, float *ga, float *gb,
                                          void *workspace, size_t workspace_bytes, pdae_stream_t stream) {
  const int rc = pair_check(a, b, idx1, idx2, bs, n, m, d, metric);
  if (rc) return rc;
  if (bs == 0 || n + m == 0) return 0;
  if (!gloss || !ga || !gb || n == 0 || m == 0) return PDAE_E_INVALID;
  if (!workspace || workspace_bytes < pdae_pair_loss_bwd_det_workspace_bytes(bs, n, m)) return PDAE_E_WORKSPACE;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  unsigned char *w = static_cast<unsigned char *>(workspace);
  RevMap rev1, rev2;
  int r = rev_map_build(idx2, bs, m, n, w, &rev1, st);
  if (r) return r;
  r = rev_map_build(idx1, bs, n, m, w + (rev_map_bytes(bs, m, n) + 255) / 256 * 256, &rev2, st);
  if (r) return r;
  const dim3 grid((n + m + 255) / 256, bs);
  pair_loss_bwd_det_kernel<<<grid, 256, 0, st>>>(PairArgs{a, b, idx1, idx2, n, m, d, metric}, gloss, w1, w2, rev1, rev2, ga, gb);
  PDAE_RETURN_IF_LAUNCH_FAILED();
  return 0;
}
