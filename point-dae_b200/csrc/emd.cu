// emd.cu -- approximate Earth Mover's Distance (Fan et al. 2017 `approxmatch` / `matchcost` / `matchcostgrad`, the
// reference's extensions/emd, module `emd_cuda`) without the (B, m, n) match matrix.
//
// approxmatch runs 10 levels of three passes each (include/pointdae_b200.h gives the arithmetic).  Per level the match
// only accumulates w(k,l) = (e_j(k,l) * ratioL_j[k]) * ratioR_j[l], so the kernel stores the per-level ratios
// (B,10,n) and (B,10,m) -- 80 bytes per point -- and every consumer of the match rebuilds it from them with the same
// expression in the same order.  Every row and column sum is one thread's sequential chain over the whole other
// cloud, so the bits do not depend on how clouds are split over CTAs: a cloud gets one CTA when the batch fills the
// GPU and a cluster of up to 8 CTAs otherwise, chosen from B and the SM count.  The CTAs of a cluster exchange
// remainR / ratioL / ratioR through the global (L2) arrays, read with ld.global.cg after one cluster barrier per pass.
// The other cloud streams through shared-memory tiles; the distance and the sums use packed f32x2 operations.  The
// bodies live in emd_core.cuh, shared with the segment entry points (segemd.cu).
#include "emd_core.cuh"

namespace pdae {

// grid: B * cs CTAs, clusters of cs (cs == 1: no cluster)
__global__ void __launch_bounds__(EMD_THREADS) emd_approxmatch_kernel(const EmdMatchArgs a) {
  __shared__ float4 tile[EMD_TILE];
  emd_approxmatch_body<false>(a, EmdSegTables{}, tile);
}

__global__ void __launch_bounds__(256) emd_cost_reduce_kernel(const float *__restrict__ rowcost, int m, float *__restrict__ cost) {
  __shared__ float p[256];
  const int b = blockIdx.x;
  emd_cost_reduce_body(rowcost + static_cast<size_t>(b) * m, m, p);
  if (threadIdx.x == 0) cost[b] = p[0];
}

static size_t emd_ws_bytes(int b, int n, int m) {
  return align256(static_cast<size_t>(b) * n * sizeof(float)) + align256(static_cast<size_t>(b) * m * sizeof(float));
}

static int emd_check(const float *xyz1, const float *xyz2, int b, int n, int m) {
  if (b < 0 || n <= 0 || m <= 0) return PDAE_E_INVALID;
  if (n > EMD_MAX_POINTS || m > EMD_MAX_POINTS || b > 65535) return PDAE_E_UNSUPPORTED;
  if (b && (!xyz1 || !xyz2)) return PDAE_E_INVALID;
  return 0;
}

}  // namespace pdae

using namespace pdae;

extern "C" size_t pdae_emd_workspace_bytes(int b, int n, int m) {
  if (b <= 0 || n <= 0 || m <= 0) return 0;
  return emd_ws_bytes(b, n, m);
}

extern "C" int pdae_emd_match_f32(const float *xyz1, const float *xyz2, int b, int n, int m, float *ratio_l, float *ratio_r,
                                  float *match, void *workspace, size_t workspace_bytes, pdae_stream_t stream) {
  const int rc = emd_check(xyz1, xyz2, b, n, m);
  if (rc || b == 0) return rc;
  if (!ratio_l || !ratio_r) return PDAE_E_INVALID;
  if (!workspace || workspace_bytes < emd_ws_bytes(b, n, m)) return PDAE_E_WORKSPACE;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  float *reml = static_cast<float *>(workspace);
  float *remr = reinterpret_cast<float *>(static_cast<unsigned char *>(workspace) + align256(static_cast<size_t>(b) * n * 4));
  const int cs = emd_cluster_size(b, n, m);
  const EmdMatchArgs args{xyz1, xyz2, n, m, cs, ratio_l, ratio_r, reml, remr};
  PDAE_CUDA_TRY(emd_launch_clusters(emd_approxmatch_kernel, b, cs, st, args));
  if (match) {
    const EmdSumArgs s{xyz1, xyz2, n, m, nullptr, ratio_l, ratio_r};
    emd_sum_kernel<false, 2><<<dim3(ceil_div(n, EMD_CHUNK), b), EMD_THREADS, 0, st>>>(s, nullptr, match, EmdSegTables{});
    PDAE_RETURN_IF_LAUNCH_FAILED();
  }
  return 0;
}

extern "C" int pdae_emd_cost_f32(const float *xyz1, const float *xyz2, int b, int n, int m, const float *match,
                                 const float *ratio_l, const float *ratio_r, float *cost, void *workspace,
                                 size_t workspace_bytes, pdae_stream_t stream) {
  const int rc = emd_check(xyz1, xyz2, b, n, m);
  if (rc || b == 0) return rc;
  if (!cost || (!match && (!ratio_l || !ratio_r))) return PDAE_E_INVALID;
  if (!workspace || workspace_bytes < emd_ws_bytes(b, n, m)) return PDAE_E_WORKSPACE;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  float *rowcost = static_cast<float *>(workspace);
  const EmdSumArgs s{xyz1, xyz2, n, m, match, ratio_l, ratio_r};
  emd_sum_kernel<true, 0><<<dim3(ceil_div(m, EMD_CHUNK), b), EMD_THREADS, 0, st>>>(s, nullptr, rowcost, EmdSegTables{});
  PDAE_RETURN_IF_LAUNCH_FAILED();
  emd_cost_reduce_kernel<<<b, 256, 0, st>>>(rowcost, m, cost);
  PDAE_RETURN_IF_LAUNCH_FAILED();
  return 0;
}

extern "C" int pdae_emd_cost_grad_f32(const float *grad_cost, const float *xyz1, const float *xyz2, int b, int n, int m,
                                      const float *match, const float *ratio_l, const float *ratio_r, float *grad1,
                                      float *grad2, pdae_stream_t stream) {
  const int rc = emd_check(xyz1, xyz2, b, n, m);
  if (rc || b == 0) return rc;
  if (!grad_cost || !grad1 || !grad2 || (!match && (!ratio_l || !ratio_r))) return PDAE_E_INVALID;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const EmdSumArgs s{xyz1, xyz2, n, m, match, ratio_l, ratio_r};
  emd_sum_kernel<false, 1><<<dim3(ceil_div(n, EMD_CHUNK), b), EMD_THREADS, 0, st>>>(s, grad_cost, grad1, EmdSegTables{});
  PDAE_RETURN_IF_LAUNCH_FAILED();
  emd_sum_kernel<true, 1><<<dim3(ceil_div(m, EMD_CHUNK), b), EMD_THREADS, 0, st>>>(s, grad_cost, grad2, EmdSegTables{});
  PDAE_RETURN_IF_LAUNCH_FAILED();
  return 0;
}
