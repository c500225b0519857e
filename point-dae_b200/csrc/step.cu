// step.cu -- one step of the hot path enqueued natively: the launch choreography a caller would otherwise write with
// two side streams and three events per step (bench.py's step; the model's order is models/PointCAE_transformer.py:
// 1010-1066: patchify the cloud, ..., Chamfer loss between prediction and cloud, backward).
//
//   stream:  Chamfer forward (prediction vs cloud)  ->  patchifier of the cloud, queued as a PROGRAMMATIC DEPENDENT: it
//            reads only the cloud, the tensor-core forward triggers its dependents at once and owns every SM, so the
//            patchifier's CTAs start where and when a forward CTA exits
//   aux:     fused mean loss (two launches)            } both wait for the forward only and run beside the patchifier;
//   side:    backward from the loss scalar (two launches) } `stream` waits for both before the call returns
//            (PDAE_STEP_DETERMINISTIC: the deterministic backward, which builds its reverse maps there first)
//
// From Python every launch costs 20-30 us of host time, so a step was replayed as a CUDA graph -- and consecutive graph
// launches on one stream leave ~10 us between them (measured: 166.7 us per step replayed, 156.7 us with the same launches
// issued eagerly and the host far enough ahead).  Issued from here the six launches cost a few microseconds of host time.
// The helper streams and events are created once per device and reused; the call is capturable (fork / join through
// events) and leaves nothing pending on the helper streams that `stream` does not wait for.
#include <mutex>

#include "common.cuh"

namespace pdae {
namespace {

struct StepStreams {
  cudaStream_t aux = nullptr, side = nullptr;
  cudaEvent_t fwd_done = nullptr, loss_done = nullptr, bwd_done = nullptr;
  bool ready = false;
};

constexpr int STEP_MAX_DEVICES = 64;
std::mutex g_step_mu;
StepStreams g_step[STEP_MAX_DEVICES];

int step_streams(StepStreams **out) {
  int dev = 0;
  PDAE_CUDA_TRY(cudaGetDevice(&dev));
  if (dev < 0 || dev >= STEP_MAX_DEVICES) return PDAE_E_UNSUPPORTED;
  std::lock_guard<std::mutex> lock(g_step_mu);
  StepStreams &s = g_step[dev];
  if (!s.ready) {
    PDAE_CUDA_TRY(cudaStreamCreateWithFlags(&s.aux, cudaStreamNonBlocking));
    PDAE_CUDA_TRY(cudaStreamCreateWithFlags(&s.side, cudaStreamNonBlocking));
    PDAE_CUDA_TRY(cudaEventCreateWithFlags(&s.fwd_done, cudaEventDisableTiming));
    PDAE_CUDA_TRY(cudaEventCreateWithFlags(&s.loss_done, cudaEventDisableTiming));
    PDAE_CUDA_TRY(cudaEventCreateWithFlags(&s.bwd_done, cudaEventDisableTiming));
    s.ready = true;
  }
  *out = &s;
  return 0;
}

}  // namespace
}  // namespace pdae

using namespace pdae;

extern "C" size_t pdae_step_workspace_bytes(int b, int n, int g, int m) { return pdae_step_ex_workspace_bytes(b, n, g, m, 0u); }

// PDAE_STEP_DETERMINISTIC adds the ordered reverse maps of the deterministic backward after the other regions
extern "C" size_t pdae_step_ex_workspace_bytes(int b, int n, int g, int m, unsigned flags) {
  if (b <= 0 || n <= 0) return 0;
  const size_t det = (flags & PDAE_STEP_DETERMINISTIC) ? align256(pdae_chamfer_bwd_det_workspace_bytes(b, n, n)) : 0;
  return align256(pdae_chamfer_fwd_workspace_bytes(b, n, n)) + align256(pdae_chamfer_loss_workspace_bytes()) +
         align256(pdae_fps_group_workspace_bytes(b, n, g, m)) + det;
}

extern "C" int pdae_step_f32(const float *cloud, const float *pred, int b, int n, int g, int m, int *fps_idx, float *center,
                             float *neighborhood, float *dist1, float *dist2, int *idx1, int *idx2, float *loss3,
                             const float *gloss, float *gpred, float *gcloud, void *workspace, size_t workspace_bytes,
                             pdae_stream_t stream) {
  return pdae_step_ex_f32(cloud, pred, b, n, g, m, fps_idx, center, neighborhood, dist1, dist2, idx1, idx2, loss3, gloss, gpred,
                          gcloud, workspace, workspace_bytes, 0u, stream);
}

extern "C" int pdae_step_ex_f32(const float *cloud, const float *pred, int b, int n, int g, int m, int *fps_idx, float *center,
                                float *neighborhood, float *dist1, float *dist2, int *idx1, int *idx2, float *loss3,
                                const float *gloss, float *gpred, float *gcloud, void *workspace, size_t workspace_bytes,
                                unsigned flags, pdae_stream_t stream) {
  if (b < 0 || n < 0 || g < 0 || m <= 0 || (flags & ~static_cast<unsigned>(PDAE_STEP_DETERMINISTIC))) return PDAE_E_INVALID;
  if (b == 0) return 0;
  if (n == 0 || m > n) return PDAE_E_INVALID;
  if (!cloud || !pred || !dist1 || !dist2 || !idx1 || !idx2 || !loss3 || !gloss || !gpred || !gcloud) return PDAE_E_INVALID;
  if (g > 0 && (!fps_idx || !center || !neighborhood)) return PDAE_E_INVALID;
  const size_t w_fwd = align256(pdae_chamfer_fwd_workspace_bytes(b, n, n));
  const size_t w_loss = align256(pdae_chamfer_loss_workspace_bytes());
  const size_t w_patch = align256(pdae_fps_group_workspace_bytes(b, n, g, m));
  const bool det = (flags & PDAE_STEP_DETERMINISTIC) != 0;
  const size_t w_det = det ? align256(pdae_chamfer_bwd_det_workspace_bytes(b, n, n)) : 0;
  if (w_fwd + w_loss + w_patch + w_det > 0 && (!workspace || workspace_bytes < w_fwd + w_loss + w_patch + w_det))
    return PDAE_E_WORKSPACE;
  unsigned char *ws = static_cast<unsigned char *>(workspace);
  StepStreams *s = nullptr;
  int rc = step_streams(&s);
  if (rc) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  // the helper streams and events are shared by every caller on this device: a wait must see the record of its own call,
  // so the enqueue sequence of a call is atomic with respect to other host threads (a wait captures the event's state
  // when it is issued; the GPU work itself is not serialised by this)
  static std::mutex enqueue_mu[STEP_MAX_DEVICES];
  int dev = 0;
  PDAE_CUDA_TRY(cudaGetDevice(&dev));
  std::lock_guard<std::mutex> enqueue_lock(enqueue_mu[dev]);

  rc = pdae_chamfer_fwd_f32(pred, cloud, b, n, n, dist1, dist2, idx1, idx2, w_fwd ? ws : nullptr, w_fwd, stream);
  if (rc) return rc;
  PDAE_CUDA_TRY(cudaEventRecord(s->fwd_done, st));
  if (g > 0) {
    rc = pdae_fps_group_ex_f32(cloud, b, n, g, m, fps_idx, center, nullptr, neighborhood, w_patch ? ws + w_fwd + w_loss : nullptr,
                               w_patch, PDAE_LAUNCH_OVERLAP_PREVIOUS, stream);
    if (rc) return rc;
  }
  PDAE_CUDA_TRY(cudaStreamWaitEvent(s->aux, s->fwd_done, 0));
  rc = pdae_chamfer_loss_f32(dist1, dist2, b, n, n, 0, loss3, ws + w_fwd, w_loss, s->aux);
  if (rc) return rc;
  PDAE_CUDA_TRY(cudaEventRecord(s->loss_done, s->aux));
  PDAE_CUDA_TRY(cudaStreamWaitEvent(s->side, s->fwd_done, 0));
  if (det)
    rc = pdae_chamfer_loss_bwd_det_f32(pred, cloud, idx1, idx2, dist1, dist2, gloss, 1.0f, 1.0f, b, n, n, 0, gpred, gcloud,
                                       ws + w_fwd + w_loss + w_patch, w_det, s->side);
  else
    rc = pdae_chamfer_loss_bwd_f32(pred, cloud, idx1, idx2, dist1, dist2, gloss, 1.0f, 1.0f, b, n, n, 0, gpred, gcloud, s->side);
  if (rc) return rc;
  PDAE_CUDA_TRY(cudaEventRecord(s->bwd_done, s->side));
  PDAE_CUDA_TRY(cudaStreamWaitEvent(st, s->loss_done, 0));
  PDAE_CUDA_TRY(cudaStreamWaitEvent(st, s->bwd_done, 0));
  return 0;
}
