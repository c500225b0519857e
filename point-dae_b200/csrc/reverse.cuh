// reverse.cuh -- per-cloud reverse index of an index array (reverse.cu), shared by the deterministic gradients and the
// EdgeConv backward.
//
// idx (b, s) holds, for every source slot j of a cloud, a target in [0, t).  The map is a CSR per cloud:
//   ptr  (b, t + 1)  bucket offsets: the sources of target p are slot[ptr[p] .. ptr[p + 1]) (offsets within the cloud)
//   slot (b, s)      the source slots, grouped by target
// Sources outside [0, t) are left out (ptr[t] then counts the rest; slot entries past ptr[t] are not written).
// The ordered form sorts every bucket ascending, so the map is a pure function of idx: a stable argsort of each cloud's
// targets.  Buckets of up to REV_SHORT slots are sorted by one thread, up to REV_MID by one CTA in shared memory
// (bitonic), longer ones by one CTA compacting the cloud's sources for that target in slot order (stable by
// construction, s reads per such bucket and at most s / REV_MID such buckets per cloud).
#pragma once
#include "common.cuh"

namespace pdae {

constexpr int REV_SHORT = 32;
constexpr int REV_MID = 8192;

struct RevMap {
  const int *ptr;    // (b, t + 1)
  const int *slot;   // (b, s)
  const int *longq;  // the buckets longer than REV_SHORT: longq[0] of them, cloud * t + target each, in no set order
};

// Unordered CSR into caller arrays: cnt (b, t) is scratch (zeroed here); slot[...] = source slot / div.
// EdgeConv's dense backward (div = k: the source point of an edge) takes this form.
template <typename I>
int rev_csr_unordered(const I *idx, int b, int s, int t, int div, int *cnt, int *ptr, int *slot, cudaStream_t st);

// Ordered map built in a workspace of rev_map_bytes(b, s, t) bytes (ptr, slot and the sort's scratch).
size_t rev_map_bytes(int b, int s, int t);
template <typename I>
int rev_map_build(const I *idx, int b, int s, int t, void *ws, RevMap *out, cudaStream_t st);

// The channel-major deterministic gradient of gather / group_points / three_interpolate:
//   g[cloud][l][p] = +0 (+) term(j) for every source slot j of target p, j ascending,
//   term(j) = gout[cloud][l][j / div] (* weight[cloud][j] when weight is given), with rounded fp32 adds and products.
// gout is (b, c, s / div), weight (b, s) or null, g (b, c, t); the map is the ordered one of the (b, s) index array.
int rev_gather_channel_major(const float *gout, const float *weight, int b, int c, int s, int t, int div, RevMap map,
                             float *g, cudaStream_t st);

}  // namespace pdae
