// The one order every exact ranking merges by: score descending, then item id ascending, and id -1 (an exhausted list)
// last.  tfr_rank_users merges its chunk lists with it (rank_users.cu) and tfr_shard_topk_merge the lists of the item
// shards (shard_rank.cu): the order is total over distinct ids, so any split of the items gives the same result.
#pragma once
#include "common.cuh"

namespace tfr {

// (v, i) ranks before (ov, oi): higher score, then lower item id; i = -1 (an exhausted list) ranks last.
__device__ __forceinline__ bool ru_before(double v, int i, double ov, int oi) {
  if (oi < 0) return i >= 0;
  if (i < 0) return false;
  return v > ov || (v == ov && i < oi);
}

// Every lane offers (wv, wi) with wl = its lane; on return every lane holds the best entry of the warp and the lane that
// offered it (the lowest such lane when entries are equal, e.g. two exhausted lists).
__device__ __forceinline__ void ru_warp_best(double& wv, int& wi, int& wl) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const double ov = __shfl_xor_sync(0xffffffffu, wv, o);
    const int oi = __shfl_xor_sync(0xffffffffu, wi, o);
    const int ol = __shfl_xor_sync(0xffffffffu, wl, o);
    if (ru_before(ov, oi, wv, wi) || (oi == wi && ol < wl)) { wv = ov; wi = oi; wl = ol; }
  }
}

}  // namespace tfr
