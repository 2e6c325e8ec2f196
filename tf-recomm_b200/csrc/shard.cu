// Row-sharded tables (SURVEY 8e, BASELINE configs[4]): rows of each table and their Adam state live on rank
// (id mod G); this is the owner's half of the per-step row exchange.  The reference has no distributed code at
// all (single tf.Session, svd_train_val.py:55) -- this is the B200-native equivalent north_star asks for.
#include "common.cuh"

namespace tfr {

template <int VEC, int L>
__global__ void __launch_bounds__(256) shard_gather_rows_kernel(const float* __restrict__ feat,
                                                                const float* __restrict__ bias, int rows_local,
                                                                int dim, int64_t fstride,
                                                                const int32_t* __restrict__ ids, int64_t B,
                                                                int n_ranks, int rank, float* __restrict__ out_feat,
                                                                float* __restrict__ out_bias,
                                                                int32_t* __restrict__ keys) {
  const int lane = threadIdx.x & (L - 1);
  const int64_t b = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) / L;
  if (b >= B) return;
  const int32_t id = ids[b];
  const bool mine = (id % n_ranks) == rank;
  const int32_t local = id / n_ranks;
  const int n_units = dim / VEC;
  for (int unit = lane; unit < n_units; unit += L) {
    if constexpr (VEC == 4) {
      float4 x = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
      if (mine) x = ld_gather_f4(reinterpret_cast<const float4*>(feat + (size_t)local * fstride) + unit);
      reinterpret_cast<float4*>(out_feat + (size_t)b * dim)[unit] = x;
    } else {
      out_feat[(size_t)b * dim + unit] = mine ? ld_gather_f1(feat + (size_t)local * fstride + unit) : 0.0f;
    }
  }
  if (lane == 0) {
    out_bias[b] = mine ? bias[local] : 0.0f;
    keys[b] = mine ? local : rows_local;
  }
}


// ================================ all-to-all exchange (north_star: ids / rows / gradients) ==============================
// Per step every rank holds a SLICE of the global batch (n = B / G occurrences, contiguous in global batch order):
//   1. bucket its ids by owner (id mod G), stably                       tfr_shard_bucket           [local]
//   2. all-to-all of the bucketed LOCAL row ids (id / G)                                            [NCCL]
//   3. owners pack the requested rows as records [row | bias | pad]     tfr_shard_gather_records   [local]
//   4. all-to-all of the records back to the requesters                                             [NCCL]
//   5. forward + d cost/d logits on the slice; one record per occurrence and table for the row's owner:
//      [PARTNER row | e | pad] -- g = e * partner + reg * own, the owner has `own`  tfr_shard_fwd_records  [local]
//   6. all-to-all of those records to the owners (same splits as 2)                                 [NCCL]
//   7. owners: keys + errors by arrival position, then the single-GPU kernels unchanged: stable sort, ordered segment
//      sums (partner rows / errors by position), ONE Adam pass over the local shard  tfr_shard_owner_prepare +
//      tfr_svd_train_step_gathered                                                                  [local]
// A received buffer is [src 0: user part | item part][src 1: ...]...: ascending position = (source rank, position in
// the source's slice) = GLOBAL BATCH ORDER, so the stable sort + in-order segment sums add duplicate rows in the order
// the single-GPU path (and TF's unsorted_segment_sum) does.  Record stride = dim + 4 floats (16-byte aligned rows).
struct ShardLayout {  // a combined buffer, by source (or destination) rank: [u_begin, i_begin) user part, [i_begin, end) item part
  int32_t n_ranks;
  int32_t u_begin[SHARD_MAX_RANKS], i_begin[SHARD_MAX_RANKS], end[SHARD_MAX_RANKS];
};
__device__ __forceinline__ bool shard_is_user(const ShardLayout& L, int64_t k) {
  bool u = false;
#pragma unroll
  for (int s = 0; s < SHARD_MAX_RANKS; ++s)
    if (s < L.n_ranks && k >= L.u_begin[s] && k < L.i_begin[s]) u = true;
  return u;
}

__global__ void __launch_bounds__(256) shard_owner_keys_kernel(const int32_t* __restrict__ users,
                                                               const int32_t* __restrict__ items, int64_t n, int G,
                                                               int32_t* __restrict__ ku, int32_t* __restrict__ ki) {
  const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n) return;
  ku[k] = users[k] % G;
  ki[k] = items[k] % G;
}

// ONE CTA: from the slice sorted by owner (stable: ascending position inside an owner's bucket) to the combined send
// layout [dst 0: users | items][dst 1: ...]: counts[2G], send_ids = local row ids, slot_u / slot_i = where occurrence
// p's user / item entry sits in the combined buffer (the records come back, and go out again, at the same index).
__global__ void __launch_bounds__(1024) shard_bucket_finish_kernel(const int32_t* __restrict__ users,
                                                                   const int32_t* __restrict__ items,
                                                                   const int32_t* __restrict__ sk_u, const int32_t* __restrict__ sp_u,
                                                                   const int32_t* __restrict__ sk_i, const int32_t* __restrict__ sp_i,
                                                                   int64_t n, int G, int32_t* __restrict__ counts,
                                                                   int32_t* __restrict__ send_ids, int32_t* __restrict__ slot_u,
                                                                   int32_t* __restrict__ slot_i) {
  __shared__ int s_start[2][SHARD_MAX_RANKS + 1], s_off[2][SHARD_MAX_RANKS];
  if (threadIdx.x < 2 * (G + 1)) {   // first index whose owner key is >= g (binary search in the sorted keys)
    const int side = threadIdx.x / (G + 1), g = threadIdx.x % (G + 1);
    const int32_t* sk = side ? sk_i : sk_u;
    int64_t lo = 0, hi = n;
    while (lo < hi) {
      const int64_t mid = (lo + hi) >> 1;
      if (sk[mid] < g) lo = mid + 1; else hi = mid;
    }
    s_start[side][g] = (int)lo;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    int at = 0;
    for (int g = 0; g < G; ++g) {
      const int cu = s_start[0][g + 1] - s_start[0][g], ci = s_start[1][g + 1] - s_start[1][g];
      counts[g] = cu; counts[G + g] = ci;
      s_off[0][g] = at; s_off[1][g] = at + cu;
      at += cu + ci;
    }
  }
  __syncthreads();
  for (int64_t k = threadIdx.x; k < n; k += blockDim.x) {
    {
      const int g = sk_u[k], p = sp_u[k];
      const int idx = s_off[0][g] + (int)(k - s_start[0][g]);
      send_ids[idx] = users[p] / G;
      slot_u[p] = idx;
    }
    {
      const int g = sk_i[k], p = sp_i[k];
      const int idx = s_off[1][g] + (int)(k - s_start[1][g]);
      send_ids[idx] = items[p] / G;
      slot_i[p] = idx;
    }
  }
}

// owner: received local row ids -> records [row | bias | pad]; one lane group per record
template <int VEC, int L>
__global__ void __launch_bounds__(256) shard_gather_records_kernel(const float* __restrict__ uf, const float* __restrict__ ubias,
                                                                   const float* __restrict__ itf, const float* __restrict__ ibias,
                                                                   int64_t fstride, int dim, int rs,
                                                                   const int32_t* __restrict__ recv_ids, ShardLayout lay,
                                                                   int64_t total, float* __restrict__ out) {
  const int lane = threadIdx.x & (L - 1);
  const int64_t k = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) / L;
  if (k >= total) return;
  const bool is_user = shard_is_user(lay, k);
  const int32_t id = recv_ids[k];
  const float* row = (is_user ? uf : itf) + (size_t)id * fstride;
  float* dst = out + (size_t)k * rs;
  const int n_units = dim / VEC;
  for (int unit = lane; unit < n_units; unit += L) {
    if constexpr (VEC == 4) reinterpret_cast<float4*>(dst)[unit] = ld_gather_f4(reinterpret_cast<const float4*>(row) + unit);
    else dst[unit] = ld_gather_f1(row + unit);
  }
  if (lane == 0) dst[dim] = (is_user ? ubias : ibias)[id];
}

// requester: forward (ops.py:44-47) + d cost/d logits (ops.py:124-126) on the slice from the records that came back;
// one outgoing record per occurrence and table: [partner row | e].  Arithmetic and reduction order of
// svd_forward_kernel (products and adds separate fp32 roundings, lane-group butterfly).
template <int VEC, int L>
__global__ void __launch_bounds__(256) shard_fwd_records_kernel(const float* __restrict__ rec_in, const int32_t* __restrict__ slot_u,
                                                                const int32_t* __restrict__ slot_i, const float* __restrict__ rates,
                                                                int64_t n, int dim, int rs, const float* __restrict__ mu_p,
                                                                const tfr_opt_scalars* __restrict__ opt, float* __restrict__ rec_out,
                                                                float* __restrict__ logits, float* __restrict__ infer,
                                                                float* __restrict__ partials, double* __restrict__ se_partials) {
  const int lane = threadIdx.x & (L - 1);
  const int flags = opt->flags;
  const bool abs_item = flags & TFR_ABS_ITEM;
  const float mu = *mu_p;
  float err_acc = 0.0f;
  double se_acc = 0.0;
  const int64_t n_groups = (int64_t)gridDim.x * blockDim.x / L;
  const int64_t group = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) / L;
  constexpr int GPW = 32 / L;
  const int64_t warp_first = group - (group % GPW);
  for (int64_t p0 = warp_first; p0 < n; p0 += n_groups) {   // whole warps iterate together (the butterflies need them)
    const int64_t p = p0 + (group % GPW);
    const bool val = p < n;
    const int su = val ? slot_u[p] : 0, si = val ? slot_i[p] : 0;
    const float* ur = rec_in + (size_t)su * rs;
    const float* vr = rec_in + (size_t)si * rs;
    float* ou = rec_out + (size_t)su * rs;   // to the USER row's owner: the item row
    float* oi = rec_out + (size_t)si * rs;   // to the ITEM row's owner: the user row
    float acc = 0.0f;
    const int n_units = dim / VEC;
    if (val) {
      for (int unit = lane; unit < n_units; unit += L) {
        if constexpr (VEC == 4) {
          const float4 a = reinterpret_cast<const float4*>(ur)[unit], q = reinterpret_cast<const float4*>(vr)[unit];
          reinterpret_cast<float4*>(ou)[unit] = q;
          reinterpret_cast<float4*>(oi)[unit] = a;
          acc = add_rn(acc, mul_rn(a.x, abs_item ? fabsf(q.x) : q.x));
          acc = add_rn(acc, mul_rn(a.y, abs_item ? fabsf(q.y) : q.y));
          acc = add_rn(acc, mul_rn(a.z, abs_item ? fabsf(q.z) : q.z));
          acc = add_rn(acc, mul_rn(a.w, abs_item ? fabsf(q.w) : q.w));
        } else {
          const float a = ur[unit], q = vr[unit];
          ou[unit] = q;
          oi[unit] = a;
          acc = add_rn(acc, mul_rn(a, abs_item ? fabsf(q) : q));
        }
      }
    }
    acc = group_sum<L>(acc);
    if (val && lane == 0) {
      float x = add_rn(acc, mu);
      x = add_rn(x, ur[dim]);
      x = add_rn(x, vr[dim]);
      const float z = rates[p];
      const float inf = (flags & TFR_LOSS_SIGMOID_CE) ? rintf(sigmoid_tf(x)) : x;
      const float e = dloss(flags, x, z);
      ou[dim] = e;
      oi[dim] = e;
      if (logits) logits[p] = x;
      if (infer) infer[p] = inf;
      err_acc = add_rn(err_acc, e);
      const double dse = (double)z - (double)inf;
      se_acc += dse * dse;
    }
  }
  __shared__ float s_err[256];
  __shared__ double s_se[256];
  s_err[threadIdx.x] = (lane == 0) ? err_acc : 0.0f;
  s_se[threadIdx.x] = (lane == 0) ? se_acc : 0.0;
  __syncthreads();
  if (threadIdx.x < 32) {
    float a = 0.0f;
    double d = 0.0;
    for (int j = threadIdx.x; j < 256; j += 32) { a = add_rn(a, s_err[j]); d += s_se[j]; }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      a = add_rn(a, __shfl_xor_sync(0xffffffffu, a, o));
      d += __shfl_xor_sync(0xffffffffu, d, o);
    }
    if (threadIdx.x == 0) { partials[blockIdx.x] = a; se_partials[blockIdx.x] = d; }
  }
}
// this rank's sums over its slice, folded in a fixed order: out2 = [sum_b e_b, sum_b (rate - infer)^2] as doubles
__global__ void __launch_bounds__(32) shard_fold_partials_kernel(const float* __restrict__ partials, const double* __restrict__ se_partials,
                                                                int n_part, double* __restrict__ out2) {
  float a = 0.0f;
  double d = 0.0;
  for (int j = threadIdx.x; j < n_part; j += 32) { a = add_rn(a, partials[j]); d += se_partials[j]; }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    a = add_rn(a, __shfl_xor_sync(0xffffffffu, a, o));
    d += __shfl_xor_sync(0xffffffffu, d, o);
  }
  if (threadIdx.x == 0) { out2[0] = (double)a; out2[1] = d; }
}
// after the all-reduce over ranks: the step's d cost/d bias_global as the fp32 the finish takes, the squared error
__global__ void shard_unfold_sums_kernel(const double* __restrict__ in2, float* __restrict__ sum_err, double* __restrict__ sum_se) {
  *sum_err = (float)in2[0];
  *sum_se = in2[1];
}

// owner: sort keys of both tables over the received buffer (entries of the other table get the "not mine" mark, sorted
// to the end and skipped), and every entry's error by arrival position
__global__ void __launch_bounds__(256) shard_owner_prepare_kernel(const int32_t* __restrict__ recv_ids, const float* __restrict__ rec,
                                                                  ShardLayout lay, int64_t total, int dim, int rs, int u_loc, int i_loc,
                                                                  int32_t* __restrict__ keys_u, int32_t* __restrict__ keys_i,
                                                                  float* __restrict__ err) {
  const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= total) return;
  const bool is_user = shard_is_user(lay, k);
  const int32_t id = recv_ids[k];
  keys_u[k] = is_user ? id : u_loc;
  keys_i[k] = is_user ? i_loc : id;
  err[k] = rec[(size_t)k * rs + dim];
}

static int make_layout(ShardLayout* L, const int32_t* cnt_u, const int32_t* cnt_i, int n_ranks, int64_t* total) {
  TFR_CHECK_ARG(cnt_u && cnt_i && n_ranks >= 1 && n_ranks <= SHARD_MAX_RANKS);
  int64_t at = 0;
  L->n_ranks = n_ranks;
  for (int s = 0; s < SHARD_MAX_RANKS; ++s) {
    const int cu = s < n_ranks ? cnt_u[s] : 0, ci = s < n_ranks ? cnt_i[s] : 0;
    TFR_CHECK_ARG(cu >= 0 && ci >= 0);
    L->u_begin[s] = (int32_t)at;
    L->i_begin[s] = (int32_t)(at + cu);
    L->end[s] = (int32_t)(at + cu + ci);
    at += cu + ci;
    TFR_CHECK_ARG(at < ((int64_t)1 << 31));
  }
  *total = at;
  return TFR_OK;
}

}  // namespace tfr

using namespace tfr;

extern "C" int tfr_shard_gather_rows(const float* feat_local, const float* bias_local, int64_t rows_local, int32_t dim,
                                     int64_t feat_stride,
                                     const int32_t* ids, int64_t B, int32_t n_ranks, int32_t rank, float* out_feat,
                                     float* out_bias, int32_t* local_keys, void* stream) {
  TFR_CHECK_ARG(B >= 0 && dim > 0 && n_ranks >= 1 && rank >= 0 && rank < n_ranks && rows_local >= 0 &&
                rows_local < ((int64_t)1 << 31));
  if (B == 0) return TFR_OK;
  TFR_CHECK_ARG(feat_local && bias_local && ids && out_feat && out_bias && local_keys);
  const RowGeom g = row_geom(dim);
  const int groups_per_cta = 256 / g.lanes;
  const unsigned grid = (unsigned)((B + groups_per_cta - 1) / groups_per_cta);
  cudaStream_t st = (cudaStream_t)stream;
#define TFR_SG_CASE(V, LL)                                                                                        \
  if (g.vec == V && g.lanes == LL) {                                                                              \
    TFR_PREP((shard_gather_rows_kernel<V, LL>));                                                                  \
    shard_gather_rows_kernel<V, LL><<<grid, 256, 0, st>>>(feat_local, bias_local, (int)rows_local, dim,              \
                                                          feat_stride ? feat_stride : (int64_t)dim, ids, B,   \
                                                          n_ranks, rank, out_feat, out_bias, local_keys);         \
    TFR_LAUNCH_CHECK();                                                                                            \
    return TFR_OK;                                                                                                 \
  }
  TFR_SG_CASE(4, 1) TFR_SG_CASE(4, 2) TFR_SG_CASE(4, 4) TFR_SG_CASE(4, 8) TFR_SG_CASE(4, 16) TFR_SG_CASE(4, 32)
  TFR_SG_CASE(1, 1) TFR_SG_CASE(1, 2) TFR_SG_CASE(1, 4) TFR_SG_CASE(1, 8) TFR_SG_CASE(1, 16) TFR_SG_CASE(1, 32)
#undef TFR_SG_CASE
  set_error("unsupported dim %d", dim);
  return TFR_ERR_INVALID;
}


extern "C" int64_t tfr_shard_bucket_workspace_bytes(int64_t n) {
  if (n < 0) return TFR_ERR_INVALID;
  return 256 + 6 * align_up(n * 4, 256) + tfr_dedup_workspace_bytes(n) + 256;
}

extern "C" int tfr_shard_bucket(const int32_t* users, const int32_t* items, int64_t n, int32_t n_ranks, int32_t* counts,
                                int32_t* send_ids, int32_t* slot_u, int32_t* slot_i, void* workspace, int64_t workspace_bytes,
                                void* stream) {
  TFR_CHECK_ARG(n >= 0 && n < ((int64_t)1 << 30) && n_ranks >= 1 && n_ranks <= SHARD_MAX_RANKS && counts);
  cudaStream_t st = (cudaStream_t)stream;
  if (n == 0) {
    TFR_CUDA(cudaMemsetAsync(counts, 0, 2 * n_ranks * sizeof(int32_t), st));
    return TFR_OK;
  }
  TFR_CHECK_ARG(users && items && send_ids && slot_u && slot_i && workspace);
  if (workspace_bytes < tfr_shard_bucket_workspace_bytes(n)) {
    set_error("shard bucket workspace too small");
    return TFR_ERR_WORKSPACE;
  }
  char* w = reinterpret_cast<char*>(align_up((int64_t)(uintptr_t)workspace, 256));
  const int64_t a4 = align_up(n * 4, 256);
  int32_t* ku = (int32_t*)w; int32_t* ki = (int32_t*)(w + a4);
  int32_t* sk_u = (int32_t*)(w + 2 * a4); int32_t* sp_u = (int32_t*)(w + 3 * a4);
  int32_t* sk_i = (int32_t*)(w + 4 * a4); int32_t* sp_i = (int32_t*)(w + 5 * a4);
  void* sort_ws = w + 6 * a4;
  shard_owner_keys_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(users, items, n, n_ranks, ku, ki);
  TFR_LAUNCH_CHECK();
  int rc = tfr_dedup_sort_pairs(ku, n_ranks, sk_u, sp_u, ki, n_ranks, sk_i, sp_i, n, sort_ws, tfr_dedup_workspace_bytes(n), stream);
  if (rc) return rc;
  shard_bucket_finish_kernel<<<1, 1024, 0, st>>>(users, items, sk_u, sp_u, sk_i, sp_i, n, n_ranks, counts, send_ids, slot_u, slot_i);
  TFR_LAUNCH_CHECK();
  return TFR_OK;
}

extern "C" int tfr_shard_gather_records(const tfr_svd_tables* t, const int32_t* recv_ids, const int32_t* cnt_u_host,
                                        const int32_t* cnt_i_host, int32_t n_ranks, float* records, void* stream) {
  TFR_CHECK_ARG(t && t->dim > 0);
  ShardLayout lay;
  int64_t total = 0;
  int rc = make_layout(&lay, cnt_u_host, cnt_i_host, n_ranks, &total);
  if (rc) return rc;
  if (total == 0) return TFR_OK;
  TFR_CHECK_ARG(recv_ids && records && t->user_feat && t->item_feat && t->user_bias && t->item_bias);
  const int dim = t->dim, rs = dim + 4;
  const RowGeom g = row_geom(dim);
  const int64_t fs = t->feat_stride ? t->feat_stride : dim;
  const int groups_per_cta = 256 / g.lanes;
  const unsigned grid = (unsigned)((total + groups_per_cta - 1) / groups_per_cta);
  cudaStream_t st = (cudaStream_t)stream;
#define TFR_SGR_CASE(V, LL)                                                                                          \
  if (g.vec == V && g.lanes == LL) {                                                                                 \
    shard_gather_records_kernel<V, LL><<<grid, 256, 0, st>>>(t->user_feat, t->user_bias, t->item_feat, t->item_bias, fs, \
                                                             dim, rs, recv_ids, lay, total, records);               \
    TFR_LAUNCH_CHECK();                                                                                              \
    return TFR_OK;                                                                                                   \
  }
  TFR_SGR_CASE(4, 1) TFR_SGR_CASE(4, 2) TFR_SGR_CASE(4, 4) TFR_SGR_CASE(4, 8) TFR_SGR_CASE(4, 16) TFR_SGR_CASE(4, 32)
  TFR_SGR_CASE(1, 1) TFR_SGR_CASE(1, 2) TFR_SGR_CASE(1, 4) TFR_SGR_CASE(1, 8) TFR_SGR_CASE(1, 16) TFR_SGR_CASE(1, 32)
#undef TFR_SGR_CASE
  set_error("unsupported dim %d", dim);
  return TFR_ERR_INVALID;
}

extern "C" int tfr_shard_fwd_records(const tfr_svd_tables* t, const tfr_opt_scalars* opt, const float* records_in,
                                     const int32_t* slot_u, const int32_t* slot_i, const float* rates, int64_t n,
                                     float* records_out, float* logits, float* infer, float* partials /* [1024] */,
                                     double* se_partials /* [1024] */, double* sums2, void* stream) {
  TFR_CHECK_ARG(t && opt && t->dim > 0 && n >= 0 && partials && se_partials && sums2 && t->mu);
  TFR_CHECK_ARG(n == 0 || (records_in && slot_u && slot_i && rates && records_out));
  const int dim = t->dim, rs = dim + 4;
  const RowGeom g = row_geom(dim);
  const int64_t rows_per_cta = 256 / g.lanes;
  int64_t grid = (n + rows_per_cta - 1) / rows_per_cta;
  if (grid > TFR_MAX_PARTIALS) grid = TFR_MAX_PARTIALS;
  if (grid < 1) grid = 1;
  cudaStream_t st = (cudaStream_t)stream;
  bool launched = false;
#define TFR_SFR_CASE(V, LL)                                                                                              \
  if (!launched && g.vec == V && g.lanes == LL) {                                                                        \
    shard_fwd_records_kernel<V, LL><<<(unsigned)grid, 256, 0, st>>>(records_in, slot_u, slot_i, rates, n, dim, rs, t->mu, opt, \
                                                                    records_out, logits, infer, partials, se_partials);  \
    launched = true;                                                                                                     \
  }
  TFR_SFR_CASE(4, 1) TFR_SFR_CASE(4, 2) TFR_SFR_CASE(4, 4) TFR_SFR_CASE(4, 8) TFR_SFR_CASE(4, 16) TFR_SFR_CASE(4, 32)
  TFR_SFR_CASE(1, 1) TFR_SFR_CASE(1, 2) TFR_SFR_CASE(1, 4) TFR_SFR_CASE(1, 8) TFR_SFR_CASE(1, 16) TFR_SFR_CASE(1, 32)
#undef TFR_SFR_CASE
  if (!launched) {
    set_error("unsupported dim %d", dim);
    return TFR_ERR_INVALID;
  }
  TFR_LAUNCH_CHECK();
  shard_fold_partials_kernel<<<1, 32, 0, st>>>(partials, se_partials, (int)grid, sums2);
  TFR_LAUNCH_CHECK();
  return TFR_OK;
}

extern "C" int tfr_shard_owner_prepare(const int32_t* recv_ids, const float* records, const int32_t* cnt_u_host,
                                       const int32_t* cnt_i_host, int32_t n_ranks, int32_t dim, int64_t users_local,
                                       int64_t items_local, int32_t* keys_u, int32_t* keys_i, float* err,
                                       const double* sums2_allreduced, float* sum_err, double* sum_se, void* stream) {
  ShardLayout lay;
  int64_t total = 0;
  int rc = make_layout(&lay, cnt_u_host, cnt_i_host, n_ranks, &total);
  if (rc) return rc;
  TFR_CHECK_ARG(dim > 0 && sums2_allreduced && sum_err && sum_se);
  cudaStream_t st = (cudaStream_t)stream;
  shard_unfold_sums_kernel<<<1, 1, 0, st>>>(sums2_allreduced, sum_err, sum_se);
  TFR_LAUNCH_CHECK();
  if (total == 0) return TFR_OK;
  TFR_CHECK_ARG(recv_ids && records && keys_u && keys_i && err);
  shard_owner_prepare_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(recv_ids, records, lay, total, dim, dim + 4,
                                                                             (int)users_local, (int)items_local, keys_u,
                                                                             keys_i, err);
  TFR_LAUNCH_CHECK();
  return TFR_OK;
}
