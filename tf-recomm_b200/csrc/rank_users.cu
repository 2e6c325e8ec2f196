// Exact float64 top-k ranking for a batch of query users (tfr_rank_users): forward.py:47-61 get_ranking for an arbitrary
// list of users, optionally over the items each user has not rated.  Same scores, same order and same bits as the
// user's row of tfr_allpairs_rank_excluding, at a cost that scales with the number of query users instead of n_users.
//
// Three kernels, all on CUDA cores (the data sheet lists the same FP64 rate for the tensor cores):
//  1. rank_users_score_kernel: score[q, i] = ((acc + b_u) + b_i) + mu in float64, acc = the in-order sum over d of
//     (double)u[d] * (double)v[d] (each product is exact in float64, so the FMA changes no bit).  A CTA scores a block of
//     32 query rows against 128 item rows, both staged in shared memory as doubles 32 dims at a time, 4 x 4 register
//     blocking per thread.  The grid is (item tiles x query blocks), so one query already spreads over every SM.
//  2. rank_users_select_kernel: per (query, chunk of RANK_CHUNK items) the exact top-k of the chunk: excluded items found
//     by binary search in the user's sorted list, a radix select (8-bit digits) on order-preserving keys of the float64
//     scores finds the k-th best, the survivors are bitonic-sorted (score descending, item id ascending).
//  3. rank_users_merge_kernel: one warp per query merges the sorted chunk lists into the final k, padding with (-inf, -1).
//     The chunks hold disjoint items and the order is total, so any chunking gives the same result.
// Scores of at most RANK_SCORE_BUDGET bytes exist at a time: larger query batches are scored and selected in passes.
//
// tfr_similar_rows (the neighbours of query rows in their own table, by float64 cosine) runs the same select and merge
// after two kernels of its own: row_norms_kernel (the norms of the candidate rows and of the query rows) and
// similar_rows_score_kernel, the scorer's main loop with a cosine epilogue.  A NaN score is never ranked, so the query's
// own row and zero rows need no exclusion list.
#include <math.h>
#include <string.h>

#include "common.cuh"
#include "rank_order.cuh"

namespace tfr {

constexpr int RU_QB = 32;          // query rows per scoring CTA
constexpr int RU_IT = 128;         // item rows per scoring CTA
constexpr int RU_DK = 32;          // dims staged per step
constexpr int RU_THREADS = 256;
constexpr int RU_SEL_THREADS = 256;
constexpr int RU_MIN_CHUNK = 1024;  // smallest selection chunk: the workspace is sized for it
constexpr int RU_MAX_CHUNK = 16384;
constexpr int RU_MAX_K = 1024;
constexpr int64_t RU_SCORE_BUDGET = (int64_t)1 << 30;   // bytes of float64 scores per pass

// ---- 1. scores -----------------------------------------------------------------------------------------------------------
// The main loop shared by the scorers: acc[x][y] = the in-order float64 dot product of query row ql = qrow + 4x of the
// CTA's block (s_qid[ql] = its table row, -1 if padding or out of range) and item row i0 + icol + 8y.  kAbsQuery / abs_item:
// the rows enter as |x|.  The epilogue gets (acc, s_qid, q0, qrow, i0, icol); a warp of padding rows does not call it.
// tid is threadIdx.x read in the kernel, where __launch_bounds__ bounds it: read here, its range is lost, the loads are
// unrolled differently, and rank_users_score_kernel would no longer compile to the instructions it had as a plain kernel.
template <bool kAbsQuery, class Epilogue>
__device__ __forceinline__ void ru_score_tile(const float* __restrict__ U, const float* __restrict__ V, int n_users,
                                              int n_items, int dim, int64_t us, int64_t is, bool abs_item,
                                              const int32_t* __restrict__ query, int nb, int tid, Epilogue epi) {
  __shared__ double sU[RU_DK][RU_QB + 1];
  __shared__ double sV[RU_DK][RU_IT + 1];
  __shared__ int s_qid[RU_QB];
  const int i0 = blockIdx.x * RU_IT, q0 = blockIdx.y * RU_QB;
  const int lane = tid & 31, w = tid >> 5;
  const int tx = lane & 7, ty = lane >> 3;
  const int wq = w >> 2, wi = w & 3;
  if (tid < RU_QB) {
    const int q = q0 + tid;
    int id = q < nb ? query[q] : -1;
    s_qid[tid] = (id >= 0 && id < n_users) ? id : -1;   // ids are device data: guarded here
  }
  const bool active = q0 + wq * 16 < nb;   // (warp-uniform) a warp whose 16 query rows are all padding computes nothing
  double acc[4][4];
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int b = 0; b < 4; ++b) acc[a][b] = 0.0;
  __syncthreads();
  for (int d0 = 0; d0 < dim; d0 += RU_DK) {
    // coalesced: a warp reads 32 consecutive dims of one row
    for (int e = tid; e < RU_IT * RU_DK; e += RU_THREADS) {
      const int r = e / RU_DK, dd = e % RU_DK;
      float x = 0.0f;
      if (i0 + r < n_items && d0 + dd < dim) x = V[(size_t)(i0 + r) * is + d0 + dd];
      sV[dd][r] = (double)(abs_item ? fabsf(x) : x);
    }
    for (int e = tid; e < RU_QB * RU_DK; e += RU_THREADS) {
      const int r = e / RU_DK, dd = e % RU_DK;
      const int id = s_qid[r];
      const float x = (id >= 0 && d0 + dd < dim) ? U[(size_t)id * us + d0 + dd] : 0.0f;
      sU[dd][r] = (double)(kAbsQuery ? fabsf(x) : x);
    }
    __syncthreads();
    if (active) {
      const int kmax = min(RU_DK, dim - d0);   // d stays in order: padding dims are never added
      for (int kk = 0; kk < kmax; ++kk) {
        double a[4], b[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) { a[j] = sU[kk][wq * 16 + ty + 4 * j]; b[j] = sV[kk][wi * 32 + tx + 8 * j]; }
#pragma unroll
        for (int x = 0; x < 4; ++x)
#pragma unroll
          for (int y = 0; y < 4; ++y) acc[x][y] = __fma_rn(a[x], b[y], acc[x][y]);
      }
    }
    __syncthreads();
  }
  if (!active) return;
  epi(acc, s_qid, q0, wq * 16 + ty, i0, wi * 32 + tx);
}

__global__ void __launch_bounds__(RU_THREADS) rank_users_score_kernel(
    const float* __restrict__ U, const float* __restrict__ V, const float* __restrict__ ub, const float* __restrict__ ib,
    const float* __restrict__ mu, int n_users, int n_items, int dim, int64_t us, int64_t is, bool abs_item,
    const int32_t* __restrict__ query, int nb, double* __restrict__ scores) {
  ru_score_tile<false>(U, V, n_users, n_items, dim, us, is, abs_item, query, nb, threadIdx.x,
                [&](const double (&acc)[4][4], const int* s_qid, int q0, int qrow, int i0, int icol) {
    const double m = (double)mu[0];
#pragma unroll
    for (int x = 0; x < 4; ++x) {
      const int ql = qrow + 4 * x, q = q0 + ql;
      const int id = s_qid[ql];
      if (q >= nb || id < 0) continue;
      const double bu = (double)ub[id];
#pragma unroll
      for (int y = 0; y < 4; ++y) {
        const int it = i0 + icol + 8 * y;
        if (it < n_items) scores[(size_t)q * n_items + it] = __dadd_rn(__dadd_rn(__dadd_rn(acc[x][y], bu), (double)ib[it]), m);
      }
    }
  });
}

// tfr_similar_rows: cos = acc / (|q| |v|), each step correctly rounded.  NaN (never ranked, see ru_key) for the skipped
// row and for a zero denominator.  Every other score is finite or NaN already: the norms of finite float rows are finite
// and their product neither overflows nor underflows in float64, and an inf or NaN entry makes acc / (|q| |v|) a NaN.
template <bool kAbs>
__global__ void __launch_bounds__(RU_THREADS) similar_rows_score_kernel(
    const float* __restrict__ Q, const float* __restrict__ V, int n_query_rows, int n_rows, int dim, int64_t qs, int64_t vs,
    const int32_t* __restrict__ query, const int32_t* __restrict__ skip, int nb,
    const double* __restrict__ qnorm, const double* __restrict__ vnorm, double* __restrict__ scores) {
  ru_score_tile<kAbs>(Q, V, n_query_rows, n_rows, dim, qs, vs, kAbs, query, nb, threadIdx.x,
                [&](const double (&acc)[4][4], const int* s_qid, int q0, int qrow, int i0, int icol) {
    double vn[4];
#pragma unroll
    for (int y = 0; y < 4; ++y) vn[y] = i0 + icol + 8 * y < n_rows ? vnorm[i0 + icol + 8 * y] : 0.0;
#pragma unroll
    for (int x = 0; x < 4; ++x) {
      const int ql = qrow + 4 * x, q = q0 + ql;
      if (q >= nb || s_qid[ql] < 0) continue;
      const double qn = qnorm[q];
      const int sk = skip ? skip[q] : -1;
#pragma unroll
      for (int y = 0; y < 4; ++y) {
        const int it = i0 + icol + 8 * y;
        if (it >= n_rows) continue;
        const double den = __dmul_rn(qn, vn[y]);
        scores[(size_t)q * n_rows + it] = (it == sk || den == 0.0) ? __longlong_as_double(0x7ff8000000000000ll)
                                                                   : __ddiv_rn(acc[x][y], den);
      }
    }
  });
}

// The float64 norms of tfr_similar_rows: out[r] = sqrt(sum over d in order from 0.0 of (double)x[d]^2), x = table row r
// (rows == null) or rows[r] (0 for an id outside [0, n_table)).  A CTA stages 32 dims of its 128 rows in shared memory
// (a warp reads 32 consecutive dims of one row); each thread then sums its own row.
constexpr int RN_ROWS = 128;
__global__ void __launch_bounds__(RN_ROWS) row_norms_kernel(const float* __restrict__ X, int n_table, int64_t stride,
                                                            int dim, const int32_t* __restrict__ rows, int n,
                                                            double* __restrict__ out) {
  __shared__ float s[RN_ROWS][RU_DK + 1];
  __shared__ int s_row[RN_ROWS];
  const int r0 = blockIdx.x * RN_ROWS;
  {
    const int r = r0 + threadIdx.x;
    int id = r < n ? (rows ? rows[r] : r) : -1;
    s_row[threadIdx.x] = (id >= 0 && id < n_table) ? id : -1;
  }
  double acc = 0.0;
  __syncthreads();
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  for (int d0 = 0; d0 < dim; d0 += RU_DK) {
    for (int rr = w; rr < RN_ROWS; rr += RN_ROWS / 32) {
      const int id = s_row[rr];
      s[rr][lane] = (id >= 0 && d0 + lane < dim) ? X[(size_t)id * stride + d0 + lane] : 0.0f;
    }
    __syncthreads();
    const int kmax = min(RU_DK, dim - d0);
    for (int kk = 0; kk < kmax; ++kk) {
      const double x = (double)s[threadIdx.x][kk];
      acc = __fma_rn(x, x, acc);
    }
    __syncthreads();
  }
  if (r0 + threadIdx.x < n) out[r0 + threadIdx.x] = s_row[threadIdx.x] >= 0 ? __dsqrt_rn(acc) : 0.0;
}

// ---- 2. exact top-k of every (query, chunk) ----------------------------------------------------------------------------
// Order-preserving key of a float64 score (larger score <-> larger key); 0 = not rankable (excluded item, NaN score).
__device__ __forceinline__ uint64_t ru_key(double v) {
  if (isnan(v)) return 0;
  if (v == 0.0) v = 0.0;   // -0.0 and +0.0 compare equal: one key
  const uint64_t b = (uint64_t)__double_as_longlong(v);
  return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}
__device__ __forceinline__ double ru_unkey(uint64_t k) {
  const uint64_t b = (k >> 63) ? (k & 0x7fffffffffffffffull) : ~k;
  return __longlong_as_double((long long)b);
}

__global__ void __launch_bounds__(RU_SEL_THREADS) rank_users_select_kernel(
    const double* __restrict__ scores, int n_users, int n_items, const int32_t* __restrict__ query, int q_base, int n_chunks,
    int chunk, int k, const int64_t* __restrict__ excl_indptr, const int32_t* __restrict__ excl_item,
    double* __restrict__ part_val, int32_t* __restrict__ part_idx) {
  extern __shared__ uint64_t s_key[];   // [chunk]
  __shared__ uint64_t s_sk[RU_MAX_K];   // survivors: key, item id
  __shared__ int s_si[RU_MAX_K];
  __shared__ int s_hist[256];
  __shared__ int s_wsum[RU_SEL_THREADS / 32];
  __shared__ int s_bcast[4];
  const int ql = blockIdx.x / n_chunks, c = blockIdx.x % n_chunks;
  const int q = q_base + ql;
  const int c0 = c * chunk, len = min(chunk, n_items - c0);
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int id = query[q];
  double* ov = part_val + ((size_t)q * n_chunks + c) * k;
  int32_t* oi = part_idx + ((size_t)q * n_chunks + c) * k;
  if (id < 0 || id >= n_users) {
    for (int r = threadIdx.x; r < k; r += RU_SEL_THREADS) { ov[r] = -INFINITY; oi[r] = -1; }
    return;
  }
  const double* line = scores + (size_t)ql * n_items + c0;
  for (int t = threadIdx.x; t < len; t += RU_SEL_THREADS) s_key[t] = ru_key(line[t]);
  __syncthreads();
  if (excl_indptr) {   // the user's excluded ids inside [c0, c0 + len): binary search for the first, then walk
    int64_t lo = excl_indptr[id], hi = excl_indptr[id + 1];
    while (lo < hi) {
      const int64_t mid = (lo + hi) >> 1;
      if (excl_item[mid] < c0) lo = mid + 1; else hi = mid;
    }
    const int64_t x1 = excl_indptr[id + 1];
    for (int64_t p = lo + threadIdx.x; p < x1; p += RU_SEL_THREADS) {
      const int it = excl_item[p];
      if (it >= c0 + len) break;
      s_key[it - c0] = 0;
    }
    __syncthreads();
  }
  // rankable items of the chunk -> need = min(k, rankable)
  int cnt = 0;
  for (int t = threadIdx.x; t < len; t += RU_SEL_THREADS) cnt += s_key[t] != 0;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
  if (lane == 0) s_wsum[w] = cnt;
  __syncthreads();
  int rankable = 0;
#pragma unroll
  for (int j = 0; j < RU_SEL_THREADS / 32; ++j) rankable += s_wsum[j];
  const int need = min(k, rankable);
  // radix select, most significant byte first: T = the need-th largest key, rem = how many keys equal to T are taken
  uint64_t prefix = 0, mask = 0;
  int rem = need, eq_count = 0;
  if (need > 0) {
    for (int shift = 56; shift >= 0; shift -= 8) {
      for (int b = threadIdx.x; b < 256; b += RU_SEL_THREADS) s_hist[b] = 0;
      __syncthreads();
      for (int t = threadIdx.x; t < len; t += RU_SEL_THREADS) {
        const uint64_t key = s_key[t];
        if (key != 0 && (key & mask) == prefix) atomicAdd(&s_hist[(key >> shift) & 255], 1);
      }
      __syncthreads();
      if (w == 0) {   // lane l holds bins 255 - 8l .. 248 - 8l (descending); find the bin where the count reaches rem
        int h[8], s = 0;
#pragma unroll
        for (int j = 0; j < 8; ++j) { h[j] = s_hist[255 - 8 * lane - j]; s += h[j]; }
        int incl = s;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const int y = __shfl_up_sync(0xffffffffu, incl, o);
          if (lane >= o) incl += y;
        }
        const int excl = incl - s;
        if (excl < rem && incl >= rem) {
          int above = excl;
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            if (above + h[j] >= rem) { s_bcast[0] = 255 - 8 * lane - j; s_bcast[1] = rem - above; s_bcast[2] = h[j]; break; }
            above += h[j];
          }
        }
      }
      __syncthreads();
      prefix |= (uint64_t)s_bcast[0] << shift;
      mask |= (uint64_t)255 << shift;
      rem = s_bcast[1];
      eq_count = s_bcast[2];
      __syncthreads();
    }
  }
  // survivors: every key > T, and the rem keys == T of the lowest item ids
  if (threadIdx.x == 0) s_bcast[3] = 0;
  __syncthreads();
  if (need > 0) {
    const uint64_t T = prefix;
    const bool all_eq = eq_count == rem;
    for (int t = threadIdx.x; t < len; t += RU_SEL_THREADS) {
      const uint64_t key = s_key[t];
      if (key > T || (all_eq && key == T)) {
        const int slot = atomicAdd(&s_bcast[3], 1);
        s_sk[slot] = key;
        s_si[slot] = c0 + t;
      }
    }
    if (!all_eq) {   // ties at the threshold: take them in item order (block-wide scan, 256 positions at a time)
      int taken = 0;
      for (int base = 0; base < len; base += RU_SEL_THREADS) {
        const int t = base + threadIdx.x;
        const bool f = t < len && s_key[t] == T;
        const unsigned bal = __ballot_sync(0xffffffffu, f);
        __syncthreads();
        if (lane == 0) s_wsum[w] = __popc(bal);
        __syncthreads();
        int before = taken, total = 0;
#pragma unroll
        for (int j = 0; j < RU_SEL_THREADS / 32; ++j) {
          if (j < w) before += s_wsum[j];
          total += s_wsum[j];
        }
        before += __popc(bal & ((1u << lane) - 1u));
        if (f && before < rem) {
          const int slot = atomicAdd(&s_bcast[3], 1);
          s_sk[slot] = T;
          s_si[slot] = c0 + t;
        }
        taken += total;
        if (taken >= rem) break;   // (uniform)
      }
    }
  }
  __syncthreads();
  // bitonic sort of the need survivors, padded to a power of two: key descending, item id ascending
  int P = 1;
  while (P < need) P <<= 1;
  for (int t = need + threadIdx.x; t < P; t += RU_SEL_THREADS) { s_sk[t] = 0; s_si[t] = 0x7fffffff; }
  __syncthreads();
  for (int size = 2; size <= P; size <<= 1) {
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      for (int t = threadIdx.x; t < P; t += RU_SEL_THREADS) {
        const int o = t ^ stride;
        if (o > t) {
          const uint64_t ka = s_sk[t], kb = s_sk[o];
          const int ia = s_si[t], ib_ = s_si[o];
          const bool a_first = ka > kb || (ka == kb && ia < ib_);
          const bool want_first = (t & size) == 0;   // this half of the bitonic sequence goes in rank order
          if (a_first != want_first) { s_sk[t] = kb; s_sk[o] = ka; s_si[t] = ib_; s_si[o] = ia; }
        }
      }
      __syncthreads();
    }
  }
  for (int r = threadIdx.x; r < k; r += RU_SEL_THREADS) {
    if (r < need) { ov[r] = ru_unkey(s_sk[r]); oi[r] = s_si[r]; }
    else { ov[r] = -INFINITY; oi[r] = -1; }
  }
}

// ---- 3. merge of the sorted chunk lists: one warp per query -----------------------------------------------------------
// (the order and the warp arg-best step: rank_order.cuh, shared with the merge of item shards)
constexpr int RU_MERGE_WARPS = 4;
__global__ void __launch_bounds__(32 * RU_MERGE_WARPS) rank_users_merge_kernel(
    const double* __restrict__ part_val, const int32_t* __restrict__ part_idx, int32_t* __restrict__ heads, int n, int n_chunks,
    int k, double* __restrict__ out_val, int32_t* __restrict__ out_idx) {
  const int lane = threadIdx.x & 31;
  const int q = blockIdx.x * RU_MERGE_WARPS + (threadIdx.x >> 5);
  if (q >= n) return;
  const double* pv = part_val + (size_t)q * n_chunks * k;
  const int32_t* pi = part_idx + (size_t)q * n_chunks * k;
  int32_t* hd = heads + (size_t)q * n_chunks;
  for (int c = lane; c < n_chunks; c += 32) hd[c] = 0;
  __syncwarp();
  // each lane keeps the best head among its lists c = lane, lane + 32, ...; only the winning lane rescans
  auto scan = [&](double& bv, int& bi, int& bc) {
    bv = -INFINITY; bi = -1; bc = -1;
    for (int c = lane; c < n_chunks; c += 32) {
      const int h = hd[c];
      if (h >= k) continue;
      const double v = pv[(size_t)c * k + h];
      const int i = pi[(size_t)c * k + h];
      if (ru_before(v, i, bv, bi)) { bv = v; bi = i; bc = c; }
    }
  };
  double bv;
  int bi, bc;
  scan(bv, bi, bc);
  for (int r = 0; r < k; ++r) {
    double wv = bv;
    int wi = bi, wl = lane;
    ru_warp_best(wv, wi, wl);
    if (wi < 0) {   // every list is exhausted: pad the rest
      for (int rr = r + lane; rr < k; rr += 32) { out_val[(size_t)q * k + rr] = -INFINITY; out_idx[(size_t)q * k + rr] = -1; }
      return;
    }
    if (lane == 0) { out_val[(size_t)q * k + r] = wv; out_idx[(size_t)q * k + r] = wi; }
    if (lane == wl) {
      hd[bc] += 1;
      scan(bv, bi, bc);
    }
    __syncwarp();
  }
}

static int ru_chunk_items() {
  int c = tune(TUNE_RANK_CHUNK);
  if (c < RU_MIN_CHUNK) c = RU_MIN_CHUNK;
  if (c > RU_MAX_CHUNK) c = RU_MAX_CHUNK;
  return (c + RU_MIN_CHUNK - 1) / RU_MIN_CHUNK * RU_MIN_CHUNK;   // a multiple of the smallest chunk: never more chunks
}

static int64_t ru_pass_queries(int64_t n, int64_t n_items) {
  const int64_t per = n_items > 0 ? n_items * 8 : 8;
  int64_t nb = RU_SCORE_BUDGET / per;
  if (nb < 1) nb = 1;
  if (nb > 65535 * (int64_t)RU_QB) nb = 65535 * (int64_t)RU_QB;
  return nb < n ? nb : n;
}

}  // namespace tfr

using namespace tfr;

extern "C" int64_t tfr_rank_users_workspace_bytes(int64_t n_queries, int64_t n_items, int32_t k) {
  if (n_queries < 0 || n_items < 0 || n_items >= ((int64_t)1 << 31) || k < 1 || k > RU_MAX_K) return TFR_ERR_INVALID;
  const int64_t chunks = (n_items + RU_MIN_CHUNK - 1) / RU_MIN_CHUNK;
  const int64_t parts = n_queries * chunks * k;
  return 256 + align_up(ru_pass_queries(n_queries, n_items) * n_items * 8, 256) + align_up(parts * 8, 256) +
         align_up(parts * 4, 256) + align_up(n_queries * chunks * 4, 256);
}

// The passes of both entries: score(q0, nb, scores) scores queries q0 .. q0 + nb - 1 into scores [nb, n_items], then the
// chunks are selected and merged.  query / n_query_rows: what the select kernel checks the ids against.
template <class Score>
static int ru_rank(Score score, const int32_t* query, int64_t n_query_rows, int64_t n_queries, int64_t n_items, int32_t k,
                   const int64_t* excl_indptr, const int32_t* excl_item, double* topk_val, int32_t* topk_idx, void* workspace,
                   cudaStream_t st) {
  const int chunk = ru_chunk_items();
  const int n_chunks = (int)((n_items + chunk - 1) / chunk);
  const int64_t max_chunks = (n_items + RU_MIN_CHUNK - 1) / RU_MIN_CHUNK;
  const int64_t nb_max = ru_pass_queries(n_queries, n_items);
  char* w = reinterpret_cast<char*>(align_up((int64_t)(uintptr_t)workspace, 256));
  double* scores = reinterpret_cast<double*>(w); w += align_up(nb_max * n_items * 8, 256);
  double* part_val = reinterpret_cast<double*>(w); w += align_up(n_queries * max_chunks * k * 8, 256);
  int32_t* part_idx = reinterpret_cast<int32_t*>(w); w += align_up(n_queries * max_chunks * k * 4, 256);
  int32_t* heads = reinterpret_cast<int32_t*>(w);
  const int stages = tune(TUNE_RANK_STAGES);
  if (n_chunks > 0) {
    const size_t smem = (size_t)chunk * 8;
    TFR_CUDA(cudaFuncSetAttribute(rank_users_select_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    for (int64_t q0 = 0; q0 < n_queries; q0 += nb_max) {
      const int nb = (int)(n_queries - q0 < nb_max ? n_queries - q0 : nb_max);
      if (stages & 1) {
        score(q0, nb, scores);
        TFR_LAUNCH_CHECK();
      }
      if (stages & 2) {
        rank_users_select_kernel<<<(unsigned)((int64_t)nb * n_chunks), RU_SEL_THREADS, smem, st>>>(
            scores, (int)n_query_rows, (int)n_items, query, (int)q0, n_chunks, chunk, k, excl_indptr, excl_item, part_val,
            part_idx);
        TFR_LAUNCH_CHECK();
      }
    }
  }
  if (stages & 4) {
    rank_users_merge_kernel<<<(unsigned)((n_queries + RU_MERGE_WARPS - 1) / RU_MERGE_WARPS), 32 * RU_MERGE_WARPS, 0, st>>>(
        part_val, part_idx, heads, (int)n_queries, n_chunks, k, topk_val, topk_idx);
    TFR_LAUNCH_CHECK();
  }
  return TFR_OK;
}

extern "C" int tfr_rank_users(const float* user_feat, const float* item_feat, const float* user_bias, const float* item_bias,
                              const float* mu, int64_t n_users, int64_t n_items, int32_t dim, int64_t user_stride,
                              int64_t item_stride, int32_t flags, const int32_t* query_users, int64_t n_queries, int32_t k,
                              const int64_t* excl_indptr, const int32_t* excl_item, double* topk_val, int32_t* topk_idx,
                              void* workspace, int64_t workspace_bytes, void* stream) {
  TFR_CHECK_ARG(dim >= 1 && dim <= 512 && k >= 1 && k <= RU_MAX_K);
  TFR_CHECK_ARG(n_users >= 0 && n_users < ((int64_t)1 << 31) && n_items >= 0 && n_items < ((int64_t)1 << 31));
  TFR_CHECK_ARG(n_queries >= 0 && n_queries < ((int64_t)1 << 31));
  if (user_stride == 0) user_stride = dim;
  if (item_stride == 0) item_stride = dim;
  TFR_CHECK_ARG(user_stride >= dim && item_stride >= dim);
  TFR_CHECK_ARG(!excl_indptr || excl_item);
  if (n_queries == 0) return TFR_OK;
  TFR_CHECK_ARG(query_users && topk_val && topk_idx);
  TFR_CHECK_ARG(n_items == 0 || (user_feat && item_feat && user_bias && item_bias && mu));
  const int64_t need = tfr_rank_users_workspace_bytes(n_queries, n_items, k);
  if (!workspace || workspace_bytes < need) {
    set_error("rank_users workspace too small (%lld bytes, need %lld)", (long long)workspace_bytes, (long long)need);
    return TFR_ERR_WORKSPACE;
  }
  cudaStream_t st = (cudaStream_t)stream;
  const bool abs_item = (flags & TFR_ABS_ITEM) != 0;
  auto score = [&](int64_t q0, int nb, double* scores) {
    dim3 grid((unsigned)((n_items + RU_IT - 1) / RU_IT), (unsigned)((nb + RU_QB - 1) / RU_QB));
    rank_users_score_kernel<<<grid, RU_THREADS, 0, st>>>(user_feat, item_feat, user_bias, item_bias, mu, (int)n_users,
                                                         (int)n_items, dim, user_stride, item_stride, abs_item,
                                                         query_users + q0, nb, scores);
  };
  return ru_rank(score, query_users, n_users, n_queries, n_items, k, excl_indptr, excl_item, topk_val, topk_idx, workspace,
                 st);
}

extern "C" int64_t tfr_similar_rows_workspace_bytes(int64_t n_queries, int64_t n_rows, int32_t k) {
  const int64_t ru = tfr_rank_users_workspace_bytes(n_queries, n_rows, k);
  if (ru < 0) return ru;
  return ru + align_up(n_rows * 8, 256) + align_up(n_queries * 8, 256);
}

extern "C" int tfr_similar_rows(const float* query_feat, int64_t n_query_rows, int64_t query_stride,
                                const int32_t* query_rows, const int32_t* skip, int64_t n_queries, const float* feat,
                                int64_t n_rows, int64_t stride, int32_t dim, int32_t abs_rows, int32_t k, double* topk_val,
                                int32_t* topk_idx, void* workspace, int64_t workspace_bytes, void* stream) {
  TFR_CHECK_ARG(dim >= 1 && dim <= 512 && k >= 1 && k <= RU_MAX_K);
  TFR_CHECK_ARG(n_query_rows >= 0 && n_query_rows < ((int64_t)1 << 31) && n_rows >= 0 && n_rows < ((int64_t)1 << 31));
  TFR_CHECK_ARG(n_queries >= 0 && n_queries < ((int64_t)1 << 31));
  if (query_stride == 0) query_stride = dim;
  if (stride == 0) stride = dim;
  TFR_CHECK_ARG(query_stride >= dim && stride >= dim);
  if (n_queries == 0) return TFR_OK;
  TFR_CHECK_ARG(query_rows && topk_val && topk_idx);
  TFR_CHECK_ARG(n_query_rows == 0 || query_feat);
  TFR_CHECK_ARG(n_rows == 0 || feat);
  const int64_t need = tfr_similar_rows_workspace_bytes(n_queries, n_rows, k);
  if (!workspace || workspace_bytes < need) {
    set_error("similar_rows workspace too small (%lld bytes, need %lld)", (long long)workspace_bytes, (long long)need);
    return TFR_ERR_WORKSPACE;
  }
  cudaStream_t st = (cudaStream_t)stream;
  // the norms go after the ranking's part of the workspace (ru_rank carves that from the aligned start)
  char* w = reinterpret_cast<char*>(align_up((int64_t)(uintptr_t)workspace, 256)) +
            (tfr_rank_users_workspace_bytes(n_queries, n_rows, k) - 256);
  double* vnorm = reinterpret_cast<double*>(w); w += align_up(n_rows * 8, 256);
  double* qnorm = reinterpret_cast<double*>(w);
  if (n_rows > 0 && (tune(TUNE_RANK_STAGES) & 1)) {
    row_norms_kernel<<<(unsigned)((n_rows + RN_ROWS - 1) / RN_ROWS), RN_ROWS, 0, st>>>(feat, (int)n_rows, stride, dim, nullptr,
                                                                                       (int)n_rows, vnorm);
    TFR_LAUNCH_CHECK();
    row_norms_kernel<<<(unsigned)((n_queries + RN_ROWS - 1) / RN_ROWS), RN_ROWS, 0, st>>>(
        query_feat, (int)n_query_rows, query_stride, dim, query_rows, (int)n_queries, qnorm);
    TFR_LAUNCH_CHECK();
  }
  auto score = [&](int64_t q0, int nb, double* scores) {
    dim3 grid((unsigned)((n_rows + RU_IT - 1) / RU_IT), (unsigned)((nb + RU_QB - 1) / RU_QB));
    auto kern = abs_rows ? similar_rows_score_kernel<true> : similar_rows_score_kernel<false>;
    kern<<<grid, RU_THREADS, 0, st>>>(query_feat, feat, (int)n_query_rows, (int)n_rows, dim, query_stride, stride,
                                      query_rows + q0, skip ? skip + q0 : nullptr, nb, qnorm + q0, vnorm, scores);
  };
  return ru_rank(score, query_rows, n_query_rows, n_queries, n_rows, k, nullptr, nullptr, topk_val, topk_idx, workspace, st);
}
