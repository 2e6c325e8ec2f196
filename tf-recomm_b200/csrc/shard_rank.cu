// Serving from row-sharded tables: exact top-k over items that live on G ranks (item i on rank i mod G, local row i / G).
// Every rank ranks its own item shard with tfr_rank_users, unchanged, against the same query rows (gathered to every rank
// by tfr_shard_gather_rows + an all-reduce).  Two pieces around that call live here:
//  1. shard_excl_count_kernel / shard_excl_fill_kernel: per query row, the excluded items this rank owns, as ascending
//     LOCAL ids in a CSR indexed by query position -- count -> scan (scan.cuh) -> fill, one warp per query.  The cost is
//     the length of the query rows' source lists, whatever the number of users or pairs of the source CSR.
//  2. shard_topk_merge_kernel: the all-gathered per-rank lists [G][n][k] merged into the global top k, one warp per query,
//     lane g holding the head of rank g's list in registers (G <= SHARD_MAX_RANKS <= 32).  Local id i of rank g is global
//     id i * G + g.  The order is rank_order.cuh's, the one tfr_rank_users merges its item chunks by: an item shard is one
//     more split of the items into disjoint sets, so the result is the single-table ranking, ids and bits.
#include "common.cuh"
#include "rank_order.cuh"
#include "scan.cuh"

namespace tfr {

constexpr int SX_WARPS = 8;          // queries per CTA of the exclusion-list kernels
constexpr int STM_WARPS = 4;         // queries per CTA of the merge
constexpr int STM_MAX_K = 1024;      // tfr_rank_users' largest k

__global__ void __launch_bounds__(32 * SX_WARPS) shard_excl_count_kernel(
    const int64_t* __restrict__ indptr, const int32_t* __restrict__ items, int n_rows, const int32_t* __restrict__ rows,
    int n, int G, int rank, int32_t* __restrict__ counts) {
  const int lane = threadIdx.x & 31;
  const int q = blockIdx.x * SX_WARPS + (threadIdx.x >> 5);
  if (q >= n) return;
  const int r = rows[q];
  int c = 0;
  if (r >= 0 && r < n_rows) {   // rows are device data: guarded here
    const int64_t p1 = indptr[r + 1];
    for (int64_t p = indptr[r] + lane; p < p1; p += 32) {
      const int it = items[p];
      c += it >= 0 && it % G == rank;
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
  if (lane == 0) counts[q] = c;
}

// the owned items of each query row in source order (ascending ids stay ascending: i -> i / G is monotone within a residue)
__global__ void __launch_bounds__(32 * SX_WARPS) shard_excl_fill_kernel(
    const int64_t* __restrict__ indptr, const int32_t* __restrict__ items, int n_rows, const int32_t* __restrict__ rows,
    int n, int G, int rank, const int64_t* __restrict__ out_indptr, int32_t* __restrict__ out_items) {
  const int lane = threadIdx.x & 31;
  const int q = blockIdx.x * SX_WARPS + (threadIdx.x >> 5);
  if (q >= n) return;
  const int r = rows[q];
  if (r < 0 || r >= n_rows) return;
  int64_t o = out_indptr[q];
  const int64_t p1 = indptr[r + 1];
  for (int64_t p0 = indptr[r]; p0 < p1; p0 += 32) {   // (warp-uniform)
    const int64_t p = p0 + lane;
    const int it = p < p1 ? items[p] : -1;
    const bool f = it >= 0 && it % G == rank;
    const unsigned bal = __ballot_sync(0xffffffffu, f);
    if (f) out_items[o + __popc(bal & ((1u << lane) - 1u))] = it / G;
    o += __popc(bal);
  }
}

__global__ void __launch_bounds__(32 * STM_WARPS) shard_topk_merge_kernel(
    const double* __restrict__ val, const int32_t* __restrict__ idx, int G, int n, int k, double* __restrict__ out_val,
    int32_t* __restrict__ out_idx) {
  const int lane = threadIdx.x & 31;
  const int q = blockIdx.x * STM_WARPS + (threadIdx.x >> 5);
  if (q >= n) return;
  int h = 0;              // lane g < G: position of the head of rank g's list
  double hv = -INFINITY;  // ... and its entry, with the global id; (-inf, -1) once the list is exhausted
  int hi = -1;
  auto load = [&]() {
    hv = -INFINITY;
    hi = -1;
    if (lane < G && h < k) {
      const size_t at = ((size_t)lane * n + q) * k + h;
      const int i = idx[at];
      if (i >= 0) { hv = val[at]; hi = i * G + lane; }   // a list ends at its first -1
    }
  };
  load();
  for (int r = 0; r < k; ++r) {
    double wv = hv;
    int wi = hi, wl = lane;
    ru_warp_best(wv, wi, wl);
    if (wi < 0) {   // every list is exhausted: pad the rest
      for (int rr = r + lane; rr < k; rr += 32) { out_val[(size_t)q * k + rr] = -INFINITY; out_idx[(size_t)q * k + rr] = -1; }
      return;
    }
    if (lane == 0) { out_val[(size_t)q * k + r] = wv; out_idx[(size_t)q * k + r] = wi; }
    if (lane == wl) {
      ++h;
      load();
    }
  }
}

static int excl_args(const int64_t* indptr, int64_t n_rows, const int32_t* rows, int64_t n, int32_t n_ranks, int32_t rank,
                     const int64_t* out_indptr) {
  TFR_CHECK_ARG(n >= 0 && n < ((int64_t)1 << 31) && n_rows >= 0 && n_rows < ((int64_t)1 << 31));
  TFR_CHECK_ARG(n_ranks >= 1 && n_ranks <= SHARD_MAX_RANKS && rank >= 0 && rank < n_ranks);
  TFR_CHECK_ARG(out_indptr);
  TFR_CHECK_ARG(n == 0 || (indptr && rows));
  return TFR_OK;
}

}  // namespace tfr

using namespace tfr;

extern "C" int64_t tfr_shard_excl_workspace_bytes(int64_t n) {
  if (n < 0 || n >= ((int64_t)1 << 31)) return TFR_ERR_INVALID;
  return 256 + align_up(n * 4, 256) + align_up(scan_tiles(n) * 8, 256);
}

extern "C" int tfr_shard_excl_indptr(const int64_t* indptr, const int32_t* items, int64_t n_rows, const int32_t* rows,
                                     int64_t n, int32_t n_ranks, int32_t rank, int64_t* out_indptr, void* workspace,
                                     int64_t workspace_bytes, void* stream) {
  int rc = excl_args(indptr, n_rows, rows, n, n_ranks, rank, out_indptr);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  if (n == 0) {
    TFR_CUDA(cudaMemsetAsync(out_indptr, 0, sizeof(int64_t), st));
    return TFR_OK;
  }
  if (!workspace || workspace_bytes < tfr_shard_excl_workspace_bytes(n)) {
    set_error("shard exclusion-list workspace too small (%lld bytes, need %lld)", (long long)workspace_bytes,
              (long long)tfr_shard_excl_workspace_bytes(n));
    return TFR_ERR_WORKSPACE;
  }
  char* w = reinterpret_cast<char*>(align_up((int64_t)(uintptr_t)workspace, 256));
  int32_t* counts = (int32_t*)w;
  int64_t* tiles = (int64_t*)(w + align_up(n * 4, 256));
  shard_excl_count_kernel<<<(unsigned)((n + SX_WARPS - 1) / SX_WARPS), 32 * SX_WARPS, 0, st>>>(
      indptr, items, (int)n_rows, rows, (int)n, n_ranks, rank, counts);
  TFR_LAUNCH_CHECK();
  return exclusive_scan(counts, n, out_indptr, tiles, st);
}

extern "C" int tfr_shard_excl_fill(const int64_t* indptr, const int32_t* items, int64_t n_rows, const int32_t* rows,
                                   int64_t n, int32_t n_ranks, int32_t rank, const int64_t* out_indptr, int32_t* out_items,
                                   void* stream) {
  int rc = excl_args(indptr, n_rows, rows, n, n_ranks, rank, out_indptr);
  if (rc) return rc;
  if (n == 0) return TFR_OK;
  shard_excl_fill_kernel<<<(unsigned)((n + SX_WARPS - 1) / SX_WARPS), 32 * SX_WARPS, 0, (cudaStream_t)stream>>>(
      indptr, items, (int)n_rows, rows, (int)n, n_ranks, rank, out_indptr, out_items);
  TFR_LAUNCH_CHECK();
  return TFR_OK;
}

extern "C" int tfr_shard_topk_merge(const double* val, const int32_t* idx, int32_t n_ranks, int64_t n, int32_t k,
                                    double* out_val, int32_t* out_idx, void* stream) {
  TFR_CHECK_ARG(n_ranks >= 1 && n_ranks <= SHARD_MAX_RANKS && k >= 1 && k <= STM_MAX_K);
  TFR_CHECK_ARG(n >= 0 && n < ((int64_t)1 << 31));
  if (n == 0) return TFR_OK;
  TFR_CHECK_ARG(val && idx && out_val && out_idx);
  shard_topk_merge_kernel<<<(unsigned)((n + STM_WARPS - 1) / STM_WARPS), 32 * STM_WARPS, 0, (cudaStream_t)stream>>>(
      val, idx, n_ranks, (int)n, k, out_val, out_idx);
  TFR_LAUNCH_CHECK();
  return TFR_OK;
}
