// Device-side pieces around the hot path that the reference computes on the host:
//   * the DISCRETE branch's metrics (svd_train_val.py:94-98,138-143): summed sigmoid cross-entropy (cost_nll), accuracy of
//     round(sigmoid(logits)) and the area under the ROC curve (sklearn.metrics.roc_auc_score = the rank statistic with
//     tied scores averaged) -- sort-based, reusing the step's stable radix sort (dedup_sort.cu) on order-preserving keys
//     of the fp32 probabilities;
//   * the KTM sparse design matrix of fm.py:61-93 (df_to_sparse: one block per active agent, hstacked) built as CSR
//     directly in HBM: count -> scan -> fill.
// Both need a prefix sum: the three-phase exclusive scan of scan.cuh, deterministic.
//   * top-k ranking metrics (hit rate, precision, recall, NDCG at k) of a ranking against a held-out relevant set.
#include <string.h>

#include "common.cuh"
#include "scan.cuh"

namespace tfr {

// ================================ binary metrics ========================================================================
// float -> uint32 whose unsigned order is the float order (negative floats reversed, sign bit flipped)
__device__ __forceinline__ uint32_t float_order_key(float f) {
  const uint32_t u = __float_as_uint(f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

// per element: p = sigmoid(x) as ops.sigmoid does (ops.py:94-95: 1 / (1 + exp(-x)), fp32), its sort key, the summed
// sigmoid cross-entropy (TF: max(x,0) - x*z + log1p(exp(-|x|)), float64 accumulation like np.sum of svd_train_val's
// per-batch costs) and the number of correct round(p) == label (svd_train_val.py:96,140).  Per-CTA partials, folded in
// a fixed order by metrics_finish_kernel.
__global__ void __launch_bounds__(256) metrics_elementwise_kernel(const float* __restrict__ logits,
                                                                  const float* __restrict__ labels, int64_t n,
                                                                  int32_t* __restrict__ keys, double* __restrict__ part) {
  __shared__ double s_nll[256], s_ok[256], s_pos[256];
  double nll = 0.0, okc = 0.0, pos = 0.0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const float x = logits[i], z = labels[i];
    const float p = sigmoid_tf(x);
    keys[i] = (int32_t)float_order_key(p);
    const float ce = add_rn(sub_rn(fmaxf(x, 0.0f), mul_rn(x, z)), log1pf(expf(-fabsf(x))));
    nll += (double)ce;
    okc += (rintf(p) == z) ? 1.0 : 0.0;
    pos += (z > 0.5f) ? 1.0 : 0.0;
  }
  s_nll[threadIdx.x] = nll; s_ok[threadIdx.x] = okc; s_pos[threadIdx.x] = pos;
  __syncthreads();
  if (threadIdx.x == 0) {
    double a = 0.0, b = 0.0, c = 0.0;
    for (int j = 0; j < 256; ++j) { a += s_nll[j]; b += s_ok[j]; c += s_pos[j]; }
    part[blockIdx.x * 3 + 0] = a; part[blockIdx.x * 3 + 1] = b; part[blockIdx.x * 3 + 2] = c;
  }
}

// over the SORTED keys: flags[k] = 1 where a run of equal keys ENDS at k; posf[k] = 1 where the element is a positive
__global__ void __launch_bounds__(256) metrics_flags_kernel(const int32_t* __restrict__ skeys, const int32_t* __restrict__ spos,
                                                            const float* __restrict__ labels, int64_t n,
                                                            int32_t* __restrict__ endf, int32_t* __restrict__ posf) {
  const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n) return;
  endf[k] = (k + 1 == n || skeys[k + 1] != skeys[k]) ? 1 : 0;
  posf[k] = labels[spos[k]] > 0.5f ? 1 : 0;
}

// at every run end: the run's record (positives up to and including it, elements up to and including it), indexed by the
// run's number (= run ends strictly before k)
__global__ void __launch_bounds__(256) metrics_runs_kernel(const int32_t* __restrict__ endf, const int64_t* __restrict__ end_ex,
                                                           const int64_t* __restrict__ pos_ex, const int32_t* __restrict__ posf,
                                                           int64_t n, int64_t* __restrict__ run_pos, int64_t* __restrict__ run_cnt) {
  const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n || !endf[k]) return;
  const int64_t r = end_ex[k];
  run_pos[r] = pos_ex[k] + posf[k];
  run_cnt[r] = k + 1;
}

// AUC = sum over runs of pos_run * (neg_before + neg_run / 2) / (n_pos * n_neg): every positive counts the negatives
// ranked below it, tied ones half (average ranks: what roc_auc_score's trapezoids give).  Fixed-order sum (one CTA).
__global__ void __launch_bounds__(1024) metrics_finish_kernel(const int64_t* __restrict__ run_pos, const int64_t* __restrict__ run_cnt,
                                                             const int64_t* __restrict__ end_ex, int64_t n,
                                                             const double* __restrict__ part, int n_part,
                                                             double* __restrict__ out) {
  __shared__ double s_sum[1024];
  const int64_t n_runs = end_ex[n];
  double acc = 0.0;
  for (int64_t r = threadIdx.x; r < n_runs; r += 1024) {
    const int64_t p1 = run_pos[r], c1 = run_cnt[r];
    const int64_t p0 = r ? run_pos[r - 1] : 0, c0 = r ? run_cnt[r - 1] : 0;
    const double pos_run = (double)(p1 - p0), neg_run = (double)((c1 - c0) - (p1 - p0)), neg_before = (double)(c0 - p0);
    acc += pos_run * (neg_before + 0.5 * neg_run);
  }
  s_sum[threadIdx.x] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double tot = 0.0, nll = 0.0, okc = 0.0, pos = 0.0;
    for (int j = 0; j < 1024; ++j) tot += s_sum[j];
    for (int j = 0; j < n_part; ++j) { nll += part[j * 3]; okc += part[j * 3 + 1]; pos += part[j * 3 + 2]; }
    const double neg = (double)n - pos;
    out[0] = nll;                                                        // summed sigmoid cross-entropy (cost_nll)
    out[1] = okc;                                                        // correct predictions
    out[2] = (pos > 0.0 && neg > 0.0) ? tot / (pos * neg) : nan("");     // roc_auc_score (undefined with one class)
    out[3] = pos;
  }
}

// ================================ ranking metrics at k ==================================================================
// One warp per ranked row u (grid-stride over the rows), relevant set R_u as CSR (strictly ascending item ids); a ranked
// id is a hit when a binary search finds it in R_u (-1 never does).  Per row, with h_r the hit flag of rank r:
//   HR = [sum h_r >= 1], precision = sum h_r / k, recall = sum h_r / |R_u|,
//   NDCG = (sum_r h_r / log2(r + 2)) / (sum_{r < min(k, |R_u|)} 1 / log2(r + 2))          (float64)
// Rows with |R_u| = 0 are not evaluated.  Each block folds its warps' sums in warp order into part[block][5]; one block
// folds the partials in a fixed order (ranking_metrics_finish_kernel): no floating-point atomics, the same bits every run.
constexpr int RM_WARPS = 8, RM_MAX_BLOCKS = 1024;
__global__ void __launch_bounds__(32 * RM_WARPS) ranking_metrics_rows_kernel(const int32_t* __restrict__ topk_idx, int64_t n_rows,
                                                                            int k, const int64_t* __restrict__ rel_indptr,
                                                                            const int32_t* __restrict__ rel_item,
                                                                            double* __restrict__ row_metrics,
                                                                            double* __restrict__ part) {
  __shared__ double s_acc[RM_WARPS][5];
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  double acc[5] = {0.0, 0.0, 0.0, 0.0, 0.0};   // (HR, precision, recall, NDCG, evaluated rows): lane 0's copy counts
  for (int64_t u = (int64_t)blockIdx.x * RM_WARPS + w; u < n_rows; u += (int64_t)gridDim.x * RM_WARPS) {
    const int64_t r0 = rel_indptr[u], r1 = rel_indptr[u + 1];
    const int64_t n_rel = r1 - r0;
    if (n_rel == 0) {
      if (row_metrics && lane < 4) row_metrics[u * 4 + lane] = nan("");   // not evaluated
      continue;
    }
    int hits = 0;
    double dcg = 0.0, idcg = 0.0;
    for (int r = lane; r < k; r += 32) {
      const int32_t it = topk_idx[u * k + r];
      const double disc = 1.0 / log2((double)(r + 2));
      if (r < n_rel) idcg += disc;
      if (it < 0) continue;
      int64_t lo = r0, hi = r1;   // first position with rel_item >= it
      while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (rel_item[mid] < it) lo = mid + 1; else hi = mid;
      }
      if (lo < r1 && rel_item[lo] == it) { ++hits; dcg += disc; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      hits += __shfl_xor_sync(0xffffffffu, hits, o);
      dcg += __shfl_xor_sync(0xffffffffu, dcg, o);
      idcg += __shfl_xor_sync(0xffffffffu, idcg, o);
    }
    const double hr = hits > 0 ? 1.0 : 0.0, prec = (double)hits / (double)k, rec = (double)hits / (double)n_rel,
                 ndcg = dcg / idcg;
    if (row_metrics && lane < 4) row_metrics[u * 4 + lane] = lane == 0 ? hr : lane == 1 ? prec : lane == 2 ? rec : ndcg;
    acc[0] += hr; acc[1] += prec; acc[2] += rec; acc[3] += ndcg; acc[4] += 1.0;
  }
  if (lane == 0) {
#pragma unroll
    for (int j = 0; j < 5; ++j) s_acc[w][j] = acc[j];
  }
  __syncthreads();
  if (threadIdx.x < 5) {
    double t = 0.0;
    for (int ww = 0; ww < RM_WARPS; ++ww) t += s_acc[ww][threadIdx.x];
    part[blockIdx.x * 5 + threadIdx.x] = t;
  }
}

__global__ void __launch_bounds__(256) ranking_metrics_finish_kernel(const double* __restrict__ part, int n_part,
                                                                     double* __restrict__ sums) {
  __shared__ double s_sum[5][256];
  for (int j = 0; j < 5; ++j) {
    double t = 0.0;
    for (int b = threadIdx.x; b < n_part; b += 256) t += part[b * 5 + j];
    s_sum[j][threadIdx.x] = t;
  }
  __syncthreads();
  if (threadIdx.x < 5) {
    double t = 0.0;
    for (int i = 0; i < 256; ++i) t += s_sum[threadIdx.x][i];
    sums[threadIdx.x] = t;
  }
}

static int ranking_metrics_blocks(int64_t n_rows) {
  const int64_t b = (n_rows + RM_WARPS - 1) / RM_WARPS;
  return (int)(b < 1 ? 1 : (b < RM_MAX_BLOCKS ? b : RM_MAX_BLOCKS));
}

// ================================ KTM design matrix (fm.py:61-93) ==========================================================
struct KtmArgs {
  const int32_t *user, *item;          // [n]
  const float *wins_col, *fails_col;   // [n] df["wins"], df["fails"] (item_wins / item_fails blocks)
  const int64_t* q_indptr; const int32_t* q_indices; const float* q_data;       // q-matrix CSR [item_num, n_skills]
  const int64_t* sw_indptr; const int32_t* sw_indices; const float* sw_data;    // skill_wins CSR [n, n_skills]
  const int64_t* sf_indptr; const int32_t* sf_indices; const float* sf_data;    // skill_fails CSR [n, n_skills]
  int64_t n;
  int32_t n_agents;
  int32_t agent[8];       // block kinds in output order: 0 users, 1 items, 2 skills, 3 attempts, 4 wins, 5 fails,
                          // 6 item_wins, 7 item_fails (ktm.AGENT_ORDER)
  int32_t col0[8];        // first column of each block
};

// entries of block `kind` in row r; emit(col, value) when filling.  attempts = skill_wins + skill_fails as scipy adds two
// CSR matrices: union of the patterns in column order, entries whose sum is zero dropped.
template <typename Emit>
__device__ __forceinline__ int ktm_block(const KtmArgs& a, int kind, int64_t r, Emit emit) {
  int cnt = 0;
  switch (kind) {
    case 0: emit(a.user[r], 1.0f); return 1;
    case 1: emit(a.item[r], 1.0f); return 1;
    case 6: emit(a.item[r], a.wins_col[r]); return 1;
    case 7: emit(a.item[r], a.fails_col[r]); return 1;
    case 2: {
      const int32_t it = a.item[r];
      for (int64_t p = a.q_indptr[it]; p < a.q_indptr[it + 1]; ++p, ++cnt) emit(a.q_indices[p], a.q_data[p]);
      return cnt;
    }
    case 4:
      for (int64_t p = a.sw_indptr[r]; p < a.sw_indptr[r + 1]; ++p, ++cnt) emit(a.sw_indices[p], a.sw_data[p]);
      return cnt;
    case 5:
      for (int64_t p = a.sf_indptr[r]; p < a.sf_indptr[r + 1]; ++p, ++cnt) emit(a.sf_indices[p], a.sf_data[p]);
      return cnt;
    case 3: {
      int64_t p = a.sw_indptr[r], q = a.sf_indptr[r];
      const int64_t pe = a.sw_indptr[r + 1], qe = a.sf_indptr[r + 1];
      while (p < pe || q < qe) {
        const int32_t cp = p < pe ? a.sw_indices[p] : 0x7fffffff, cq = q < qe ? a.sf_indices[q] : 0x7fffffff;
        const int32_t c = cp < cq ? cp : cq;
        float v = 0.0f;
        if (cp == c) v += a.sw_data[p++];
        if (cq == c) v += a.sf_data[q++];
        if (v != 0.0f) { emit(c, v); ++cnt; }
      }
      return cnt;
    }
  }
  return 0;
}

__global__ void __launch_bounds__(256) ktm_count_kernel(KtmArgs a, int32_t* __restrict__ row_nnz) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= a.n) return;
  int cnt = 0;
  for (int g = 0; g < a.n_agents; ++g) cnt += ktm_block(a, a.agent[g], r, [](int32_t, float) {});
  row_nnz[r] = cnt;
}

__global__ void __launch_bounds__(256) ktm_fill_kernel(KtmArgs a, const int64_t* __restrict__ indptr,
                                                       int32_t* __restrict__ indices, float* __restrict__ data) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= a.n) return;
  int64_t at = indptr[r];
  for (int g = 0; g < a.n_agents; ++g) {
    const int32_t c0 = a.col0[g];
    ktm_block(a, a.agent[g], r, [&](int32_t c, float v) { indices[at] = c0 + c; data[at] = v; ++at; });
  }
}

}  // namespace tfr

using namespace tfr;

extern "C" int64_t tfr_binary_metrics_workspace_bytes(int64_t n) {
  if (n < 0) return TFR_ERR_INVALID;
  const int64_t a4 = align_up(n * 4, 256), a8 = align_up((n + 1) * 8, 256);
  return 256 + 5 * a4 + 4 * a8 + 2 * align_up(scan_tiles(n) * 8, 256) + align_up(1024 * 3 * 8, 256) +
         tfr_dedup_workspace_bytes(n) + 256;
}

extern "C" int tfr_binary_metrics(const float* logits, const float* labels, int64_t n, void* workspace,
                                  int64_t workspace_bytes, double* out4, void* stream) {
  TFR_CHECK_ARG(n >= 0 && out4 && n < ((int64_t)1 << 31));
  cudaStream_t st = (cudaStream_t)stream;
  if (n == 0) {
    TFR_CUDA(cudaMemsetAsync(out4, 0, 4 * sizeof(double), st));
    return TFR_OK;
  }
  TFR_CHECK_ARG(logits && labels && workspace);
  if (workspace_bytes < tfr_binary_metrics_workspace_bytes(n)) {
    set_error("binary-metrics workspace too small");
    return TFR_ERR_WORKSPACE;
  }
  char* w = reinterpret_cast<char*>(align_up((int64_t)(uintptr_t)workspace, 256));
  const int64_t a4 = align_up(n * 4, 256), a8 = align_up((n + 1) * 8, 256);
  auto take = [&](int64_t bytes) { char* p = w; w += bytes; return p; };
  int32_t* keys = (int32_t*)take(a4);
  int32_t* skeys = (int32_t*)take(a4);
  int32_t* spos = (int32_t*)take(a4);
  int32_t* endf = (int32_t*)take(a4);
  int32_t* posf = (int32_t*)take(a4);
  int64_t* end_ex = (int64_t*)take(a8);
  int64_t* pos_ex = (int64_t*)take(a8);
  int64_t* run_pos = (int64_t*)take(a8);
  int64_t* run_cnt = (int64_t*)take(a8);
  int64_t* tiles_a = (int64_t*)take(align_up(scan_tiles(n) * 8, 256));
  int64_t* tiles_b = (int64_t*)take(align_up(scan_tiles(n) * 8, 256));
  double* part = (double*)take(align_up(1024 * 3 * 8, 256));
  void* sort_ws = w;
  const int n_part = (int)((n + 255) / 256 < 1024 ? (n + 255) / 256 : 1024);
  metrics_elementwise_kernel<<<n_part, 256, 0, st>>>(logits, labels, n, keys, part);
  TFR_LAUNCH_CHECK();
  // the step's stable radix sort, on all 32 key bits (four 8-bit passes)
  int rc = tfr_dedup_sort_pairs(keys, (int64_t)1 << 32, skeys, spos, nullptr, 1, nullptr, nullptr, n, sort_ws,
                                tfr_dedup_workspace_bytes(n), stream);
  if (rc) return rc;
  const unsigned gb = (unsigned)((n + 255) / 256);
  metrics_flags_kernel<<<gb, 256, 0, st>>>(skeys, spos, labels, n, endf, posf);
  TFR_LAUNCH_CHECK();
  if ((rc = exclusive_scan(endf, n, end_ex, tiles_a, st))) return rc;
  if ((rc = exclusive_scan(posf, n, pos_ex, tiles_b, st))) return rc;
  metrics_runs_kernel<<<gb, 256, 0, st>>>(endf, end_ex, pos_ex, posf, n, run_pos, run_cnt);
  TFR_LAUNCH_CHECK();
  metrics_finish_kernel<<<1, 1024, 0, st>>>(run_pos, run_cnt, end_ex, n, part, n_part, out4);
  TFR_LAUNCH_CHECK();
  return TFR_OK;
}

extern "C" int64_t tfr_ranking_metrics_workspace_bytes(int64_t n_rows, int32_t k) {
  if (n_rows < 0 || k <= 0) return TFR_ERR_INVALID;
  return 256 + align_up((int64_t)ranking_metrics_blocks(n_rows) * 5 * 8, 256);
}

extern "C" int tfr_ranking_metrics(const int32_t* topk_idx, int64_t n_rows, int32_t k, const int64_t* rel_indptr,
                                   const int32_t* rel_item, double* row_metrics, double* sums, void* workspace,
                                   int64_t workspace_bytes, void* stream) {
  TFR_CHECK_ARG(n_rows >= 0 && k > 0 && sums);
  cudaStream_t st = (cudaStream_t)stream;
  if (n_rows == 0) {
    TFR_CUDA(cudaMemsetAsync(sums, 0, 5 * sizeof(double), st));
    return TFR_OK;
  }
  TFR_CHECK_ARG(topk_idx && rel_indptr && rel_item && workspace);
  if (workspace_bytes < tfr_ranking_metrics_workspace_bytes(n_rows, k)) {
    set_error("ranking-metrics workspace too small");
    return TFR_ERR_WORKSPACE;
  }
  double* part = reinterpret_cast<double*>(align_up((int64_t)(uintptr_t)workspace, 256));
  const int nb = ranking_metrics_blocks(n_rows);
  ranking_metrics_rows_kernel<<<nb, 32 * RM_WARPS, 0, st>>>(topk_idx, n_rows, k, rel_indptr, rel_item, row_metrics, part);
  TFR_LAUNCH_CHECK();
  ranking_metrics_finish_kernel<<<1, 256, 0, st>>>(part, nb, sums);
  TFR_LAUNCH_CHECK();
  return TFR_OK;
}

static int ktm_args(KtmArgs* a, const int32_t* user, const int32_t* item, const float* wins_col, const float* fails_col,
                    const int64_t* q_indptr, const int32_t* q_indices, const float* q_data, const int64_t* sw_indptr,
                    const int32_t* sw_indices, const float* sw_data, const int64_t* sf_indptr, const int32_t* sf_indices,
                    const float* sf_data, int64_t n, const int32_t* agents, const int32_t* col0, int32_t n_agents) {
  TFR_CHECK_ARG(n >= 0 && n_agents >= 1 && n_agents <= 8 && agents && col0 && user && item);
  memset(a, 0, sizeof(*a));
  a->user = user; a->item = item; a->wins_col = wins_col; a->fails_col = fails_col;
  a->q_indptr = q_indptr; a->q_indices = q_indices; a->q_data = q_data;
  a->sw_indptr = sw_indptr; a->sw_indices = sw_indices; a->sw_data = sw_data;
  a->sf_indptr = sf_indptr; a->sf_indices = sf_indices; a->sf_data = sf_data;
  a->n = n; a->n_agents = n_agents;
  for (int g = 0; g < n_agents; ++g) {
    const int k = agents[g];
    TFR_CHECK_ARG(k >= 0 && k <= 7);
    TFR_CHECK_ARG(k != 2 || (q_indptr && q_indices && q_data));
    TFR_CHECK_ARG((k != 3 && k != 4) || (sw_indptr && sw_indices && sw_data));
    TFR_CHECK_ARG((k != 3 && k != 5) || (sf_indptr && sf_indices && sf_data));
    TFR_CHECK_ARG(k != 6 || wins_col);
    TFR_CHECK_ARG(k != 7 || fails_col);
    a->agent[g] = k; a->col0[g] = col0[g];
  }
  return TFR_OK;
}

extern "C" int64_t tfr_ktm_workspace_bytes(int64_t n) {
  if (n < 0) return TFR_ERR_INVALID;
  return 256 + align_up(n * 4, 256) + align_up(scan_tiles(n) * 8, 256) + 256;
}

extern "C" int tfr_ktm_csr_indptr(const int32_t* user, const int32_t* item, const float* wins_col, const float* fails_col,
                                  const int64_t* q_indptr, const int32_t* q_indices, const float* q_data,
                                  const int64_t* sw_indptr, const int32_t* sw_indices, const float* sw_data,
                                  const int64_t* sf_indptr, const int32_t* sf_indices, const float* sf_data, int64_t n,
                                  const int32_t* agents_host, const int32_t* col0_host, int32_t n_agents, int64_t* indptr,
                                  void* workspace, int64_t workspace_bytes, void* stream) {
  KtmArgs a;
  int rc = ktm_args(&a, user, item, wins_col, fails_col, q_indptr, q_indices, q_data, sw_indptr, sw_indices, sw_data,
                    sf_indptr, sf_indices, sf_data, n, agents_host, col0_host, n_agents);
  if (rc) return rc;
  TFR_CHECK_ARG(indptr && workspace && workspace_bytes >= tfr_ktm_workspace_bytes(n));
  cudaStream_t st = (cudaStream_t)stream;
  if (n == 0) {
    TFR_CUDA(cudaMemsetAsync(indptr, 0, sizeof(int64_t), st));
    return TFR_OK;
  }
  char* w = reinterpret_cast<char*>(align_up((int64_t)(uintptr_t)workspace, 256));
  int32_t* row_nnz = (int32_t*)w;
  int64_t* tiles = (int64_t*)(w + align_up(n * 4, 256));
  ktm_count_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(a, row_nnz);
  TFR_LAUNCH_CHECK();
  return exclusive_scan(row_nnz, n, indptr, tiles, st);
}

extern "C" int tfr_ktm_csr_fill(const int32_t* user, const int32_t* item, const float* wins_col, const float* fails_col,
                                const int64_t* q_indptr, const int32_t* q_indices, const float* q_data,
                                const int64_t* sw_indptr, const int32_t* sw_indices, const float* sw_data,
                                const int64_t* sf_indptr, const int32_t* sf_indices, const float* sf_data, int64_t n,
                                const int32_t* agents_host, const int32_t* col0_host, int32_t n_agents,
                                const int64_t* indptr, int32_t* indices, float* data, void* stream) {
  KtmArgs a;
  int rc = ktm_args(&a, user, item, wins_col, fails_col, q_indptr, q_indices, q_data, sw_indptr, sw_indices, sw_data,
                    sf_indptr, sf_indices, sf_data, n, agents_host, col0_host, n_agents);
  if (rc) return rc;
  if (n == 0) return TFR_OK;
  TFR_CHECK_ARG(indptr && indices && data);
  ktm_fill_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(a, indptr, indices, data);
  TFR_LAUNCH_CHECK();
  return TFR_OK;
}
