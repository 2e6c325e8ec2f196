// The half-sweeps of alternating least squares on the device, explicit (ALS: tfr_als_half_sweep) and implicit feedback
// (iALS: tfr_ials_half_sweep, the rest of iALS in ials.cu), and the ALS objective (tfr_svd_objective).
//
// ALS minimises the training loss the Adam / SGD step minimises (ops.py:81-89,124-126, squared error), summed over every
// training occurrence (duplicates count):
//     L = sum_(u,i,r) [ 1/2 (r - mu - b_u - b_i - p_u.q_i)^2 + 1/2 reg (|p_u|^2 + |q_i|^2) (+ 1/2 reg (b_u^2 + b_i^2), REG_BIAS) ]
// With one side and mu fixed, L restricted to one row of the other side is the ridge regression fold-in solves
// (fold_in.cuh): a half-sweep solves every row of a side exactly, in float64, and rounds it to fp32.  A sweep is user rows,
// then item rows (reading the fp32 user rows just written), then mu <- mu + sum e / N (tfr_svd_objective): three exact block
// minimisations, each of which can only lower L in exact arithmetic.  iALS solves the confidence-weighted system of
// ials.cu's header against the Gram G of the fixed side.
//
// A half-sweep, for the rows of one side (CSR of the solved side: partner ids and ratings or weights, in the plan's row
// lists), is one set of kernels templated on the form of the system (FiRatings for ALS, FiImplicit for iALS):
//  - light rows (<= chunk entries): half_sweep_rows_kernel, one CTA per row, fold-in's code (Gram in CSR order, from 0.0 or
//    from G, Cholesky, substitution), the solution written straight into the row of the (possibly interleaved) output table;
//  - heavy rows (> chunk entries, e.g. the Zipf head of the item side): half_sweep_chunk_gram_kernel, one CTA per chunk of
//    `chunk` consecutive CSR entries, writes the chunk's packed float64 triangle and right-hand side to the workspace; then
//    half_sweep_heavy_solve_kernel, one CTA per heavy row, sums the row's chunk partials in chunk order (a fixed order that
//    no launch geometry changes) from 0.0 or from G, adds reg * n or lambda, factors and solves with the same device code.
//    No CTA walks more than `chunk` entries.
// A row without entries gets zeros.  A row whose pivot is not > 0 (unreachable with reg > 0) or that names a partner id out
// of range keeps its previous values and is counted in *n_failed: no NaN ever enters the model.  ALS writes the solved
// bias; iALS writes 0 into the bias when a bias table is given.
//
// The ALS objective: als_objective_rows_kernel, one warp per user row (its ratings, a lane per occurrence, e in float64 from
// the fp32 tables) and per item row (its regulariser terms), fixed-order block partials; als_objective_finish_kernel folds
// them in a fixed order (the scheme of ranking_metrics_finish_kernel, no floating-point atomics: the same bits every run)
// and, when asked, writes mu + sum e / N rounded to fp32.
#include <float.h>
#include <math.h>

#include "fold_in.cuh"

namespace tfr {

constexpr int ALS_MIN_CHUNK = FI_TILE, ALS_MAX_CHUNK = 1 << 20;
constexpr int OBJ_SUMS = 5;

// Lane i of the solving warp writes entries i + 32 q of the solution: the dim features to of, then the bias entry to *ob
// (F::bias), or 0 to *ob when ob is given (no bias column).
template <class F>
__device__ __forceinline__ void write_row(float* of, float* ob, int dim, const double (&v)[FI_SOLVE_REGS]) {
  const int lane = threadIdx.x & 31;
#pragma unroll
  for (int q = 0; q < FI_SOLVE_REGS; ++q) {
    const int i = lane + 32 * q;
    if (i < dim) of[i] = __double2float_rn(v[q]);
    else if (F::bias && i == dim) *ob = __double2float_rn(v[q]);
  }
  if (!F::bias && lane == 0 && ob) *ob = 0.0f;
}

// The kernels take the union of the two forms' parameters: fb, mu and reg_bias are FiRatings', G and alpha FiImplicit's;
// the other form leaves them alone.

// Light rows: fold_in_kernel's steps for the rows rows[blockIdx.x], the triangle started from G when F::weighted; output
// rows of stride os.
template <class F>
__global__ void __launch_bounds__(FI_THREADS, 2) half_sweep_rows_kernel(
    const float* __restrict__ V, const float* __restrict__ fb, const float* __restrict__ mu, const double* __restrict__ G,
    double alpha, int n_fixed, int dim, int64_t fs, bool reg_bias, float reg, const int64_t* __restrict__ indptr,
    const int32_t* __restrict__ partner, const float* __restrict__ vals, const int32_t* __restrict__ rows,
    float* __restrict__ out_feat, int64_t os, float* __restrict__ out_bias, int32_t* __restrict__ n_failed) {
  extern __shared__ __align__(16) unsigned char fi_raw[];
  __shared__ int s_bad;
  const FiSmem L = fi_smem<F>(dim);
  double* tri = reinterpret_cast<double*>(fi_raw + L.tri);
  const double* rhs = reinterpret_cast<const double*>(fi_raw + L.rhs);
  const int r = rows[blockIdx.x], tid = threadIdx.x;
  const int64_t p0 = indptr[r], cnt = indptr[r + 1] - p0;
  float* of = out_feat + (size_t)r * os;
  if (cnt <= 0) {
    for (int c = tid; c < dim; c += FI_THREADS) of[c] = 0.0f;
    if (tid == 0 && (F::bias || out_bias)) out_bias[r] = 0.0f;
    return;
  }
  fi_gram<F, F::weighted>(V, fb, F::weighted ? 0.0 : (double)mu[0], n_fixed, dim, fs, false, partner, vals, p0, cnt, fi_raw,
                          &s_bad, alpha, G);
  const int status = s_bad ? -1 : fi_cholesky<F>(tri, dim, reg_bias, reg, cnt);
  if (status != 0) {
    if (tid == 0) atomicAdd(n_failed, 1);
    return;
  }
  if (tid >= 32) return;
  double v[FI_SOLVE_REGS];
  fi_solve<F>(tri, rhs, dim, v);
  write_row<F>(of, (F::bias || out_bias) ? out_bias + r : nullptr, dim, v);
}

// Heavy rows, part 1: chunk c of heavy row h = chunk_heavy[c] is its entries [chunk * (c - heavy_ptr[h]), + chunk); its
// Gram (without G) and right-hand side go to part[c] = [packed triangle | rhs] (doubles).  A partner id out of range makes
// entry (0, 0) NaN, so that the row's first pivot fails.
template <class F>
__global__ void __launch_bounds__(FI_THREADS, 2) half_sweep_chunk_gram_kernel(
    const float* __restrict__ V, const float* __restrict__ fb, const float* __restrict__ mu, double alpha, int n_fixed,
    int dim, int64_t fs, const int64_t* __restrict__ indptr, const int32_t* __restrict__ partner,
    const float* __restrict__ vals, const int32_t* __restrict__ heavy_rows, const int64_t* __restrict__ heavy_ptr,
    const int32_t* __restrict__ chunk_heavy, int chunk, double* __restrict__ part) {
  extern __shared__ __align__(16) unsigned char fi_raw[];
  __shared__ int s_bad;
  const FiSmem L = fi_smem<F>(dim);
  const double* tri = reinterpret_cast<const double*>(fi_raw + L.tri);
  const double* rhs = reinterpret_cast<const double*>(fi_raw + L.rhs);
  const int64_t c = blockIdx.x;
  const int h = chunk_heavy[c], r = heavy_rows[h];
  const int64_t p0 = indptr[r] + (c - heavy_ptr[h]) * (int64_t)chunk, cnt = min((int64_t)chunk, indptr[r + 1] - p0);
  fi_gram<F, false>(V, fb, F::weighted ? 0.0 : (double)mu[0], n_fixed, dim, fs, false, partner, vals, p0, cnt, fi_raw,
                    &s_bad, alpha);
  const int D = dim + F::extra, n_tri = fi_tri(D, 0);
  double* out = part + c * (int64_t)(n_tri + D);
  for (int e = threadIdx.x; e < n_tri + D; e += FI_THREADS) out[e] = e < n_tri ? tri[e] : rhs[e - n_tri];
  if (threadIdx.x == 0 && s_bad) out[0] = __longlong_as_double(0x7ff8000000000000ll);
}

// Heavy rows, part 2: one CTA per heavy row sums its chunk partials in chunk order, from G when F::weighted, else from 0.0;
// then factors and solves.
template <class F>
__global__ void __launch_bounds__(FI_THREADS, 2) half_sweep_heavy_solve_kernel(
    int dim, const double* __restrict__ G, bool reg_bias, float reg, const int64_t* __restrict__ indptr,
    const int32_t* __restrict__ heavy_rows, const int64_t* __restrict__ heavy_ptr, const double* __restrict__ part,
    float* __restrict__ out_feat, int64_t os, float* __restrict__ out_bias, int32_t* __restrict__ n_failed) {
  extern __shared__ __align__(16) unsigned char fi_raw[];
  const FiSmem L = fi_smem<F>(dim);
  double* tri = reinterpret_cast<double*>(fi_raw + L.tri);
  double* rhs = reinterpret_cast<double*>(fi_raw + L.rhs);
  const int h = blockIdx.x, r = heavy_rows[h], tid = threadIdx.x;
  const int D = dim + F::extra, n_tri = fi_tri(D, 0);
  const int64_t c0 = heavy_ptr[h], c1 = heavy_ptr[h + 1], cnt = indptr[r + 1] - indptr[r];
  for (int e = tid; e < n_tri + D; e += FI_THREADS) {   // consecutive threads read consecutive entries of a partial
    double acc = (F::weighted && e < n_tri) ? G[e] : 0.0;
    for (int64_t c = c0; c < c1; ++c) acc = __dadd_rn(acc, part[c * (n_tri + D) + e]);
    if (e < n_tri) tri[e] = acc;
    else rhs[e - n_tri] = acc;
  }
  __syncthreads();
  if (fi_cholesky<F>(tri, dim, reg_bias, reg, cnt) != 0) {
    if (tid == 0) atomicAdd(n_failed, 1);
    return;
  }
  if (tid >= 32) return;
  double v[FI_SOLVE_REGS];
  fi_solve<F>(tri, rhs, dim, v);
  write_row<F>(out_feat + (size_t)r * os, (F::bias || out_bias) ? out_bias + r : nullptr, dim, v);
}

__device__ __forceinline__ double row_norm2(const float* x, int dim) {   // sum_d x[d]^2 in order from 0.0, float64
  double t = 0.0;
  for (int d = 0; d < dim; ++d) t = __fma_rn((double)x[d], (double)x[d], t);
  return t;
}

// ---- the objective ----------------------------------------------------------------------------------------------------
// Rows [0, n_users) are users: e = (((r - mu) - b_u) - b_i) - p_u.q~_i per occurrence, the dot summed over d in order from
// 0.0, all in float64 from the fp32 tables (q~ = |q| with ABS_ITEM); items only add their regulariser terms.  Per block:
// part[b] = (sum e, sum e^2, sum_rows n |x|^2, sum_rows n b^2, N), each lane's terms in its occurrence order, lanes and warps
// folded in a fixed order.
__global__ void __launch_bounds__(32 * OBJ_WARPS) als_objective_rows_kernel(
    const float* __restrict__ P, const float* __restrict__ pb, const float* __restrict__ Q, const float* __restrict__ qb,
    const float* __restrict__ mu, int64_t n_users, int64_t n_items, int dim, int64_t ps, int64_t qs, bool abs_item,
    const int64_t* __restrict__ u_indptr, const int32_t* __restrict__ u_items, const float* __restrict__ u_rates,
    const int64_t* __restrict__ i_indptr, double* __restrict__ part) {
  __shared__ double s_acc[OBJ_WARPS][OBJ_SUMS];
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const double m = (double)mu[0];
  double se = 0.0, se2 = 0.0, pen = 0.0, pen_b = 0.0, n_occ = 0.0;
  const int64_t wid = (int64_t)blockIdx.x * OBJ_WARPS + w, n_w = (int64_t)gridDim.x * OBJ_WARPS;
  for (int64_t u = wid; u < n_users; u += n_w) {
    const int64_t p0 = u_indptr[u], n = u_indptr[u + 1] - p0;
    const float* p = P + (size_t)u * ps;
    const double b = (double)pb[u];
    for (int64_t j = p0 + lane; j < p0 + n; j += 32) {
      const int it = u_items[j];
      const bool ok = it >= 0 && it < n_items;   // an id out of range is never read through: it poisons the sums
      const float* q = Q + (size_t)(ok ? it : 0) * qs;
      double dot = 0.0;
      for (int d = 0; d < dim; ++d) {
        const float qv = __ldg(q + d);
        dot = __fma_rn((double)__ldg(p + d), (double)(abs_item ? fabsf(qv) : qv), dot);
      }
      double e = __dsub_rn(__dsub_rn(__dsub_rn(__dsub_rn((double)u_rates[j], m), b), (double)qb[ok ? it : 0]), dot);
      if (!ok) e = __longlong_as_double(0x7ff8000000000000ll);
      se = __dadd_rn(se, e);
      se2 = __fma_rn(e, e, se2);
    }
    if (lane == 0 && n > 0) {
      pen = __fma_rn((double)n, row_norm2(p, dim), pen);
      pen_b = __fma_rn((double)n, __dmul_rn(b, b), pen_b);
      n_occ = __dadd_rn(n_occ, (double)n);
    }
  }
  for (int64_t i = wid; i < n_items; i += n_w) {
    const int64_t n = i_indptr[i + 1] - i_indptr[i];
    if (lane == 0 && n > 0) {
      const double b = (double)qb[i];
      pen = __fma_rn((double)n, row_norm2(Q + (size_t)i * qs, dim), pen);
      pen_b = __fma_rn((double)n, __dmul_rn(b, b), pen_b);
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    se = __dadd_rn(se, __shfl_xor_sync(0xffffffffu, se, o));
    se2 = __dadd_rn(se2, __shfl_xor_sync(0xffffffffu, se2, o));
    pen = __dadd_rn(pen, __shfl_xor_sync(0xffffffffu, pen, o));
    pen_b = __dadd_rn(pen_b, __shfl_xor_sync(0xffffffffu, pen_b, o));
    n_occ = __dadd_rn(n_occ, __shfl_xor_sync(0xffffffffu, n_occ, o));
  }
  if (lane == 0) {
    s_acc[w][0] = se; s_acc[w][1] = se2; s_acc[w][2] = pen; s_acc[w][3] = pen_b; s_acc[w][4] = n_occ;
  }
  __syncthreads();
  if (threadIdx.x < OBJ_SUMS) {
    double t = 0.0;
    for (int ww = 0; ww < OBJ_WARPS; ++ww) t = __dadd_rn(t, s_acc[ww][threadIdx.x]);
    part[blockIdx.x * OBJ_SUMS + threadIdx.x] = t;
  }
}

// out6 = (L, sum e^2, sum e, sum n |x|^2, sum n b^2, N); mu_out (optional) = fl32(mu + sum e / N) when N > 0.
__global__ void __launch_bounds__(256) als_objective_finish_kernel(const double* __restrict__ part, int n_part,
                                                                   const float* __restrict__ mu, float reg, bool reg_bias,
                                                                   double* __restrict__ out6, float* __restrict__ mu_out) {
  __shared__ double s_sum[OBJ_SUMS][256];
  for (int j = 0; j < OBJ_SUMS; ++j) {
    double t = 0.0;
    for (int b = threadIdx.x; b < n_part; b += 256) t = __dadd_rn(t, part[b * OBJ_SUMS + j]);
    s_sum[j][threadIdx.x] = t;
  }
  __syncthreads();
  if (threadIdx.x != 0) return;
  double s[OBJ_SUMS];
  for (int j = 0; j < OBJ_SUMS; ++j) {
    double t = 0.0;
    for (int i = 0; i < 256; ++i) t = __dadd_rn(t, s_sum[j][i]);
    s[j] = t;
  }
  const double rg = (double)reg, pen = reg_bias ? __dadd_rn(s[2], s[3]) : s[2];
  if (out6) {
    out6[0] = __fma_rn(0.5, s[1], __dmul_rn(__dmul_rn(0.5, rg), pen));
    out6[1] = s[1]; out6[2] = s[0]; out6[3] = s[2]; out6[4] = s[3]; out6[5] = s[4];
  }
  if (mu_out && s[4] > 0.0) mu_out[0] = __double2float_rn(__dadd_rn((double)mu[0], __ddiv_rn(s[0], s[4])));
}

// Bytes of workspace for n_chunks chunk partials of D = dim + F::extra rows each.
template <class F>
static int64_t half_sweep_workspace_bytes(int64_t n_chunks, int32_t dim) {
  if (n_chunks < 0 || dim < 1 || dim > FI_MAX_DIM) return TFR_ERR_INVALID;
  const int64_t D = dim + F::extra;
  return 256 + align_up(n_chunks * (D * (D + 1) / 2 + D) * 8, 256);
}

// The checks both forms share (every refusal before any CUDA call), then the heavy rows' two launches and the light rows'.
// vals are ratings (FiRatings) or weights (FiImplicit); fixed_bias, mu and out_bias are FiRatings', fixed_gram and alpha
// FiImplicit's (out_bias optional).
template <class F>
static int half_sweep(const float* fixed_feat, const float* fixed_bias, const float* mu, const double* fixed_gram,
                      double alpha, int64_t n_fixed, int32_t dim, int64_t fixed_stride, bool reg_bias, float reg,
                      const int64_t* indptr, const int32_t* partner, const float* vals, const int32_t* light_rows,
                      int64_t n_light, const int32_t* heavy_rows, const int64_t* heavy_ptr, int64_t n_heavy,
                      const int32_t* chunk_heavy, int64_t n_chunks, int32_t chunk, float* out_feat, int64_t out_stride,
                      float* out_bias, int32_t* n_failed, void* workspace, int64_t workspace_bytes, void* stream) {
  TFR_CHECK_ARG(dim >= 1 && dim <= FI_MAX_DIM);
  TFR_CHECK_ARG(reg_ok(reg));
  TFR_CHECK_ARG(n_fixed >= 0 && n_fixed < ((int64_t)1 << 31) && n_light >= 0 && n_light < ((int64_t)1 << 31));
  TFR_CHECK_ARG(n_heavy >= 0 && n_heavy < ((int64_t)1 << 31) && n_chunks >= 0 && n_chunks < ((int64_t)1 << 31));
  TFR_CHECK_ARG((n_heavy == 0) == (n_chunks == 0));
  if (fixed_stride == 0) fixed_stride = dim;
  if (out_stride == 0) out_stride = dim;
  TFR_CHECK_ARG(fixed_stride >= dim && out_stride >= dim);
  if (n_light == 0 && n_heavy == 0) return TFR_OK;
  TFR_CHECK_ARG(fixed_feat && indptr && partner && vals && out_feat && n_failed);
  TFR_CHECK_ARG(F::weighted ? fixed_gram != nullptr : (fixed_bias && mu && out_bias));
  TFR_CHECK_ARG(n_light == 0 || light_rows);
  if (n_heavy > 0) {
    TFR_CHECK_ARG(heavy_rows && heavy_ptr && chunk_heavy && workspace && chunk >= 1);
    if (workspace_bytes < half_sweep_workspace_bytes<F>(n_chunks, dim)) {
      set_error("half-sweep workspace too small");
      return TFR_ERR_WORKSPACE;
    }
  }
  cudaStream_t st = (cudaStream_t)stream;
  const FiSmem s = fi_smem<F>(dim);
  if (n_heavy > 0) {
    double* part = reinterpret_cast<double*>(align_up((int64_t)(uintptr_t)workspace, 256));
    TFR_CUDA(cudaFuncSetAttribute(half_sweep_chunk_gram_kernel<F>, cudaFuncAttributeMaxDynamicSharedMemorySize, s.total));
    half_sweep_chunk_gram_kernel<F><<<(unsigned)n_chunks, FI_THREADS, s.total, st>>>(
        fixed_feat, fixed_bias, mu, alpha, (int)n_fixed, dim, fixed_stride, indptr, partner, vals, heavy_rows, heavy_ptr,
        chunk_heavy, chunk, part);
    TFR_LAUNCH_CHECK();
    TFR_CUDA(cudaFuncSetAttribute(half_sweep_heavy_solve_kernel<F>, cudaFuncAttributeMaxDynamicSharedMemorySize, s.x));
    half_sweep_heavy_solve_kernel<F><<<(unsigned)n_heavy, FI_THREADS, s.x, st>>>(
        dim, fixed_gram, reg_bias, reg, indptr, heavy_rows, heavy_ptr, part, out_feat, out_stride, out_bias, n_failed);
    TFR_LAUNCH_CHECK();
  }
  if (n_light > 0) {
    TFR_CUDA(cudaFuncSetAttribute(half_sweep_rows_kernel<F>, cudaFuncAttributeMaxDynamicSharedMemorySize, s.total));
    half_sweep_rows_kernel<F><<<(unsigned)n_light, FI_THREADS, s.total, st>>>(
        fixed_feat, fixed_bias, mu, fixed_gram, alpha, (int)n_fixed, dim, fixed_stride, reg_bias, reg, indptr, partner,
        vals, light_rows, out_feat, out_stride, out_bias, n_failed);
    TFR_LAUNCH_CHECK();
  }
  return TFR_OK;
}

}  // namespace tfr

using namespace tfr;

extern "C" int32_t tfr_als_chunk(void) {
  int c = tune(TUNE_ALS_CHUNK);
  if (c < ALS_MIN_CHUNK) c = ALS_MIN_CHUNK;
  if (c > ALS_MAX_CHUNK) c = ALS_MAX_CHUNK;
  return (c + FI_TILE - 1) / FI_TILE * FI_TILE;   // whole staging tiles
}

extern "C" int64_t tfr_als_workspace_bytes(int64_t n_chunks, int32_t dim) {
  return half_sweep_workspace_bytes<FiRatings>(n_chunks, dim);
}

extern "C" int64_t tfr_ials_workspace_bytes(int64_t n_chunks, int32_t dim) {
  return half_sweep_workspace_bytes<FiImplicit>(n_chunks, dim);
}

extern "C" int tfr_als_half_sweep(const float* fixed_feat, const float* fixed_bias, const float* mu, int64_t n_fixed,
                                  int32_t dim, int64_t fixed_stride, int32_t flags, int32_t var_mask, float reg,
                                  const int64_t* indptr, const int32_t* partner, const float* rates,
                                  const int32_t* light_rows, int64_t n_light, const int32_t* heavy_rows,
                                  const int64_t* heavy_ptr, int64_t n_heavy, const int32_t* chunk_heavy, int64_t n_chunks,
                                  int32_t chunk, float* out_feat, int64_t out_stride, float* out_bias, int32_t* n_failed,
                                  void* workspace, int64_t workspace_bytes, void* stream) {
  TFR_CHECK_ARG(!(flags & (TFR_LOSS_SIGMOID_CE | TFR_ABS_ITEM)));   // least squares, and quadratic in q_i
  TFR_CHECK_ARG(var_mask == TFR_VAR_ALL);
  return half_sweep<FiRatings>(fixed_feat, fixed_bias, mu, nullptr, 0.0, n_fixed, dim, fixed_stride,
                               (flags & TFR_REG_BIAS) != 0, reg, indptr, partner, rates, light_rows, n_light, heavy_rows,
                               heavy_ptr, n_heavy, chunk_heavy, n_chunks, chunk, out_feat, out_stride, out_bias, n_failed,
                               workspace, workspace_bytes, stream);
}

extern "C" int tfr_ials_half_sweep(const float* fixed_feat, int64_t n_fixed, int32_t dim, int64_t fixed_stride,
                                   const double* fixed_gram, float alpha, float reg, const int64_t* indptr,
                                   const int32_t* partner, const float* weight, const int32_t* light_rows,
                                   int64_t n_light, const int32_t* heavy_rows, const int64_t* heavy_ptr, int64_t n_heavy,
                                   const int32_t* chunk_heavy, int64_t n_chunks, int32_t chunk, float* out_feat,
                                   int64_t out_stride, float* out_bias, int32_t* n_failed, void* workspace,
                                   int64_t workspace_bytes, void* stream) {
  TFR_CHECK_ARG(alpha_ok(alpha));
  return half_sweep<FiImplicit>(fixed_feat, nullptr, nullptr, fixed_gram, (double)alpha, n_fixed, dim, fixed_stride, false,
                                reg, indptr, partner, weight, light_rows, n_light, heavy_rows, heavy_ptr, n_heavy,
                                chunk_heavy, n_chunks, chunk, out_feat, out_stride, out_bias, n_failed, workspace,
                                workspace_bytes, stream);
}

extern "C" int64_t tfr_svd_objective_workspace_bytes(int64_t n_users, int64_t n_items) {
  if (n_users < 0 || n_items < 0) return TFR_ERR_INVALID;
  return 256 + align_up((int64_t)objective_blocks(n_users + n_items) * OBJ_SUMS * 8, 256);
}

extern "C" int tfr_svd_objective(const float* user_feat, const float* user_bias, const float* item_feat,
                                 const float* item_bias, const float* mu, int64_t n_users, int64_t n_items, int32_t dim,
                                 int64_t user_stride, int64_t item_stride, int32_t flags, float reg,
                                 const int64_t* user_indptr, const int32_t* user_items, const float* user_rates,
                                 const int64_t* item_indptr, double* out6, float* mu_out, void* workspace,
                                 int64_t workspace_bytes, void* stream) {
  TFR_CHECK_ARG(dim >= 1);
  TFR_CHECK_ARG(!(flags & TFR_LOSS_SIGMOID_CE));
  TFR_CHECK_ARG(reg >= 0.0f && reg <= FLT_MAX);
  TFR_CHECK_ARG(n_users >= 0 && n_users < ((int64_t)1 << 31) && n_items >= 0 && n_items < ((int64_t)1 << 31));
  if (user_stride == 0) user_stride = dim;
  if (item_stride == 0) item_stride = dim;
  TFR_CHECK_ARG(user_stride >= dim && item_stride >= dim);
  TFR_CHECK_ARG(out6 || mu_out);
  TFR_CHECK_ARG(user_feat && user_bias && item_feat && item_bias && mu && user_indptr && item_indptr && workspace);
  TFR_CHECK_ARG(user_items && user_rates);
  if (workspace_bytes < tfr_svd_objective_workspace_bytes(n_users, n_items)) {
    set_error("objective workspace too small");
    return TFR_ERR_WORKSPACE;
  }
  cudaStream_t st = (cudaStream_t)stream;
  double* part = reinterpret_cast<double*>(align_up((int64_t)(uintptr_t)workspace, 256));
  const int nb = objective_blocks(n_users + n_items);
  als_objective_rows_kernel<<<nb, 32 * OBJ_WARPS, 0, st>>>(user_feat, user_bias, item_feat, item_bias, mu, n_users,
                                                           n_items, dim, user_stride, item_stride,
                                                           (flags & TFR_ABS_ITEM) != 0, user_indptr, user_items,
                                                           user_rates, item_indptr, part);
  TFR_LAUNCH_CHECK();
  als_objective_finish_kernel<<<1, 256, 0, st>>>(part, nb, mu, reg, (flags & TFR_REG_BIAS) != 0, out6, mu_out);
  TFR_LAUNCH_CHECK();
  return TFR_OK;
}
