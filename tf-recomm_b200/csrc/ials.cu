// Implicit-feedback alternating least squares on the device (iALS, Hu, Koren and Volinsky, ICDM 2008): tfr_gram_rows,
// tfr_ials_half_sweep, tfr_ials_objective.  Interactions (u, i) carry a weight w_ui > 0 (duplicates merged, weights
// summed); p_ui = 1 on an interaction, 0 elsewhere; c_ui = 1 + alpha w_ui on an interaction, 1 elsewhere; s_ui = x_u . y_i.
//     L = sum_(u,i) c_ui (p_ui - s_ui)^2 + lambda (sum_u |x_u|^2 + sum_i |y_i|^2)   over all U x I pairs.
// With Y fixed, the row of user u solves (items are symmetric)
//     (Y^T Y + sum_(i in R(u)) alpha w_ui y_i y_i^T + lambda I) x_u = sum_(i in R(u)) (1 + alpha w_ui) y_i,
// and a row without interactions is 0.  Y^T Y is shared by every row: tfr_gram_rows computes it once per half-sweep, and each
// row's system costs only its own interactions (fold_in.cuh's code, FiImplicit form).
//
//  - gram_rows_kernel: one CTA per GRAM_ROWS consecutive rows of an fp32 table stages them FI_TILE at a time as doubles and
//    sums their packed lower float64 triangle (fi_tile_gram: each entry over the rows in order from 0.0) into the workspace;
//    gram_combine_kernel sums the partials in CTA order.  GRAM_ROWS and FI_THREADS are constants, so the bits are the same on
//    every GPU and every run (no floating-point atomics).
//  - a half-sweep on the ALS plan (als.cu): light rows (<= chunk interactions) one CTA each, the triangle starting from G
//    (read from global memory, L2-resident), then alpha w y y^T and (1 + alpha w) y in CSR order, lambda on the diagonal,
//    Cholesky, substitution.  Heavy rows: ials_chunk_gram_kernel writes each chunk's weighted partials (without G) to the
//    workspace; ials_heavy_solve_kernel starts from G, adds the chunks in chunk order, then lambda, factors and solves.  The
//    fp32 row goes into the row's [var|m|v] slot (m / v never touched) and 0 into its bias (when a bias table is given).
//    A pivot failure or a partner id out of range leaves the row as it was and counts in *n_failed.
//  - the objective without the U x I matrix:
//        L = sum_ab (X^T X o Y^T Y)_ab + sum_(u,i) in R [c_ui (1 - s_ui)^2 - s_ui^2] + lambda (tr X^T X + tr Y^T Y),
//    the observed part by ials_objective_rows_kernel (a warp per user row, a lane per interaction, float64 from the fp32
//    tables, fixed-order block partials) and the rest from the two Grams by ials_objective_finish_kernel (one block, fixed
//    order: the same bits every run).
#include <float.h>
#include <math.h>

#include "fold_in.cuh"

namespace tfr {

constexpr int GRAM_ROWS = 1024;   // rows per CTA of gram_rows_kernel: a constant, so that the summation order is one order
constexpr int IOBJ_WARPS = 8, IOBJ_MAX_BLOCKS = 1024, IOBJ_SUMS = 2;

static int64_t gram_ctas(int64_t n_rows) { return (n_rows + GRAM_ROWS - 1) / GRAM_ROWS; }

// Part 1: CTA b writes the packed triangle of rows [b GRAM_ROWS, (b + 1) GRAM_ROWS) of F (stride fs) to part[b].
__global__ void __launch_bounds__(FI_THREADS, 2) gram_rows_kernel(const float* __restrict__ F, int64_t n_rows, int dim,
                                                                   int64_t fs, double* __restrict__ part) {
  extern __shared__ __align__(16) unsigned char fi_raw[];
  const FiSmem L = fi_smem<FiPlain>(dim);
  double* tri = reinterpret_cast<double*>(fi_raw + L.tri);
  double* X = reinterpret_cast<double*>(fi_raw + L.x);   // [FI_TILE][Dp]
  const int D = dim, Dp = (D + 3) / 4 * 4, Db = Dp / 4, n_blk = Db * (Db + 1) / 2, n_tri = fi_tri(D, 0);
  const int tid = threadIdx.x;
  const int64_t r0 = (int64_t)blockIdx.x * GRAM_ROWS, cnt = min((int64_t)GRAM_ROWS, n_rows - r0);
  for (int e = tid; e < n_tri; e += FI_THREADS) tri[e] = 0.0;
  for (int64_t t0 = 0; t0 < cnt; t0 += FI_TILE) {
    const int tn = (int)min((int64_t)FI_TILE, cnt - t0);
    __syncthreads();   // the previous tile has been consumed (and, first time round, the zeroing is done)
    for (int e = tid; e < tn * Dp; e += FI_THREADS) {   // coalesced: consecutive threads read consecutive dims of a row
      const int t = e / Dp, c = e % Dp;
      X[t * Dp + c] = c < dim ? (double)F[(size_t)(r0 + t0 + t) * fs + c] : 0.0;
    }
    __syncthreads();
    fi_tile_gram<FiPlain>(tri, X, nullptr, D, Dp, n_blk, tid, tn);
  }
  __syncthreads();
  double* out = part + (int64_t)blockIdx.x * n_tri;
  for (int e = tid; e < n_tri; e += FI_THREADS) out[e] = tri[e];
}

// Part 2: G[e] = sum of the n_part partials' entry e, in CTA order from 0.0.
__global__ void __launch_bounds__(256) gram_combine_kernel(const double* __restrict__ part, int n_part, int n_tri,
                                                           double* __restrict__ G) {
  const int e = blockIdx.x * 256 + threadIdx.x;
  if (e >= n_tri) return;
  double acc = 0.0;
  for (int p = 0; p < n_part; ++p) acc = __dadd_rn(acc, part[(int64_t)p * n_tri + e]);
  G[e] = acc;
}

__device__ __forceinline__ void ials_write_row(float* of, float* ob, int dim, const double (&v)[FI_SOLVE_REGS]) {
  const int lane = threadIdx.x & 31;
#pragma unroll
  for (int q = 0; q < FI_SOLVE_REGS; ++q) {
    const int i = lane + 32 * q;
    if (i < dim) of[i] = __double2float_rn(v[q]);
  }
  if (lane == 0 && ob) *ob = 0.0f;
}

// Light rows: rows[blockIdx.x], the triangle started from G; output rows of stride os.
__global__ void __launch_bounds__(FI_THREADS, 2) ials_rows_kernel(
    const float* __restrict__ V, int n_fixed, int dim, int64_t fs, const double* __restrict__ G, double alpha, float reg,
    const int64_t* __restrict__ indptr, const int32_t* __restrict__ partner, const float* __restrict__ weight,
    const int32_t* __restrict__ rows, float* __restrict__ out_feat, int64_t os, float* __restrict__ out_bias,
    int32_t* __restrict__ n_failed) {
  extern __shared__ __align__(16) unsigned char fi_raw[];
  __shared__ int s_bad;
  const FiSmem L = fi_smem<FiImplicit>(dim);
  double* tri = reinterpret_cast<double*>(fi_raw + L.tri);
  const double* rhs = reinterpret_cast<const double*>(fi_raw + L.rhs);
  const int r = rows[blockIdx.x], tid = threadIdx.x;
  const int64_t p0 = indptr[r], cnt = indptr[r + 1] - p0;
  float* of = out_feat + (size_t)r * os;
  if (cnt <= 0) {
    for (int c = tid; c < dim; c += FI_THREADS) of[c] = 0.0f;
    if (tid == 0 && out_bias) out_bias[r] = 0.0f;
    return;
  }
  fi_gram<FiImplicit, true>(V, nullptr, 0.0, n_fixed, dim, fs, false, partner, weight, p0, cnt, fi_raw, &s_bad, alpha, G);
  const int status = s_bad ? -1 : fi_cholesky<FiImplicit>(tri, dim, false, reg, cnt);
  if (status != 0) {
    if (tid == 0) atomicAdd(n_failed, 1);
    return;
  }
  if (tid >= 32) return;
  double v[FI_SOLVE_REGS];
  fi_solve<FiImplicit>(tri, rhs, dim, v);
  ials_write_row(of, out_bias ? out_bias + r : nullptr, dim, v);
}

// Heavy rows, part 1: chunk c of heavy row h = chunk_heavy[c] is its interactions [chunk * (c - heavy_ptr[h]), + chunk); its
// weighted Gram (without G) and right-hand side go to part[c] = [packed triangle | rhs].  A partner id out of range makes
// entry (0, 0) NaN, so that the row's first pivot fails.
__global__ void __launch_bounds__(FI_THREADS, 2) ials_chunk_gram_kernel(
    const float* __restrict__ V, int n_fixed, int dim, int64_t fs, double alpha, const int64_t* __restrict__ indptr,
    const int32_t* __restrict__ partner, const float* __restrict__ weight, const int32_t* __restrict__ heavy_rows,
    const int64_t* __restrict__ heavy_ptr, const int32_t* __restrict__ chunk_heavy, int chunk, double* __restrict__ part) {
  extern __shared__ __align__(16) unsigned char fi_raw[];
  __shared__ int s_bad;
  const FiSmem L = fi_smem<FiImplicit>(dim);
  const double* tri = reinterpret_cast<const double*>(fi_raw + L.tri);
  const double* rhs = reinterpret_cast<const double*>(fi_raw + L.rhs);
  const int64_t c = blockIdx.x;
  const int h = chunk_heavy[c], r = heavy_rows[h];
  const int64_t p0 = indptr[r] + (c - heavy_ptr[h]) * (int64_t)chunk, cnt = min((int64_t)chunk, indptr[r + 1] - p0);
  fi_gram<FiImplicit, false>(V, nullptr, 0.0, n_fixed, dim, fs, false, partner, weight, p0, cnt, fi_raw, &s_bad, alpha);
  const int n_tri = fi_tri(dim, 0);
  double* out = part + c * (int64_t)(n_tri + dim);
  for (int e = threadIdx.x; e < n_tri + dim; e += FI_THREADS) out[e] = e < n_tri ? tri[e] : rhs[e - n_tri];
  if (threadIdx.x == 0 && s_bad) out[0] = __longlong_as_double(0x7ff8000000000000ll);
}

// Heavy rows, part 2: one CTA per heavy row: G, then its chunk partials in chunk order, then lambda; factor and solve.
__global__ void __launch_bounds__(FI_THREADS, 2) ials_heavy_solve_kernel(
    int dim, const double* __restrict__ G, float reg, const int64_t* __restrict__ indptr,
    const int32_t* __restrict__ heavy_rows, const int64_t* __restrict__ heavy_ptr, const double* __restrict__ part,
    float* __restrict__ out_feat, int64_t os, float* __restrict__ out_bias, int32_t* __restrict__ n_failed) {
  extern __shared__ __align__(16) unsigned char fi_raw[];
  const FiSmem L = fi_smem<FiImplicit>(dim);
  double* tri = reinterpret_cast<double*>(fi_raw + L.tri);
  double* rhs = reinterpret_cast<double*>(fi_raw + L.rhs);
  const int h = blockIdx.x, r = heavy_rows[h], tid = threadIdx.x;
  const int n_tri = fi_tri(dim, 0);
  const int64_t c0 = heavy_ptr[h], c1 = heavy_ptr[h + 1], cnt = indptr[r + 1] - indptr[r];
  for (int e = tid; e < n_tri + dim; e += FI_THREADS) {   // consecutive threads read consecutive entries of a partial
    double acc = e < n_tri ? G[e] : 0.0;
    for (int64_t c = c0; c < c1; ++c) acc = __dadd_rn(acc, part[c * (n_tri + dim) + e]);
    if (e < n_tri) tri[e] = acc;
    else rhs[e - n_tri] = acc;
  }
  __syncthreads();
  if (fi_cholesky<FiImplicit>(tri, dim, false, reg, cnt) != 0) {
    if (tid == 0) atomicAdd(n_failed, 1);
    return;
  }
  if (tid >= 32) return;
  double v[FI_SOLVE_REGS];
  fi_solve<FiImplicit>(tri, rhs, dim, v);
  ials_write_row(out_feat + (size_t)r * os, out_bias ? out_bias + r : nullptr, dim, v);
}

// ---- the objective ----------------------------------------------------------------------------------------------------
// part[b] = (sum over the block's interactions of c (1 - s)^2 - s^2, number of interactions): a warp per user row, a lane
// per interaction in its order, s = x_u . y_i summed over d in order from 0.0, lanes and warps folded in a fixed order.
__global__ void __launch_bounds__(32 * IOBJ_WARPS) ials_objective_rows_kernel(
    const float* __restrict__ X, const float* __restrict__ Y, int64_t n_users, int64_t n_items, int dim, int64_t xs,
    int64_t ys, double alpha, const int64_t* __restrict__ indptr, const int32_t* __restrict__ items,
    const float* __restrict__ weight, double* __restrict__ part) {
  __shared__ double s_acc[IOBJ_WARPS][IOBJ_SUMS];
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  double obs = 0.0, n_obs = 0.0;
  const int64_t wid = (int64_t)blockIdx.x * IOBJ_WARPS + w, n_w = (int64_t)gridDim.x * IOBJ_WARPS;
  for (int64_t u = wid; u < n_users; u += n_w) {
    const int64_t p0 = indptr[u], n = indptr[u + 1] - p0;
    const float* x = X + (size_t)u * xs;
    for (int64_t j = p0 + lane; j < p0 + n; j += 32) {
      const int it = items[j];
      const bool ok = it >= 0 && it < n_items;   // an id out of range is never read through: it poisons the sums
      const float* y = Y + (size_t)(ok ? it : 0) * ys;
      double s = 0.0;
      for (int d = 0; d < dim; ++d) s = __fma_rn((double)__ldg(x + d), (double)__ldg(y + d), s);
      const double c = __fma_rn(alpha, (double)weight[j], 1.0), e = __dsub_rn(1.0, s);
      double t = __fma_rn(c, __dmul_rn(e, e), -__dmul_rn(s, s));
      if (!ok) t = __longlong_as_double(0x7ff8000000000000ll);
      obs = __dadd_rn(obs, t);
    }
    if (lane == 0) n_obs = __dadd_rn(n_obs, (double)n);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    obs = __dadd_rn(obs, __shfl_xor_sync(0xffffffffu, obs, o));
    n_obs = __dadd_rn(n_obs, __shfl_xor_sync(0xffffffffu, n_obs, o));
  }
  if (lane == 0) {
    s_acc[w][0] = obs;
    s_acc[w][1] = n_obs;
  }
  __syncthreads();
  if (threadIdx.x < IOBJ_SUMS) {
    double t = 0.0;
    for (int ww = 0; ww < IOBJ_WARPS; ++ww) t = __dadd_rn(t, s_acc[ww][threadIdx.x]);
    part[blockIdx.x * IOBJ_SUMS + threadIdx.x] = t;
  }
}

// out5 = (L, observed part, all-pairs part sum_ab (Gx o Gy)_ab, lambda (tr Gx + tr Gy), interactions), Gx / Gy packed lower
// triangles of the symmetric Grams (an off-diagonal entry stands for two).
__global__ void __launch_bounds__(256) ials_objective_finish_kernel(const double* __restrict__ part, int n_part,
                                                                    const double* __restrict__ Gx,
                                                                    const double* __restrict__ Gy, int dim, float reg,
                                                                    double* __restrict__ out5) {
  __shared__ double s_sum[IOBJ_SUMS + 2][256];
  double t[IOBJ_SUMS + 2] = {0.0, 0.0, 0.0, 0.0};   // observed, n, all pairs, traces
  for (int b = threadIdx.x; b < n_part; b += 256) {
    t[0] = __dadd_rn(t[0], part[b * IOBJ_SUMS]);
    t[1] = __dadd_rn(t[1], part[b * IOBJ_SUMS + 1]);
  }
  for (int i = 0; i < dim; ++i) {
    const double* gx = Gx + fi_tri(i, 0);
    const double* gy = Gy + fi_tri(i, 0);
    for (int j = threadIdx.x; j <= i; j += 256) {
      const double p = __dmul_rn(gx[j], gy[j]);
      t[2] = j == i ? __dadd_rn(t[2], p) : __fma_rn(2.0, p, t[2]);
      if (j == i) t[3] = __dadd_rn(t[3], __dadd_rn(gx[j], gy[j]));
    }
  }
  for (int k = 0; k < IOBJ_SUMS + 2; ++k) s_sum[k][threadIdx.x] = t[k];
  __syncthreads();
  if (threadIdx.x != 0) return;
  double s[IOBJ_SUMS + 2];
  for (int k = 0; k < IOBJ_SUMS + 2; ++k) {
    double a = 0.0;
    for (int i = 0; i < 256; ++i) a = __dadd_rn(a, s_sum[k][i]);
    s[k] = a;
  }
  const double pen = __dmul_rn((double)reg, s[3]);
  out5[0] = __dadd_rn(__dadd_rn(s[2], s[0]), pen);
  out5[1] = s[0];
  out5[2] = s[2];
  out5[3] = pen;
  out5[4] = s[1];
}

static int ials_objective_blocks(int64_t n_rows) {
  const int64_t b = (n_rows + IOBJ_WARPS - 1) / IOBJ_WARPS;
  return (int)(b < 1 ? 1 : (b < IOBJ_MAX_BLOCKS ? b : IOBJ_MAX_BLOCKS));
}

static bool ials_reg_ok(float reg) { return reg > 0.0f && reg <= FLT_MAX; }        // refuses 0, negative, NaN and inf
static bool ials_alpha_ok(float alpha) { return alpha >= 0.0f && alpha <= FLT_MAX; }   // refuses negative, NaN and inf

}  // namespace tfr

using namespace tfr;

extern "C" int64_t tfr_gram_workspace_bytes(int64_t n_rows, int32_t dim) {
  if (n_rows < 0 || n_rows >= ((int64_t)1 << 31) || dim < 1 || dim > FI_MAX_DIM) return TFR_ERR_INVALID;
  return 256 + align_up(gram_ctas(n_rows) * (int64_t)fi_tri(dim, 0) * 8, 256);
}

extern "C" int tfr_gram_rows(const float* feat, int64_t n_rows, int32_t dim, int64_t stride, double* gram_out,
                             void* workspace, int64_t workspace_bytes, void* stream) {
  TFR_CHECK_ARG(dim >= 1 && dim <= FI_MAX_DIM);
  TFR_CHECK_ARG(n_rows >= 0 && n_rows < ((int64_t)1 << 31));
  if (stride == 0) stride = dim;
  TFR_CHECK_ARG(stride >= dim);
  TFR_CHECK_ARG(gram_out && workspace && (feat || n_rows == 0));
  if (workspace_bytes < tfr_gram_workspace_bytes(n_rows, dim)) {
    set_error("Gram workspace too small");
    return TFR_ERR_WORKSPACE;
  }
  cudaStream_t st = (cudaStream_t)stream;
  double* part = reinterpret_cast<double*>(align_up((int64_t)(uintptr_t)workspace, 256));
  const int n_part = (int)gram_ctas(n_rows), n_tri = fi_tri(dim, 0);
  if (n_part > 0) {
    const FiSmem s = fi_smem<FiPlain>(dim);
    TFR_CUDA(cudaFuncSetAttribute(gram_rows_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, s.total));
    gram_rows_kernel<<<n_part, FI_THREADS, s.total, st>>>(feat, n_rows, dim, stride, part);
    TFR_LAUNCH_CHECK();
  }
  gram_combine_kernel<<<(n_tri + 255) / 256, 256, 0, st>>>(part, n_part, n_tri, gram_out);
  TFR_LAUNCH_CHECK();
  return TFR_OK;
}

extern "C" int64_t tfr_ials_workspace_bytes(int64_t n_chunks, int32_t dim) {
  if (n_chunks < 0 || dim < 1 || dim > FI_MAX_DIM) return TFR_ERR_INVALID;
  const int64_t D = dim;
  return 256 + align_up(n_chunks * (D * (D + 1) / 2 + D) * 8, 256);
}

extern "C" int tfr_ials_half_sweep(const float* fixed_feat, int64_t n_fixed, int32_t dim, int64_t fixed_stride,
                                   const double* fixed_gram, float alpha, float reg, const int64_t* indptr,
                                   const int32_t* partner, const float* weight, const int32_t* light_rows,
                                   int64_t n_light, const int32_t* heavy_rows, const int64_t* heavy_ptr, int64_t n_heavy,
                                   const int32_t* chunk_heavy, int64_t n_chunks, int32_t chunk, float* out_feat,
                                   int64_t out_stride, float* out_bias, int32_t* n_failed, void* workspace,
                                   int64_t workspace_bytes, void* stream) {
  TFR_CHECK_ARG(dim >= 1 && dim <= FI_MAX_DIM);
  TFR_CHECK_ARG(ials_reg_ok(reg) && ials_alpha_ok(alpha));
  TFR_CHECK_ARG(n_fixed >= 0 && n_fixed < ((int64_t)1 << 31) && n_light >= 0 && n_light < ((int64_t)1 << 31));
  TFR_CHECK_ARG(n_heavy >= 0 && n_heavy < ((int64_t)1 << 31) && n_chunks >= 0 && n_chunks < ((int64_t)1 << 31));
  TFR_CHECK_ARG((n_heavy == 0) == (n_chunks == 0));
  if (fixed_stride == 0) fixed_stride = dim;
  if (out_stride == 0) out_stride = dim;
  TFR_CHECK_ARG(fixed_stride >= dim && out_stride >= dim);
  if (n_light == 0 && n_heavy == 0) return TFR_OK;
  TFR_CHECK_ARG(fixed_feat && fixed_gram && indptr && partner && weight && out_feat && n_failed);
  TFR_CHECK_ARG(n_light == 0 || light_rows);
  if (n_heavy > 0) {
    TFR_CHECK_ARG(heavy_rows && heavy_ptr && chunk_heavy && workspace && chunk >= 1);
    if (workspace_bytes < tfr_ials_workspace_bytes(n_chunks, dim)) {
      set_error("iALS workspace too small");
      return TFR_ERR_WORKSPACE;
    }
  }
  cudaStream_t st = (cudaStream_t)stream;
  const FiSmem s = fi_smem<FiImplicit>(dim);
  const double a = (double)alpha;
  if (n_heavy > 0) {
    double* part = reinterpret_cast<double*>(align_up((int64_t)(uintptr_t)workspace, 256));
    TFR_CUDA(cudaFuncSetAttribute(ials_chunk_gram_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, s.total));
    ials_chunk_gram_kernel<<<(unsigned)n_chunks, FI_THREADS, s.total, st>>>(
        fixed_feat, (int)n_fixed, dim, fixed_stride, a, indptr, partner, weight, heavy_rows, heavy_ptr, chunk_heavy, chunk,
        part);
    TFR_LAUNCH_CHECK();
    TFR_CUDA(cudaFuncSetAttribute(ials_heavy_solve_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, s.x));
    ials_heavy_solve_kernel<<<(unsigned)n_heavy, FI_THREADS, s.x, st>>>(dim, fixed_gram, reg, indptr, heavy_rows, heavy_ptr,
                                                                        part, out_feat, out_stride, out_bias, n_failed);
    TFR_LAUNCH_CHECK();
  }
  if (n_light > 0) {
    TFR_CUDA(cudaFuncSetAttribute(ials_rows_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, s.total));
    ials_rows_kernel<<<(unsigned)n_light, FI_THREADS, s.total, st>>>(fixed_feat, (int)n_fixed, dim, fixed_stride,
                                                                     fixed_gram, a, reg, indptr, partner, weight,
                                                                     light_rows, out_feat, out_stride, out_bias, n_failed);
    TFR_LAUNCH_CHECK();
  }
  return TFR_OK;
}

extern "C" int64_t tfr_ials_objective_workspace_bytes(int64_t n_users) {
  if (n_users < 0) return TFR_ERR_INVALID;
  return 256 + align_up((int64_t)ials_objective_blocks(n_users) * IOBJ_SUMS * 8, 256);
}

extern "C" int tfr_ials_objective(const float* user_feat, const float* item_feat, int64_t n_users, int64_t n_items,
                                  int32_t dim, int64_t user_stride, int64_t item_stride, const double* user_gram,
                                  const double* item_gram, float alpha, float reg, const int64_t* user_indptr,
                                  const int32_t* user_items, const float* user_weight, double* out5, void* workspace,
                                  int64_t workspace_bytes, void* stream) {
  TFR_CHECK_ARG(dim >= 1 && dim <= FI_MAX_DIM);
  TFR_CHECK_ARG(ials_reg_ok(reg) && ials_alpha_ok(alpha));
  TFR_CHECK_ARG(n_users >= 0 && n_users < ((int64_t)1 << 31) && n_items >= 0 && n_items < ((int64_t)1 << 31));
  if (user_stride == 0) user_stride = dim;
  if (item_stride == 0) item_stride = dim;
  TFR_CHECK_ARG(user_stride >= dim && item_stride >= dim);
  TFR_CHECK_ARG(user_feat && item_feat && user_gram && item_gram && user_indptr && user_items && user_weight && out5 &&
                workspace);
  if (workspace_bytes < tfr_ials_objective_workspace_bytes(n_users)) {
    set_error("iALS objective workspace too small");
    return TFR_ERR_WORKSPACE;
  }
  cudaStream_t st = (cudaStream_t)stream;
  double* part = reinterpret_cast<double*>(align_up((int64_t)(uintptr_t)workspace, 256));
  const int nb = ials_objective_blocks(n_users);
  ials_objective_rows_kernel<<<nb, 32 * IOBJ_WARPS, 0, st>>>(user_feat, item_feat, n_users, n_items, dim, user_stride,
                                                             item_stride, (double)alpha, user_indptr, user_items,
                                                             user_weight, part);
  TFR_LAUNCH_CHECK();
  ials_objective_finish_kernel<<<1, 256, 0, st>>>(part, nb, user_gram, item_gram, dim, reg, out5);
  TFR_LAUNCH_CHECK();
  return TFR_OK;
}
