// Implicit-feedback alternating least squares on the device (iALS, Hu, Koren and Volinsky, ICDM 2008): tfr_gram_rows and
// tfr_ials_objective; tfr_ials_half_sweep is in als.cu, one template with the ALS half-sweep.  Interactions (u, i) carry a
// weight w_ui > 0 (duplicates merged, weights summed); p_ui = 1 on an interaction, 0 elsewhere; c_ui = 1 + alpha w_ui on an
// interaction, 1 elsewhere; s_ui = x_u . y_i.
//     L = sum_(u,i) c_ui (p_ui - s_ui)^2 + lambda (sum_u |x_u|^2 + sum_i |y_i|^2)   over all U x I pairs.
// With Y fixed, the row of user u solves (items are symmetric)
//     (Y^T Y + sum_(i in R(u)) alpha w_ui y_i y_i^T + lambda I) x_u = sum_(i in R(u)) (1 + alpha w_ui) y_i,
// and a row without interactions is 0.  Y^T Y is shared by every row: tfr_gram_rows computes it once per half-sweep, and each
// row's system costs only its own interactions (fold_in.cuh's code, FiImplicit form; the half-sweep reads G from global
// memory, L2-resident).
//
//  - gram_rows_kernel: one CTA per GRAM_ROWS consecutive rows of an fp32 table stages them FI_TILE at a time as doubles and
//    sums their packed lower float64 triangle (fi_tile_gram: each entry over the rows in order from 0.0) into the workspace;
//    gram_combine_kernel sums the partials in CTA order.  GRAM_ROWS and FI_THREADS are constants, so the bits are the same on
//    every GPU and every run (no floating-point atomics).
//  - the objective without the U x I matrix:
//        L = sum_ab (X^T X o Y^T Y)_ab + sum_(u,i) in R [c_ui (1 - s_ui)^2 - s_ui^2] + lambda (tr X^T X + tr Y^T Y),
//    the observed part by ials_objective_rows_kernel (a warp per user row, a lane per interaction, float64 from the fp32
//    tables, fixed-order block partials) and the rest from the two Grams by ials_objective_finish_kernel (one block, fixed
//    order: the same bits every run).
#include <math.h>

#include "fold_in.cuh"

namespace tfr {

constexpr int GRAM_ROWS = 1024;   // rows per CTA of gram_rows_kernel: a constant, so that the summation order is one order
constexpr int IOBJ_SUMS = 2;

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

// ---- the objective ----------------------------------------------------------------------------------------------------
// part[b] = (sum over the block's interactions of c (1 - s)^2 - s^2, number of interactions): a warp per user row, a lane
// per interaction in its order, s = x_u . y_i summed over d in order from 0.0, lanes and warps folded in a fixed order.
__global__ void __launch_bounds__(32 * OBJ_WARPS) ials_objective_rows_kernel(
    const float* __restrict__ X, const float* __restrict__ Y, int64_t n_users, int64_t n_items, int dim, int64_t xs,
    int64_t ys, double alpha, const int64_t* __restrict__ indptr, const int32_t* __restrict__ items,
    const float* __restrict__ weight, double* __restrict__ part) {
  __shared__ double s_acc[OBJ_WARPS][IOBJ_SUMS];
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  double obs = 0.0, n_obs = 0.0;
  const int64_t wid = (int64_t)blockIdx.x * OBJ_WARPS + w, n_w = (int64_t)gridDim.x * OBJ_WARPS;
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
    for (int ww = 0; ww < OBJ_WARPS; ++ww) t = __dadd_rn(t, s_acc[ww][threadIdx.x]);
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

extern "C" int64_t tfr_ials_objective_workspace_bytes(int64_t n_users) {
  if (n_users < 0) return TFR_ERR_INVALID;
  return 256 + align_up((int64_t)objective_blocks(n_users) * IOBJ_SUMS * 8, 256);
}

extern "C" int tfr_ials_objective(const float* user_feat, const float* item_feat, int64_t n_users, int64_t n_items,
                                  int32_t dim, int64_t user_stride, int64_t item_stride, const double* user_gram,
                                  const double* item_gram, float alpha, float reg, const int64_t* user_indptr,
                                  const int32_t* user_items, const float* user_weight, double* out5, void* workspace,
                                  int64_t workspace_bytes, void* stream) {
  TFR_CHECK_ARG(dim >= 1 && dim <= FI_MAX_DIM);
  TFR_CHECK_ARG(reg_ok(reg) && alpha_ok(alpha));
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
  const int nb = objective_blocks(n_users);
  ials_objective_rows_kernel<<<nb, 32 * OBJ_WARPS, 0, st>>>(user_feat, item_feat, n_users, n_items, dim, user_stride,
                                                             item_stride, (double)alpha, user_indptr, user_items,
                                                             user_weight, part);
  TFR_LAUNCH_CHECK();
  ials_objective_finish_kernel<<<1, 256, 0, st>>>(part, nb, user_gram, item_gram, dim, reg, out5);
  TFR_LAUNCH_CHECK();
  return TFR_OK;
}
