// Fold-in of new users into a trained model (tfr_fold_in_users): with the item table, item biases and mu fixed, the
// training loss restricted to one user (ops.py:81-89,124-126, squared error) is a ridge regression in theta = [p_u ; b_u]
// whose minimiser solves the (dim+1) x (dim+1) SPD system
//     (sum_j x_j x_j^T + reg * n * D) theta = sum_j (r_j - mu - b_{i_j}) x_j,   x_j = [v~_{i_j} ; 1],
//     D = diag(1, ..., 1, REG_BIAS ? 1 : 0),   v~ = |v| with TFR_ABS_ITEM, else v,
// over the user's n rating occurrences (duplicates count, as in training).
//
// One kernel, one CTA per fold-in row, float64 on CUDA cores throughout:
//  1. Gram + RHS: the row's ratings are staged FI_TILE at a time in shared memory as doubles (x_j, constant 1 appended,
//     zero-padded to a multiple of 4), and every thread owns fixed 4 x 4 blocks of the packed lower triangle (register
//     blocking, accumulators in shared memory between tiles).  Each entry is summed in CSR order from 0.0 by one thread:
//     no atomics, so a row's result depends on its own ratings only (same bits whatever the batch, its order or size).
//  2. reg * n is added to the diagonal, then a right-looking Cholesky factorisation of the packed triangle in shared
//     memory (a warp per trailing row), and forward / back substitution by one warp with the right-hand side in registers.
//  3. p_u, b_u are written rounded to fp32 (the tables' precision); info[r] = 0 ok, j + 1 if pivot j was not > 0 (only
//     reachable with reg = 0), -1 if an item id is outside [0, n_items) (never read through); both give a NaN row.  A row
//     without ratings gets p = 0, b = 0, info 0.
#include <float.h>

#include "fold_in.cuh"

namespace tfr {

// Steps 1-3 with the shared device code of fold_in.cuh (also used by the ALS half-sweeps, als.cu).
__global__ void __launch_bounds__(FI_THREADS, 2) fold_in_kernel(
    const float* __restrict__ V, const float* __restrict__ ib, const float* __restrict__ mu, int n_items, int dim,
    int64_t is, bool abs_item, bool reg_bias, float reg, const int64_t* __restrict__ indptr,
    const int32_t* __restrict__ items, const float* __restrict__ rates, float* __restrict__ out_feat,
    float* __restrict__ out_bias, int32_t* __restrict__ info) {
  extern __shared__ __align__(16) unsigned char fi_raw[];
  __shared__ int s_bad;
  const FiSmem L = fi_smem(dim);
  double* tri = reinterpret_cast<double*>(fi_raw + L.tri);
  const double* rhs = reinterpret_cast<const double*>(fi_raw + L.rhs);
  const int r = blockIdx.x, tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  const int64_t p0 = indptr[r], cnt = indptr[r + 1] - p0;
  float* of = out_feat + (size_t)r * dim;
  if (cnt <= 0) {   // no ratings: the model then scores the row by mu + b_i
    for (int c = tid; c < dim; c += FI_THREADS) of[c] = 0.0f;
    if (tid == 0) { out_bias[r] = 0.0f; info[r] = 0; }
    return;
  }
  // ---- 1. Gram + RHS, FI_TILE ratings at a time, in CSR order ----
  fi_gram(V, ib, (double)mu[0], n_items, dim, is, abs_item, items, rates, p0, cnt, fi_raw, &s_bad);
  int status = s_bad ? -1 : 0;
  // ---- 2. A + reg * n * D, Cholesky A = L L^T in place ----
  if (status == 0) status = fi_cholesky(tri, dim, reg_bias, reg, cnt);
  if (status != 0) {
    for (int c = tid; c < dim; c += FI_THREADS) of[c] = __int_as_float(0x7fc00000);
    if (tid == 0) { out_bias[r] = __int_as_float(0x7fc00000); info[r] = status; }
    return;
  }
  // ---- 3. L z = rhs, L^T theta = z: one warp ----
  if (w != 0) return;
  double v[FI_SOLVE_REGS];
  fi_solve(tri, rhs, dim, v);
#pragma unroll
  for (int q = 0; q < FI_SOLVE_REGS; ++q) {
    const int i = lane + 32 * q;
    if (i < dim) of[i] = __double2float_rn(v[q]);
    else if (i == dim) { out_bias[r] = __double2float_rn(v[q]); info[r] = 0; }
  }
}

}  // namespace tfr

using namespace tfr;

extern "C" int tfr_fold_in_users(const float* item_feat, const float* item_bias, const float* mu, int64_t n_items,
                                 int32_t dim, int64_t item_stride, int32_t flags, float reg, const int64_t* indptr,
                                 const int32_t* items, const float* rates, int64_t n, float* out_feat, float* out_bias,
                                 int32_t* info, void* stream) {
  TFR_CHECK_ARG(dim >= 1 && dim <= FI_MAX_DIM);
  TFR_CHECK_ARG(!(flags & TFR_LOSS_SIGMOID_CE));
  TFR_CHECK_ARG(reg >= 0.0f && reg <= FLT_MAX);   // refuses negative, NaN and infinite values
  TFR_CHECK_ARG(n >= 0 && n < ((int64_t)1 << 31) && n_items >= 0 && n_items < ((int64_t)1 << 31));
  if (item_stride == 0) item_stride = dim;
  TFR_CHECK_ARG(item_stride >= dim);
  if (n == 0) return TFR_OK;
  TFR_CHECK_ARG(item_feat && item_bias && mu && indptr && items && rates && out_feat && out_bias && info);
  const FiSmem s = fi_smem(dim);
  TFR_CUDA(cudaFuncSetAttribute(fold_in_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, s.total));
  fold_in_kernel<<<(unsigned)n, FI_THREADS, s.total, (cudaStream_t)stream>>>(
      item_feat, item_bias, mu, (int)n_items, dim, item_stride, (flags & TFR_ABS_ITEM) != 0, (flags & TFR_REG_BIAS) != 0,
      reg, indptr, items, rates, out_feat, out_bias, info);
  TFR_LAUNCH_CHECK();
  return TFR_OK;
}
