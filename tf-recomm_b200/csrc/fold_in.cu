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
#include <math.h>

#include "common.cuh"

namespace tfr {

constexpr int FI_THREADS = 256;
constexpr int FI_TILE = 32;      // ratings staged per tile
constexpr int FI_MAX_DIM = 128;  // D = dim + 1 <= 129: the packed triangle (67 KB) + tile (34 KB) fit two CTAs per SM
constexpr int FI_SOLVE_REGS = (FI_MAX_DIM + 1 + 31) / 32;   // right-hand-side entries per lane of the solving warp

__host__ __device__ inline int fi_align16(int x) { return (x + 15) & ~15; }
__host__ __device__ inline int fi_tri(int i, int j) { return i * (i + 1) / 2 + j; }   // (i, j), j <= i, packed row-major

struct FiSmem {   // byte offsets of the dynamic shared memory of one CTA
  int tri, rhs, x, y, item, total;
};
__host__ __device__ inline FiSmem fi_smem(int dim) {
  const int D = dim + 1, Dp = (D + 3) / 4 * 4;
  FiSmem s;
  s.tri = 0;
  s.rhs = fi_align16(fi_tri(D, 0) * 8);
  s.x = fi_align16(s.rhs + D * 8);
  s.y = s.x + FI_TILE * Dp * 8;
  s.item = s.y + FI_TILE * 8;
  s.total = s.item + FI_TILE * 4;
  return s;
}

__global__ void __launch_bounds__(FI_THREADS, 2) fold_in_kernel(
    const float* __restrict__ V, const float* __restrict__ ib, const float* __restrict__ mu, int n_items, int dim,
    int64_t is, bool abs_item, bool reg_bias, float reg, const int64_t* __restrict__ indptr,
    const int32_t* __restrict__ items, const float* __restrict__ rates, float* __restrict__ out_feat,
    float* __restrict__ out_bias, int32_t* __restrict__ info) {
  extern __shared__ __align__(16) unsigned char fi_raw[];
  __shared__ int s_bad;
  const int D = dim + 1, Dp = (D + 3) / 4 * 4, Db = Dp / 4;
  const FiSmem L = fi_smem(dim);
  double* tri = reinterpret_cast<double*>(fi_raw + L.tri);
  double* rhs = reinterpret_cast<double*>(fi_raw + L.rhs);
  double* X = reinterpret_cast<double*>(fi_raw + L.x);   // [FI_TILE][Dp]
  double* Y = reinterpret_cast<double*>(fi_raw + L.y);   // [FI_TILE]
  int* s_item = reinterpret_cast<int*>(fi_raw + L.item);
  const int r = blockIdx.x, tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  const int64_t p0 = indptr[r], cnt = indptr[r + 1] - p0;
  float* of = out_feat + (size_t)r * dim;
  if (cnt <= 0) {   // no ratings: the model then scores the row by mu + b_i
    for (int c = tid; c < dim; c += FI_THREADS) of[c] = 0.0f;
    if (tid == 0) { out_bias[r] = 0.0f; info[r] = 0; }
    return;
  }
  const int n_tri = fi_tri(D, 0);
  for (int e = tid; e < n_tri; e += FI_THREADS) tri[e] = 0.0;
  for (int e = tid; e < D; e += FI_THREADS) rhs[e] = 0.0;
  if (tid == 0) s_bad = 0;
  const double m = (double)mu[0];
  const int n_blk = Db * (Db + 1) / 2;
  // ---- 1. Gram + RHS, FI_TILE ratings at a time, in CSR order ----
  for (int64_t t0 = 0; t0 < cnt; t0 += FI_TILE) {
    const int tn = (int)min((int64_t)FI_TILE, cnt - t0);
    __syncthreads();   // the previous tile has been consumed (and, first time round, the zeroing is done)
    if (tid < tn) {
      const int it = items[p0 + t0 + tid];
      const bool ok = it >= 0 && it < n_items;   // ids are device data: guarded here
      if (!ok) s_bad = 1;
      s_item[tid] = ok ? it : -1;
      Y[tid] = ok ? __dsub_rn(__dsub_rn((double)rates[p0 + t0 + tid], m), (double)ib[it]) : 0.0;
    }
    __syncthreads();
    for (int e = tid; e < tn * Dp; e += FI_THREADS) {   // coalesced: consecutive threads read consecutive dims of a row
      const int t = e / Dp, c = e % Dp;
      const int it = s_item[t];
      double x = 0.0;
      if (c < dim) {
        if (it >= 0) {
          const float v = V[(size_t)it * is + c];
          x = (double)(abs_item ? fabsf(v) : v);
        }
      } else if (c == dim) {
        x = 1.0;
      }
      X[t * Dp + c] = x;
    }
    __syncthreads();
    for (int b = tid; b < n_blk; b += FI_THREADS) {   // block (I, J), J <= I, of the lower triangle
      int I = (int)((sqrtf(8.0f * (float)b + 1.0f) - 1.0f) * 0.5f);
      while (fi_tri(I + 1, 0) <= b) ++I;
      while (fi_tri(I, 0) > b) --I;
      const int J = b - fi_tri(I, 0);
      double acc[4][4];
#pragma unroll
      for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          const int i = 4 * I + a, j = 4 * J + c;
          acc[a][c] = (i < D && j <= i) ? tri[fi_tri(i, j)] : 0.0;
        }
      for (int t = 0; t < tn; ++t) {
        const double2* xr = reinterpret_cast<const double2*>(X + t * Dp);
        const double2 a01 = xr[2 * I], a23 = xr[2 * I + 1], b01 = xr[2 * J], b23 = xr[2 * J + 1];
        const double av[4] = {a01.x, a01.y, a23.x, a23.y}, bv[4] = {b01.x, b01.y, b23.x, b23.y};
#pragma unroll
        for (int a = 0; a < 4; ++a)
#pragma unroll
          for (int c = 0; c < 4; ++c) acc[a][c] = __fma_rn(av[a], bv[c], acc[a][c]);
      }
#pragma unroll
      for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          const int i = 4 * I + a, j = 4 * J + c;
          if (i < D && j <= i) tri[fi_tri(i, j)] = acc[a][c];
        }
    }
    // the right-hand side on the last threads (those with the fewest Gram blocks)
    for (int i = FI_THREADS - 1 - tid; i < D; i += FI_THREADS) {
      double acc = rhs[i];
      for (int t = 0; t < tn; ++t) acc = __fma_rn(Y[t], X[t * Dp + i], acc);
      rhs[i] = acc;
    }
  }
  __syncthreads();
  int status = s_bad ? -1 : 0;
  if (status == 0) {
    // ---- 2. A + reg * n * D, Cholesky A = L L^T in place ----
    const double rn = __dmul_rn((double)reg, (double)cnt);
    for (int i = tid; i < (reg_bias ? D : dim); i += FI_THREADS) tri[fi_tri(i, i)] = __dadd_rn(tri[fi_tri(i, i)], rn);
    __syncthreads();
    for (int j = 0; j < D; ++j) {
      const double piv = tri[fi_tri(j, j)];   // (uniform: every thread reads the same finished value)
      if (!(piv > 0.0)) { status = j + 1; break; }
      const double ljj = sqrt(piv);
      for (int i = j + 1 + tid; i < D; i += FI_THREADS) tri[fi_tri(i, j)] = __ddiv_rn(tri[fi_tri(i, j)], ljj);
      __syncthreads();
      if (tid == 0) tri[fi_tri(j, j)] = ljj;   // nobody reads (j, j) in this step's trailing update
      for (int i = j + 1 + w; i < D; i += FI_THREADS / 32) {
        const double lij = tri[fi_tri(i, j)];
        double* row = tri + fi_tri(i, 0);
        for (int k = j + 1 + lane; k <= i; k += 32) row[k] = __fma_rn(-lij, tri[fi_tri(k, j)], row[k]);
      }
      __syncthreads();
    }
  }
  if (status != 0) {
    for (int c = tid; c < dim; c += FI_THREADS) of[c] = __int_as_float(0x7fc00000);
    if (tid == 0) { out_bias[r] = __int_as_float(0x7fc00000); info[r] = status; }
    return;
  }
  // ---- 3. L z = rhs, L^T theta = z: one warp, entry i = lane + 32 q in register v[q] of lane i % 32 ----
  if (w != 0) return;
  double v[FI_SOLVE_REGS];
#pragma unroll
  for (int q = 0; q < FI_SOLVE_REGS; ++q) {
    const int i = lane + 32 * q;
    v[q] = i < D ? rhs[i] : 0.0;
  }
  // j = 32 qj + jj with qj unrolled, so that the register holding entry j is named at compile time
#pragma unroll
  for (int qj = 0; qj < FI_SOLVE_REGS; ++qj) {
    for (int jj = 0; jj < 32 && 32 * qj + jj < D; ++jj) {
      const int j = 32 * qj + jj;
      const double zj = __ddiv_rn(__shfl_sync(0xffffffffu, v[qj], jj), tri[fi_tri(j, j)]);
#pragma unroll
      for (int q = qj; q < FI_SOLVE_REGS; ++q) {
        const int i = lane + 32 * q;
        if (i == j) v[q] = zj;
        else if (i > j && i < D) v[q] = __fma_rn(-tri[fi_tri(i, j)], zj, v[q]);
      }
    }
  }
#pragma unroll
  for (int qj = FI_SOLVE_REGS - 1; qj >= 0; --qj) {
    for (int jj = 31; jj >= 0; --jj) {
      const int j = 32 * qj + jj;
      if (j >= D) continue;
      const double tj = __ddiv_rn(__shfl_sync(0xffffffffu, v[qj], jj), tri[fi_tri(j, j)]);
      const double* row = tri + fi_tri(j, 0);
#pragma unroll
      for (int q = 0; q <= qj; ++q) {
        const int i = lane + 32 * q;
        if (i == j) v[q] = tj;
        else if (i < j) v[q] = __fma_rn(-row[i], tj, v[q]);
      }
    }
  }
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
