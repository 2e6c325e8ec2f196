// Device code shared by fold-in (fold_in.cu), the ALS and iALS half-sweeps (als.cu) and the iALS Gram (ials.cu): the float64
// normal equations of one row of the model with the other side fixed, built in shared memory, factored and solved by one
// CTA.  The form of the system is a compile-time parameter (FiForm).  Explicit ratings (FiRatings, fold-in and ALS):
//     (sum_j x_j x_j^T + reg * n * D) theta = sum_j (r_j - mu - b_{k_j}) x_j,   x_j = [v~_{k_j} ; 1],
//     D = diag(1, ..., 1, REG_BIAS ? 1 : 0),
// over the row's n rating occurrences, k_j the partner row (an item for a user row, a user for an item row).  Implicit
// feedback (FiImplicit, iALS, Hu et al. 2008), no bias column, over the row's interactions with weights w_j:
//     (G + sum_j alpha w_j y_j y_j^T + lambda I) x = sum_j (1 + alpha w_j) y_j,   y_j = v_{k_j},   G = V^T V,
// G added either as the triangle's starting value (FROM_G) or by the caller.
//  - fi_gram: Gram + right-hand side of a run of ratings, FI_TILE at a time in CSR order.  The ratings are staged in shared
//    memory as doubles (x_j, constant 1 appended, zero-padded to a multiple of 4), and every thread owns fixed 4 x 4 blocks of
//    the packed lower triangle (register blocking, accumulators in shared memory between tiles).  Each entry is summed in
//    CSR order from 0.0 by one thread: no atomics, so the result depends on the run's ratings only.
//  - fi_cholesky: reg * n (or lambda) added to the diagonal, then a right-looking Cholesky factorisation of the packed triangle in place
//    (a warp per trailing row).
//  - fi_solve: forward / back substitution by one warp with the right-hand side in registers.
#pragma once
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

// The form of a row's system:
//  - BIAS: x_j = [v_j ; 1], D = dim + 1 (the bias column of the explicit model), else x_j = v_j, D = dim;
//  - WEIGHTED: Gram terms g_j x_j x_j^T with g_j = alpha w_j and right-hand-side coefficients 1 + alpha w_j (w_j the
//    interaction's weight), else g_j = 1 and r_j - mu - b_{k_j} (r_j the rating);
//  - REG_N: reg * n on the diagonal (n the row's ratings; the bias entry only with reg_bias), else reg on every entry.
template <bool BIAS, bool WEIGHTED, bool REG_N>
struct FiForm {
  static constexpr bool bias = BIAS, weighted = WEIGHTED, reg_n = REG_N;
  static constexpr int extra = BIAS ? 1 : 0;   // D = dim + extra rows
};
using FiRatings = FiForm<true, false, true>;     // fold-in, ALS
using FiImplicit = FiForm<false, true, false>;   // iALS
using FiPlain = FiForm<false, false, false>;     // a bare Gram F^T F (gram_rows)

struct FiSmem {   // byte offsets of the dynamic shared memory of one CTA
  int tri, rhs, x, y, w, item, total;
};
template <class F = FiRatings>
__host__ __device__ inline FiSmem fi_smem(int dim) {
  const int D = dim + F::extra, Dp = (D + 3) / 4 * 4;
  FiSmem s;
  s.tri = 0;
  s.rhs = fi_align16(fi_tri(D, 0) * 8);
  s.x = fi_align16(s.rhs + D * 8);
  s.y = s.x + FI_TILE * Dp * 8;
  s.w = s.y + FI_TILE * 8;   // [FI_TILE] Gram weights, WEIGHTED only
  s.item = s.w + (F::weighted ? FI_TILE * 8 : 0);
  s.total = s.item + FI_TILE * 4;
  return s;
}

// tri += sum_t g_t X_t X_t^T over the tn staged rows X [FI_TILE][Dp] (g_t = W[t] when WEIGHTED, else 1), D rows, n_blk =
// Db (Db + 1) / 2 blocks, Db = Dp / 4: every thread owns fixed 4 x 4 blocks of the packed lower triangle and sums each of
// its entries over t in order.
template <class F>
__device__ __forceinline__ void fi_tile_gram(double* tri, const double* X, const double* W, int D, int Dp, int n_blk, int tid, int tn) {
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
      double av[4] = {a01.x, a01.y, a23.x, a23.y};
      const double bv[4] = {b01.x, b01.y, b23.x, b23.y};
      if constexpr (F::weighted) {
        const double g = W[t];
#pragma unroll
        for (int a = 0; a < 4; ++a) av[a] = __dmul_rn(g, av[a]);
      }
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
}

// tri / rhs := Gram and right-hand side of the run partner / vals [p0, p0 + cnt) against the fixed rows V (stride is,
// n_fixed rows).  FiRatings: vals are ratings, target r - m - fb[k].  FiImplicit: vals are weights w, Gram weight alpha w,
// right-hand-side coefficient 1 + alpha w, and the triangle starts from G (packed, D rows) with FROM_G, else from 0.0
// (fb and m are then unused).  *s_bad := 1 if a partner id is outside [0, n_fixed) (such an entry is never read through).
// Every thread of the CTA calls it; it ends with a barrier.
template <class F = FiRatings, bool FROM_G = false>
__device__ __forceinline__ void fi_gram(const float* __restrict__ V, const float* __restrict__ fb, double m, int n_fixed,
                                        int dim, int64_t is, bool abs_item, const int32_t* __restrict__ partner,
                                        const float* __restrict__ vals, int64_t p0, int64_t cnt, unsigned char* raw,
                                        int* s_bad, double alpha = 0.0, const double* __restrict__ G = nullptr) {
  const int D = dim + F::extra, Dp = (D + 3) / 4 * 4, Db = Dp / 4;
  const FiSmem L = fi_smem<F>(dim);
  double* tri = reinterpret_cast<double*>(raw + L.tri);
  double* rhs = reinterpret_cast<double*>(raw + L.rhs);
  double* X = reinterpret_cast<double*>(raw + L.x);   // [FI_TILE][Dp]
  double* Y = reinterpret_cast<double*>(raw + L.y);   // [FI_TILE]
  double* W = reinterpret_cast<double*>(raw + L.w);   // [FI_TILE], WEIGHTED only
  int* s_item = reinterpret_cast<int*>(raw + L.item);
  const int tid = threadIdx.x;
  const int n_tri = fi_tri(D, 0);
  for (int e = tid; e < n_tri; e += FI_THREADS) tri[e] = FROM_G ? G[e] : 0.0;
  for (int e = tid; e < D; e += FI_THREADS) rhs[e] = 0.0;
  if (tid == 0) *s_bad = 0;
  const int n_blk = Db * (Db + 1) / 2;
  for (int64_t t0 = 0; t0 < cnt; t0 += FI_TILE) {
    const int tn = (int)min((int64_t)FI_TILE, cnt - t0);
    __syncthreads();   // the previous tile has been consumed (and, first time round, the zeroing is done)
    if (tid < tn) {
      const int it = partner[p0 + t0 + tid];
      const bool ok = it >= 0 && it < n_fixed;   // ids are device data: guarded here
      if (!ok) *s_bad = 1;
      s_item[tid] = ok ? it : -1;
      if constexpr (F::weighted) {
        const double g = ok ? __dmul_rn(alpha, (double)vals[p0 + t0 + tid]) : 0.0;
        W[tid] = g;
        Y[tid] = ok ? __dadd_rn(1.0, g) : 0.0;
      } else {
        Y[tid] = ok ? __dsub_rn(__dsub_rn((double)vals[p0 + t0 + tid], m), (double)fb[it]) : 0.0;
      }
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
      } else if (F::bias && c == dim) {
        x = 1.0;
      }
      X[t * Dp + c] = x;
    }
    __syncthreads();
    fi_tile_gram<F>(tri, X, W, D, Dp, n_blk, tid, tn);
    // the right-hand side on the last threads (those with the fewest Gram blocks)
    for (int i = FI_THREADS - 1 - tid; i < D; i += FI_THREADS) {
      double acc = rhs[i];
      for (int t = 0; t < tn; ++t) acc = __fma_rn(Y[t], X[t * Dp + i], acc);
      rhs[i] = acc;
    }
  }
  __syncthreads();
}

// A + reg * n * D (REG_N) or A + reg I, then A = L L^T in place (the packed triangle tri, dim + F::extra rows).  -> 0, or j + 1
// if pivot j was not > 0 (NaN included); the same value in every thread.  Every thread of the CTA calls it.
template <class F = FiRatings>
__device__ __forceinline__ int fi_cholesky(double* tri, int dim, bool reg_bias, float reg, int64_t cnt) {
  const int D = dim + F::extra, tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  const double rn = F::reg_n ? __dmul_rn((double)reg, (double)cnt) : (double)reg;
  const int n_diag = F::reg_n ? (reg_bias ? D : dim) : D;
  for (int i = tid; i < n_diag; i += FI_THREADS) tri[fi_tri(i, i)] = __dadd_rn(tri[fi_tri(i, i)], rn);
  __syncthreads();
  for (int j = 0; j < D; ++j) {
    const double piv = tri[fi_tri(j, j)];   // (uniform: every thread reads the same finished value)
    if (!(piv > 0.0)) return j + 1;
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
  return 0;
}

// L z = rhs, L^T theta = z by one warp (dim + F::extra rows): entry i = lane + 32 q of theta ends in v[q] of lane i % 32.
template <class F = FiRatings>
__device__ __forceinline__ void fi_solve(const double* tri, const double* rhs, int dim, double (&v)[FI_SOLVE_REGS]) {
  const int D = dim + F::extra, lane = threadIdx.x & 31;
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
}

// ---- host helpers of the ALS and iALS entry points (als.cu, ials.cu) --------------------------------------------------
constexpr int OBJ_WARPS = 8, OBJ_MAX_BLOCKS = 1024;   // the objectives' row kernels: warps per block, blocks at most

inline int objective_blocks(int64_t n_rows) {
  const int64_t b = (n_rows + OBJ_WARPS - 1) / OBJ_WARPS;
  return (int)(b < 1 ? 1 : (b < OBJ_MAX_BLOCKS ? b : OBJ_MAX_BLOCKS));
}

inline bool reg_ok(float reg) { return reg > 0.0f && reg <= FLT_MAX; }          // refuses 0, negative, NaN and infinite
inline bool alpha_ok(float alpha) { return alpha >= 0.0f && alpha <= FLT_MAX; }   // refuses negative, NaN and infinite

}  // namespace tfr
