// K5 (forward): 2nd-order factorization machine on CSR rows.
// Replaces forward.py:21-22  fma(x) = mu + x.W + 0.5*(||xV||^2 - sum_f sum_i x_i^2 V_if^2)
// (forward.py writes x.dot(V**2), valid for the 0/1 features fm.py:61-93 builds; the canonical x_i^2
// form is computed, they coincide on one-hot / multi-hot rows -- SURVEY 8a row a19).
// One lane group per CSR row; a lane keeps s_f and q_f for its VEC-wide slice of the factors.
#include <string.h>

#include "common.cuh"

namespace tfr {

int adam_pass_and_finish(const tfr_adam_table* tabs, int nt, const tfr_svd_tables* t, tfr_opt_scalars* opt,
                         const tfr_svd_step_ws* ws, int n_partials, int tl_slot, void* stream);

template <int VEC, int L, int UNITS>
__global__ void __launch_bounds__(256) fm_forward_kernel(int64_t n_rows, const int64_t* __restrict__ indptr,
                                                         const int32_t* __restrict__ indices,
                                                         const float* __restrict__ data, const float* __restrict__ w0,
                                                         const float* __restrict__ W, const float* __restrict__ V,
                                                         int dim, float* __restrict__ yhat, float* __restrict__ sums) {
  const int lane = threadIdx.x & (L - 1);
  const int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) / L;
  if (r >= n_rows) return;
  const int n_units = dim / VEC;
  float s[UNITS][VEC], q[UNITS][VEC];
#pragma unroll
  for (int u = 0; u < UNITS; ++u)
#pragma unroll
    for (int c = 0; c < VEC; ++c) { s[u][c] = 0.0f; q[u][c] = 0.0f; }
  float lin = 0.0f;
  const int64_t p0 = indptr[r], p1 = indptr[r + 1];
  for (int64_t p = p0; p < p1; ++p) {
    const int32_t fi = indices[p];
    const float x = data[p];
    if (lane == 0) lin = add_rn(lin, mul_rn(ld_gather_f1(W + fi), x));
    const float* vr = V + (size_t)fi * dim;
#pragma unroll
    for (int u = 0; u < UNITS; ++u) {
      const int unit = lane + u * L;
      if (unit < n_units) {
        float vv[VEC];
        if constexpr (VEC == 4) {
          const float4 t4 = ld_gather_f4(reinterpret_cast<const float4*>(vr) + unit);
          vv[0] = t4.x; vv[1] = t4.y; vv[2] = t4.z; vv[3] = t4.w;
        } else {
          vv[0] = ld_gather_f1(vr + unit);
        }
#pragma unroll
        for (int c = 0; c < VEC; ++c) {
          const float t = mul_rn(vv[c], x);
          s[u][c] = add_rn(s[u][c], t);
          q[u][c] = add_rn(q[u][c], mul_rn(t, t));
        }
      }
    }
  }
  float inter = 0.0f;
#pragma unroll
  for (int u = 0; u < UNITS; ++u) {
    const int unit = lane + u * L;
    if (unit < n_units) {
#pragma unroll
      for (int c = 0; c < VEC; ++c) inter = add_rn(inter, sub_rn(mul_rn(s[u][c], s[u][c]), q[u][c]));
      if (sums) {
#pragma unroll
        for (int c = 0; c < VEC; ++c) sums[(size_t)r * dim + unit * VEC + c] = s[u][c];
      }
    }
  }
  // group butterfly (sub-warp groups may be partially populated at the grid's tail: use the group mask)
  const unsigned gmask = (L == 32) ? 0xffffffffu : (((1u << L) - 1u) << ((threadIdx.x & 31) & ~(L - 1)));
#pragma unroll
  for (int o = L / 2; o > 0; o >>= 1) inter = add_rn(inter, __shfl_xor_sync(gmask, inter, o, L));
  if (lane == 0) yhat[r] = add_rn(add_rn(*w0, lin), mul_rn(0.5f, inter));
}

// d cost / d yhat per CSR row + fixed-order per-CTA partial sums (for w0's dense gradient and the metric);
// also fills rowof[p] = CSR row of non-zero p (the segment sums reach a non-zero's error and row sums through it)
__global__ void __launch_bounds__(256) fm_err_kernel(const tfr_opt_scalars* __restrict__ opt, const float* __restrict__ yhat,
                                                     const float* __restrict__ y, const int64_t* __restrict__ indptr,
                                                     int64_t n, float* __restrict__ err, int32_t* __restrict__ rowof,
                                                     float* __restrict__ partials, double* __restrict__ se_partials) {
  const int flags = opt->flags;
  float acc = 0.0f;
  double se = 0.0;
  for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n; r += (int64_t)gridDim.x * blockDim.x) {
    const float e = dloss(flags, yhat[r], y[r]);
    err[r] = e;
    for (int64_t p = indptr[r]; p < indptr[r + 1]; ++p) rowof[p] = (int32_t)r;
    acc = add_rn(acc, e);
    const double dd = (double)y[r] - (double)yhat[r];
    se += dd * dd;
  }
  __shared__ float s_e[256];
  __shared__ double s_s[256];
  s_e[threadIdx.x] = acc;
  s_s[threadIdx.x] = se;
  __syncthreads();
  if (threadIdx.x == 0) {
    float a = 0.0f;
    double d = 0.0;
    for (int j = 0; j < 256; ++j) { a = add_rn(a, s_e[j]); d += s_s[j]; }
    partials[blockIdx.x] = a;
    se_partials[blockIdx.x] = d;
  }
}

}  // namespace tfr

using namespace tfr;

// Every (VEC, L, UNITS) fm_forward_kernel is instantiated for: (VEC, L) is row_geom's, UNITS = ceil(dim / VEC / L)
// rounded up to 1, 2, 4, 8 or 16 (surplus units are masked), so every dim of 1..512 has a member of this list
// (tests/test_fm_geometry.py mirrors the dispatch).  8 and 16 only occur for rows of 129..511 floats with dim % 4 != 0.
#define TFR_FM_CASES(X)                                                                     \
  X(4, 1, 1) X(4, 2, 1) X(4, 4, 1) X(4, 8, 1) X(4, 16, 1) X(4, 32, 1) X(4, 32, 2) X(4, 32, 4) \
  X(1, 1, 1) X(1, 2, 1) X(1, 4, 1) X(1, 8, 1) X(1, 16, 1) X(1, 32, 1) X(1, 32, 2) X(1, 32, 4) \
  X(1, 32, 8) X(1, 32, 16)

extern "C" int tfr_fm_forward(int64_t n_rows, const int64_t* indptr, const int32_t* indices, const float* data,
                              const float* w0, const float* W, const float* V, int32_t dim, float* yhat, float* sums,
                              void* stream) {
  TFR_CHECK_ARG(n_rows >= 0);
  if (dim <= 0 || dim > 512) {
    set_error("FM dim %d: the FM takes dims of 1 to 512", dim);
    return TFR_ERR_INVALID;
  }
  if (n_rows == 0) return TFR_OK;
  TFR_CHECK_ARG(indptr && indices && data && w0 && W && V && yhat);
  const RowGeom g = row_geom(dim);
  const int u = (dim / g.vec + g.lanes - 1) / g.lanes;
  const int units = u <= 1 ? 1 : u <= 2 ? 2 : u <= 4 ? 4 : u <= 8 ? 8 : 16;
  const int groups_per_cta = 256 / g.lanes;
  const unsigned grid = (unsigned)((n_rows + groups_per_cta - 1) / groups_per_cta);
  cudaStream_t st = (cudaStream_t)stream;
#define TFR_FM_CASE(VV, LL, UU)                                                                               \
  if (g.vec == VV && g.lanes == LL && units == UU) {                                                          \
    fm_forward_kernel<VV, LL, UU><<<grid, 256, 0, st>>>(n_rows, indptr, indices, data, w0, W, V, dim, yhat, sums); \
    TFR_LAUNCH_CHECK();                                                                                        \
    return TFR_OK;                                                                                             \
  }
  TFR_FM_CASES(TFR_FM_CASE)
#undef TFR_FM_CASE
  set_error("unsupported FM dim %d (vec %d lanes %d units %d)", dim, g.vec, g.lanes, units);
  return TFR_ERR_INVALID;
}

// ---- FM train step: the SVD step's structure on CSR rows (north_star: "the same SE/L2/Adam step") -------------------
// forward (sums kept) -> d cost/d yhat -> sort of the batch's feature ids -> ordered segment sums of the per-non-zero
// gradients -> ONE TF-Adam pass over V and W (or SGD slice) -> dense update of w0 + bookkeeping.
extern "C" int tfr_fm_train_step(const tfr_fm_tables* t, tfr_opt_scalars* opt, int64_t n_rows, const int64_t* indptr,
                                 const int32_t* indices, const float* data, int32_t* rowof, int64_t nnz,
                                 const float* y, float* yhat, float* sums, float* err, int32_t flags, void* workspace,
                                 int64_t workspace_bytes, void* stream) {
  TFR_CHECK_ARG(t && opt && n_rows > 0 && nnz > 0 && indptr && indices && data && rowof && y && yhat && sums && err);
  TFR_CHECK_ARG(t->n_feat > 0 && t->w0 && t->W && t->V && t->slot);
  if (t->dim <= 0 || t->dim > 512) {
    set_error("FM dim %d: the FM takes dims of 1 to 512", t->dim);
    return TFR_ERR_INVALID;
  }
  const bool sgd = flags & TFR_OPT_SGD;
  TFR_CHECK_ARG(sgd || (t->m_w0 && t->v_w0 && t->m_W && t->v_W && t->m_V && t->v_V));
  tfr_svd_step_ws ws;
  int rc = tfr_svd_step_carve(workspace, workspace_bytes, nnz, t->dim, &ws);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  if ((rc = tfr_fm_forward(n_rows, indptr, indices, data, t->w0, t->W, t->V, t->dim, yhat, sums, stream))) return rc;
  int64_t grid = (n_rows + 255) / 256;
  if (grid > TFR_MAX_PARTIALS) grid = TFR_MAX_PARTIALS;
  fm_err_kernel<<<(unsigned)grid, 256, 0, st>>>(opt, yhat, y, indptr, n_rows, err, rowof, ws.partials, ws.se_partials);
  TFR_LAUNCH_CHECK();
  if (!(flags & TFR_FM_PRESORTED) &&
      (rc = tfr_dedup_sort_pairs(indices, (int64_t)t->n_feat + 1, ws.su_ids, ws.su_pos, nullptr, 1, nullptr, nullptr,
                                 nnz, ws.sort_ws, ws.sort_ws_bytes, stream)))
    return rc;
  if ((rc = tfr_fm_segment_grads(t->V, t->W, t->slot, t->n_feat, t->dim, opt, sums, err, data, rowof, nnz, &ws, stream)))
    return rc;
  // w0 is to the FM what bias_global is to the SVD: dense gradient sum_r e_r, same end-of-step arithmetic
  tfr_svd_tables fin;
  memset(&fin, 0, sizeof(fin));
  fin.user_num = fin.item_num = t->n_feat;
  fin.dim = t->dim;
  fin.mu = t->w0; fin.m_mu = t->m_w0; fin.v_mu = t->v_w0;
  if (!sgd) {
    tfr_adam_table tabs[2] = {{t->V, t->m_V, t->v_V, t->n_feat, t->dim, t->slot, ws.gsum_uf, 0},
                              {t->W, t->m_W, t->v_W, t->n_feat, 1, t->slot, ws.gsum_ub, 0}};
    return adam_pass_and_finish(tabs, 2, &fin, opt, &ws, (int)grid, TFR_TL_STREAM_UF, stream);
  }
  tfr_slice_update side{t->V, nullptr, nullptr, t->W, nullptr, nullptr, ws.su_ids, ws.gsum_uf, ws.gsum_ub, 0};
  if ((rc = tfr_adam_slice_multi(&side, 1, t->dim, nnz, opt, 1, TFR_TL_TOUCHED_U, stream))) return rc;
  return tfr_svd_finish_step(&fin, opt, indices, indices, nnz, &ws, (int)grid, stream);
}
