/*
 * oracle/tfr_oracle.c -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.
 *
 * CPU restatement (plain C, explicit fp32, one rounding per TensorFlow op) of the
 * TF-recomm matrix-factorization train step.  Only tests/, __graft_entry__.smoke()
 * and bench.py's cpu_baseline / --impl reference legs may load this library; the
 * product path (tf-recomm_b200/) never does and fails loudly without its CUDA library.
 *
 * PARITY UNPINNED for the train step: the arithmetic of this path lives in TensorFlow 1.x
 * (requirements.txt:3, un-pinned, absent from /root/reference and not installable here) and
 * the reference holds no golden vectors / known-answer tests for it (SURVEY.md section 4).
 * What pins this file instead: (i) a numpy mirror written independently (oracle/np_oracle.py),
 * (ii) torch-CPU autograd of the same loss for the gradients, (iii) a dense-Adam-with-zero-
 * gradient formulation for the sparse Adam, all in tests/test_oracle_*.py.  The batch
 * composition (dataio iterators) and the KTM feature encoder ARE pinned by fixtures
 * generated from the real reference code (tests/golden/).
 *
 * Every function cites the reference lines (into /root/reference) it restates; "TF:" cites
 * TensorFlow 1.x source by file name (SURVEY.md Appendix A) because TF is not in the tree.
 *
 * Build: make -C oracle   (gcc -O2 -fopenmp -ffp-contract=off; contraction is disabled so
 * that "m*beta1" and "+ g*(1-beta1)" stay two roundings, as they are two TF kernels).
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#define ORC_API __attribute__((visibility("default")))

/* ---- model variants ----------------------------------------------------------------- */
/* flags for orc_svd_* : README mode = 0 (README.md:31-39, doc/graph_svd.png);           */
/* fork-as-written = ORC_ABS_ITEM|ORC_LOSS_SIGMOID_CE|ORC_REG_BIAS|ORC_OPT_SGD.           */
enum {
  ORC_ABS_ITEM = 1,        /* ops.py:44   tf.abs(feat_items) inside the dot            */
  ORC_LOSS_SIGMOID_CE = 2, /* ops.py:125  sigmoid_cross_entropy_with_logits, summed    */
  ORC_REG_BIAS = 4,        /* ops.py:85-89 l2_loss on the gathered biases too          */
  ORC_OPT_SGD = 8          /* ops.py:145  GradientDescentOptimizer instead of Adam     */
};
/* var_list bits (ops.py:118,147-149; adaptive_test.py:28 trains user side only) */
enum { ORC_VAR_MU = 1, ORC_VAR_UB = 2, ORC_VAR_UF = 4, ORC_VAR_IB = 8, ORC_VAR_IF = 16, ORC_VAR_ALL = 31 };

typedef struct {
  int32_t user_num, item_num, dim, flags;
  float *mu;          /* bias_global   []        ops.py:8  */
  float *user_bias;   /* user_bias     [U]       ops.py:9  */
  float *item_bias;   /* item_bias     [I]       ops.py:11 */
  float *user_feat;   /* user_features [U,dim]   ops.py:29 */
  float *item_feat;   /* item_features [I,dim]   ops.py:31 */
  /* Adam slots (TF: adam.py _create_slots: zeros_like each variable) */
  float *m_mu, *v_mu, *m_ub, *v_ub, *m_ib, *v_ib, *m_uf, *v_uf, *m_if, *v_if;
  float beta1_power, beta2_power; /* TF: adam.py _create_slots: initialised to beta1, beta2 */
  int64_t global_step;            /* svd_train_val.py:48 */
  float lr, reg, beta1, beta2, eps;
  int32_t var_mask;
} orc_svd_state;

/* ---- forward: ops.py:13-14,37-38 (gathers), :44-47 (dot + three bias adds), :76-78 (head) -- */
/* logits[b] = ((sum_k u[b,k]*v'[b,k] + mu) + b_u) + b_i ; v' = |v| when ORC_ABS_ITEM.      */
/* tf.multiply rounds every product to fp32; the ORDER of tf.reduce_sum inside TF/Eigen (a    */
/* SIMD packet tree) is unspecified, so the restatement returns the order-independent value:   */
/* the fp32 products summed exactly (double accumulator) and rounded once.  Any fp32 summation */
/* order, TF's included, lies within a few ulp of it.                                          */
static inline float orc_logit(const orc_svd_state *s, int32_t u, int32_t i) {
  const int d = s->dim;
  const float *pu = s->user_feat + (size_t)u * d, *qi = s->item_feat + (size_t)i * d;
  double dacc = 0.0;
  if (s->flags & ORC_ABS_ITEM)
    for (int k = 0; k < d; ++k) { float pr = pu[k] * fabsf(qi[k]); dacc += (double)pr; }
  else
    for (int k = 0; k < d; ++k) { float pr = pu[k] * qi[k]; dacc += (double)pr; }
  float acc = (float)dacc;
  acc = acc + s->mu[0];         /* ops.py:45 */
  acc = acc + s->user_bias[u];  /* ops.py:46 */
  acc = acc + s->item_bias[i];  /* ops.py:47 */
  return acc;
}

/* TF: tf.sigmoid = 1/(1+exp(-x)) (Eigen scalar_logistic_op); tf.round = half-to-even (A.2) */
static inline float orc_sigmoid(float x) { return 1.0f / (1.0f + expf(-x)); }

ORC_API void orc_svd_forward(const orc_svd_state *s, const int32_t *users, const int32_t *items,
                             int64_t B, float *logits, float *infer) {
#pragma omp parallel for schedule(static)
  for (int64_t b = 0; b < B; ++b) {
    float x = orc_logit(s, users[b], items[b]);
    if (logits) logits[b] = x;
    if (infer) {
      if (s->flags & ORC_LOSS_SIGMOID_CE) infer[b] = rintf(orc_sigmoid(x)); /* ops.py:77-78 */
      else infer[b] = x; /* README mode: infer is the raw score (svd_train_val.py:49,104) */
    }
  }
}

/* ---- d cost / d logits per occurrence ------------------------------------------------- */
/* README: cost_l2 = l2_loss(infer - rate) (ops.py:124) -> e = infer - rate.                 */
/* fork:   sum sigmoid_cross_entropy_with_logits (ops.py:125-126); TF nn_impl.py builds it as  */
/*         relu(x) - x*z + log1p(exp(-|x|)); autodiff of that graph (A.2):                    */
/*         [x>=0] - z + (x>=0 ? -1 : 1) * exp(n)/(1+exp(n)),  n = -|x|.                        */
static inline float orc_dloss(int flags, float x, float z) {
  if (!(flags & ORC_LOSS_SIGMOID_CE)) return x - z;
  int cond = x >= 0.0f;
  float n = cond ? -x : x;
  float t = expf(n);
  float sgm = (1.0f / (1.0f + t)) * t;
  float g = (cond ? 1.0f : 0.0f) - z;
  return g + (cond ? -sgm : sgm);
}

/* scalar losses, for the `cost` fetch (ops.py:124-126,140) */
ORC_API double orc_svd_data_loss(const orc_svd_state *s, const float *logits, const float *rates, int64_t B) {
  double acc = 0.0;
  for (int64_t b = 0; b < B; ++b) {
    float x = logits[b], z = rates[b];
    if (s->flags & ORC_LOSS_SIGMOID_CE) {
      float relu = x >= 0.0f ? x : 0.0f, n = x >= 0.0f ? -x : x;
      acc += (double)((relu - x * z) + log1pf(expf(n)));
    } else {
      float e = x - z;
      acc += 0.5 * (double)(e * e);
    }
  }
  return acc;
}

/* regulariser scalar: ops.py:81-89; l2_loss(t) = sum(t^2)/2 over the GATHERED rows, i.e. once */
/* per batch occurrence (A.3).  README: user+item embeddings only; fork adds the two biases.  */
ORC_API double orc_svd_regularizer(const orc_svd_state *s, const int32_t *users, const int32_t *items, int64_t B) {
  double acc = 0.0;
  const int d = s->dim;
  for (int64_t b = 0; b < B; ++b) {
    const float *pu = s->user_feat + (size_t)users[b] * d, *qi = s->item_feat + (size_t)items[b] * d;
    for (int k = 0; k < d; ++k) acc += 0.5 * ((double)pu[k] * pu[k] + (double)qi[k] * qi[k]);
    if (s->flags & ORC_REG_BIAS) {
      float bu = s->user_bias[users[b]], bi = s->item_bias[items[b]];
      acc += 0.5 * ((double)bu * bu + (double)bi * bi);
    }
  }
  return acc;
}

/* ---- backward (TF autodiff under Optimizer.minimize, ops.py:143-149; SURVEY 8a row a10) --- */
/* Per occurrence b, with e = d cost/d logits[b]:                                              */
/*   g_u[b,:] = e*v'[b,:] + reg*u[b,:]                                                         */
/*   g_v[b,:] = e*u[b,:]*(sign(v) if ABS_ITEM) + reg*v[b,:]                                    */
/*   g_bu[b] = e (+ reg*b_u if REG_BIAS), g_bi likewise;  g_mu = sum_b e (dense).              */
/* Each product and the final add are separate fp32 roundings (separate TF kernels + AddN).   */
ORC_API void orc_svd_grads(const orc_svd_state *s, const int32_t *users, const int32_t *items,
                           const float *rates, int64_t B, float *logits_out, float *err_out,
                           float *g_uf, float *g_if, float *g_ub, float *g_ib, float *g_mu) {
  const int d = s->dim;
  const float reg = s->reg;
#pragma omp parallel for schedule(static)
  for (int64_t b = 0; b < B; ++b) {
    const int32_t u = users[b], i = items[b];
    float x = orc_logit(s, u, i);
    float e = orc_dloss(s->flags, x, rates[b]);
    if (logits_out) logits_out[b] = x;
    if (err_out) err_out[b] = e;
    const float *pu = s->user_feat + (size_t)u * d, *qi = s->item_feat + (size_t)i * d;
    float *gu = g_uf + (size_t)b * d, *gv = g_if + (size_t)b * d;
    for (int k = 0; k < d; ++k) {
      float vk = qi[k], uk = pu[k];
      if (s->flags & ORC_ABS_ITEM) {
        float sg = (vk > 0.0f) - (vk < 0.0f);
        float du = e * fabsf(vk);
        float dv = (e * uk) * sg;
        gu[k] = du + reg * uk;
        gv[k] = dv + reg * vk;
      } else {
        float du = e * vk;
        float dv = e * uk;
        gu[k] = du + reg * uk;
        gv[k] = dv + reg * vk;
      }
    }
    if (s->flags & ORC_REG_BIAS) {
      g_ub[b] = e + reg * s->user_bias[u];
      g_ib[b] = e + reg * s->item_bias[i];
    } else {
      g_ub[b] = e;
      g_ib[b] = e;
    }
  }
  /* d cost / d bias_global: reduce_sum of the upstream gradient over the batch (A.3).       */
  /* Eigen's reduction order is unspecified: order-independent restatement as for the dot.   */
  double acc = 0.0;
  for (int64_t b = 0; b < B; ++b) acc += (double)err_out[b];
  *g_mu = (float)acc;
}

/* ---- dedup: TF optimizer.py::_deduplicate_indexed_slices (A.3) --------------------------- */
/* unique_ids, idx = tf.unique(ids): unique_ids in ORDER OF FIRST OCCURRENCE; idx[b] indexes it. */
/* Returns n_uniq. Integer work: bit-exact contract.                                          */
ORC_API int64_t orc_unique_first_occurrence(const int32_t *ids, int64_t B, int32_t *uniq, int32_t *idx) {
  if (B <= 0) return 0;
  uint64_t cap = 16;
  while (cap < (uint64_t)B * 2) cap <<= 1;
  int32_t *keys = (int32_t *)malloc(cap * sizeof(int32_t));
  int32_t *vals = (int32_t *)malloc(cap * sizeof(int32_t));
  memset(vals, 0xff, cap * sizeof(int32_t)); /* -1 = empty */
  int64_t n = 0;
  for (int64_t b = 0; b < B; ++b) {
    uint32_t id = (uint32_t)ids[b];
    uint64_t h = ((uint64_t)id * 0x9E3779B97F4A7C15ull) >> 20 & (cap - 1);
    for (;;) {
      if (vals[h] < 0) { keys[h] = ids[b]; vals[h] = (int32_t)n; uniq[n] = ids[b]; idx[b] = (int32_t)n; ++n; break; }
      if (keys[h] == ids[b]) { idx[b] = vals[h]; break; }
      h = (h + 1) & (cap - 1);
    }
  }
  free(keys); free(vals);
  return n;
}

/* tf.unsorted_segment_sum CPU kernel (A.3): zero-init, then out[idx[b]] += values[b] for b = 0..B-1 IN ORDER */
/* Summation order of the segment sums.  0 (default) = batch order, what TF's CPU kernel does (A.3).  1 = reverse batch  */
/* order: an equally legitimate fp32 evaluation of the same sum (TF's GPU unsorted_segment_sum adds with atomics, in no   */
/* specified order).  Used only by tests/test_oracle.py to MEASURE how far two legitimate orders of this very oracle      */
/* drift apart -- the yardstick for the fp32 parity bar of tests/test_gpu_parity.py (DESIGN.md section 4).                */
static int g_segment_order = 0;
ORC_API void orc_set_segment_order(int order) { g_segment_order = order; }

ORC_API void orc_segment_sum(const float *values, const int32_t *idx, int64_t B, int32_t width,
                             int64_t n_uniq, float *out) {
  memset(out, 0, (size_t)n_uniq * width * sizeof(float));
  for (int64_t bb = 0; bb < B; ++bb) {
    const int64_t b = g_segment_order == 1 ? B - 1 - bb : bb;
    float *o = out + (size_t)idx[b] * width;
    const float *v = values + (size_t)b * width;
    for (int k = 0; k < width; ++k) o[k] = o[k] + v[k];
  }
}

/* ---- TF sparse Adam: adam.py::_apply_sparse_shared (A.4) --------------------------------- */
/* lr_t = lr*sqrt(1-beta2_power)/(1-beta1_power);  m = m*beta1 (WHOLE table);                  */
/* m[uq] += g*(1-beta1); v = v*beta2 (WHOLE table); v[uq] += (g*g)*(1-beta2);                  */
/* var -= (lr_t*m)/(sqrt(v)+eps) (WHOLE table).  Untouched rows keep moving while m != 0.      */
ORC_API float orc_adam_lr_t(float lr, float beta1_power, float beta2_power) {
  float t = sqrtf(1.0f - beta2_power);
  t = lr * t;
  return t / (1.0f - beta1_power);
}

ORC_API void orc_adam_sparse(float *var, float *m, float *v, int64_t rows, int32_t width,
                             const int32_t *uniq, int64_t n_uniq, const float *gsum, float lr_t,
                             float beta1, float beta2, float eps) {
  const int64_t n = rows * (int64_t)width;
  const float omb1 = 1.0f - beta1, omb2 = 1.0f - beta2;
#pragma omp parallel for schedule(static)
  for (int64_t j = 0; j < n; ++j) { m[j] = m[j] * beta1; v[j] = v[j] * beta2; }
#pragma omp parallel for schedule(static)
  for (int64_t q = 0; q < n_uniq; ++q) { /* uniq has no duplicates: rows are independent */
    float *mr = m + (size_t)uniq[q] * width, *vr = v + (size_t)uniq[q] * width;
    const float *g = gsum + (size_t)q * width;
    for (int k = 0; k < width; ++k) {
      float ms = g[k] * omb1;
      mr[k] = mr[k] + ms;
      float vs = (g[k] * g[k]) * omb2;
      vr[k] = vr[k] + vs;
    }
  }
#pragma omp parallel for schedule(static)
  for (int64_t j = 0; j < n; ++j) {
    float den = sqrtf(v[j]) + eps;
    float num = lr_t * m[j];
    var[j] = var[j] - num / den;
  }
}

/* TF dense Adam: training_ops.cc::ApplyAdam (A.5), used for bias_global (dense gradient) */
ORC_API void orc_adam_dense(float *var, float *m, float *v, int64_t n, const float *g, float lr,
                            float beta1_power, float beta2_power, float beta1, float beta2, float eps) {
  float alpha = sqrtf(1.0f - beta2_power);
  alpha = lr * alpha;
  alpha = alpha / (1.0f - beta1_power);
  const float omb1 = 1.0f - beta1, omb2 = 1.0f - beta2;
  for (int64_t j = 0; j < n; ++j) {
    float dm = (g[j] - m[j]) * omb1;
    m[j] = m[j] + dm;
    float dv = (g[j] * g[j] - v[j]) * omb2;
    v[j] = v[j] + dv;
    float num = m[j] * alpha;
    var[j] = var[j] - num / (sqrtf(v[j]) + eps);
  }
}

/* TF GradientDescentOptimizer (ops.py:145): sparse -> scatter_sub(var, ids, lr*values), duplicates */
/* accumulate in batch order, no dedup (A.3); dense -> var -= lr*g.                              */
ORC_API void orc_sgd_scatter(float *var, int32_t width, const int32_t *ids, int64_t B, const float *values, float lr) {
  for (int64_t b = 0; b < B; ++b) {
    float *r = var + (size_t)ids[b] * width;
    const float *g = values + (size_t)b * width;
    for (int k = 0; k < width; ++k) r[k] = r[k] - lr * g[k];
  }
}

/* ---- one full train step: svd_train_val.py:70-72  sess.run([train_op, logits, infer]) ------ */
/* logits/infer are returned from the PRE-update parameters (A.7). Work buffers are malloc'd per */
/* call (this is a checker, not a product).                                                    */
ORC_API int orc_svd_train_step(orc_svd_state *s, const int32_t *users, const int32_t *items,
                               const float *rates, int64_t B, float *logits_out, float *infer_out) {
  const int d = s->dim;
  float *err = (float *)malloc((size_t)B * sizeof(float));
  float *lg = (float *)malloc((size_t)B * sizeof(float));
  float *g_uf = (float *)malloc((size_t)B * d * sizeof(float));
  float *g_if = (float *)malloc((size_t)B * d * sizeof(float));
  float *g_ub = (float *)malloc((size_t)B * sizeof(float));
  float *g_ib = (float *)malloc((size_t)B * sizeof(float));
  float g_mu = 0.0f;
  if (!err || !lg || !g_uf || !g_if || !g_ub || !g_ib) return -1;
  orc_svd_grads(s, users, items, rates, B, lg, err, g_uf, g_if, g_ub, g_ib, &g_mu);
  for (int64_t b = 0; b < B; ++b) {
    if (logits_out) logits_out[b] = lg[b];
    if (infer_out) infer_out[b] = (s->flags & ORC_LOSS_SIGMOID_CE) ? rintf(orc_sigmoid(lg[b])) : lg[b];
  }
  if (s->flags & ORC_OPT_SGD) {
    if (s->var_mask & ORC_VAR_UF) orc_sgd_scatter(s->user_feat, d, users, B, g_uf, s->lr);
    if (s->var_mask & ORC_VAR_IF) orc_sgd_scatter(s->item_feat, d, items, B, g_if, s->lr);
    if (s->var_mask & ORC_VAR_UB) orc_sgd_scatter(s->user_bias, 1, users, B, g_ub, s->lr);
    if (s->var_mask & ORC_VAR_IB) orc_sgd_scatter(s->item_bias, 1, items, B, g_ib, s->lr);
    if (s->var_mask & ORC_VAR_MU) s->mu[0] = s->mu[0] - s->lr * g_mu;
  } else {
    int32_t *uq = (int32_t *)malloc((size_t)B * sizeof(int32_t));
    int32_t *idx = (int32_t *)malloc((size_t)B * sizeof(int32_t));
    float *gs = (float *)malloc((size_t)B * d * sizeof(float));
    float *gsb = (float *)malloc((size_t)B * sizeof(float));
    const float lr_t = orc_adam_lr_t(s->lr, s->beta1_power, s->beta2_power);
    int64_t n = orc_unique_first_occurrence(users, B, uq, idx);
    if (s->var_mask & ORC_VAR_UF) {
      orc_segment_sum(g_uf, idx, B, d, n, gs);
      orc_adam_sparse(s->user_feat, s->m_uf, s->v_uf, s->user_num, d, uq, n, gs, lr_t, s->beta1, s->beta2, s->eps);
    }
    if (s->var_mask & ORC_VAR_UB) {
      orc_segment_sum(g_ub, idx, B, 1, n, gsb);
      orc_adam_sparse(s->user_bias, s->m_ub, s->v_ub, s->user_num, 1, uq, n, gsb, lr_t, s->beta1, s->beta2, s->eps);
    }
    n = orc_unique_first_occurrence(items, B, uq, idx);
    if (s->var_mask & ORC_VAR_IF) {
      orc_segment_sum(g_if, idx, B, d, n, gs);
      orc_adam_sparse(s->item_feat, s->m_if, s->v_if, s->item_num, d, uq, n, gs, lr_t, s->beta1, s->beta2, s->eps);
    }
    if (s->var_mask & ORC_VAR_IB) {
      orc_segment_sum(g_ib, idx, B, 1, n, gsb);
      orc_adam_sparse(s->item_bias, s->m_ib, s->v_ib, s->item_num, 1, uq, n, gsb, lr_t, s->beta1, s->beta2, s->eps);
    }
    if (s->var_mask & ORC_VAR_MU)
      orc_adam_dense(s->mu, s->m_mu, s->v_mu, 1, &g_mu, s->lr, s->beta1_power, s->beta2_power, s->beta1, s->beta2, s->eps);
    /* TF: adam.py::_finish -- powers advance after all applies */
    s->beta1_power = s->beta1_power * s->beta1;
    s->beta2_power = s->beta2_power * s->beta2;
    free(uq); free(idx); free(gs); free(gsb);
  }
  s->global_step += 1; /* minimize(..., global_step=global_step) */
  free(err); free(lg); free(g_uf); free(g_if); free(g_ub); free(g_ib);
  return 0;
}

/* ---- FM forward: forward.py:21-22  fma(x) = mu + x.W + 0.5*(||xV||^2 - sum_f sum_i x_i^2 V_if^2) */
/* forward.py:22 writes x.dot(V**2) (valid for 0/1 features); the canonical x_i^2 form is     */
/* restated (they coincide on the one-hot/multi-hot inputs fm.py:61-93 builds; SURVEY row a19). */
/* X is CSR (indptr[n+1], indices[nnz], data[nnz]).  sum[f] is also returned when non-NULL     */
/* (needed by the backward).                                                                   */
ORC_API void orc_fm_forward(int64_t n_rows, const int64_t *indptr, const int32_t *indices, const float *data,
                            const float *w0, const float *W, const float *V, int32_t dim,
                            float *yhat, float *sums) {
#pragma omp parallel
  {
    /* one s_f / q_f pair of dim floats per thread (rows of any dim, not a fixed stack array) */
    float *s_f = (float *)malloc((size_t)(dim > 0 ? dim : 1) * 2 * sizeof(float));
    float *q_f = s_f + (dim > 0 ? dim : 1);
#pragma omp for schedule(static)
    for (int64_t r = 0; r < n_rows; ++r) {
      float lin = 0.0f;
      for (int f = 0; f < dim; ++f) { s_f[f] = 0.0f; q_f[f] = 0.0f; }
      for (int64_t p = indptr[r]; p < indptr[r + 1]; ++p) {
        const float x = data[p];
        const float *vr = V + (size_t)indices[p] * dim;
        lin = lin + W[indices[p]] * x;
        for (int f = 0; f < dim; ++f) {
          float t = vr[f] * x;
          s_f[f] = s_f[f] + t;
          q_f[f] = q_f[f] + t * t;
        }
      }
      float inter = 0.0f;
      for (int f = 0; f < dim; ++f) inter = inter + (s_f[f] * s_f[f] - q_f[f]);
      yhat[r] = (w0[0] + lin) + 0.5f * inter;
      if (sums) for (int f = 0; f < dim; ++f) sums[(size_t)r * dim + f] = s_f[f];
    }
    free(s_f);
  }
}

/* FM train step in the SVD step's terms (north_star: "the same SE/L2/Adam step"):             */
/* cost = data_loss(yhat, y) + reg * sum over nonzero occurrences of l2_loss(V[row]) (+ W^2 if  */
/* ORC_REG_BIAS), per-nonzero gradients, tf.unique dedup over the batch's feature ids, sparse  */
/* Adam on W and V, dense Adam on w0.  Gradients: d yhat/d W_i = x_i;                          */
/* d yhat/d V_if = x_i*(s_f - V_if*x_i)  (Rendle 2010, eq. 4).                                  */
typedef struct {
  int32_t n_feat, dim, flags;
  float *w0, *W, *V;
  float *m_w0, *v_w0, *m_W, *v_W, *m_V, *v_V;
  float beta1_power, beta2_power;
  int64_t global_step;
  float lr, reg, beta1, beta2, eps;
} orc_fm_state;

ORC_API int orc_fm_train_step(orc_fm_state *s, int64_t n_rows, const int64_t *indptr, const int32_t *indices,
                              const float *data, const float *y, float *yhat_out) {
  const int d = s->dim;
  const int64_t nnz = indptr[n_rows] - indptr[0];
  const int64_t base = indptr[0];
  float *yhat = (float *)malloc((size_t)n_rows * sizeof(float));
  float *sums = (float *)malloc((size_t)n_rows * d * sizeof(float));
  float *gV = (float *)malloc((size_t)(nnz > 0 ? nnz : 1) * d * sizeof(float));
  float *gW = (float *)malloc((size_t)(nnz > 0 ? nnz : 1) * sizeof(float));
  orc_fm_forward(n_rows, indptr, indices, data, s->w0, s->W, s->V, d, yhat, sums);
  double g0_acc = 0.0; /* reduction order unspecified in TF/Eigen: order-independent value, as for the SVD's g_mu */
  for (int64_t r = 0; r < n_rows; ++r) {
    float e = orc_dloss(s->flags, yhat[r], y[r]);
    g0_acc += (double)e;
    for (int64_t p = indptr[r]; p < indptr[r + 1]; ++p) {
      const float x = data[p];
      const int32_t fi = indices[p];
      const float *vr = s->V + (size_t)fi * d;
      float *g = gV + (size_t)(p - base) * d;
      for (int f = 0; f < d; ++f) {
        float t = sums[(size_t)r * d + f] - vr[f] * x;
        t = x * t;
        g[f] = e * t + s->reg * vr[f];
      }
      float gw = e * x;
      if (s->flags & ORC_REG_BIAS) gw = gw + s->reg * s->W[fi];
      gW[p - base] = gw;
    }
  }
  if (yhat_out) memcpy(yhat_out, yhat, (size_t)n_rows * sizeof(float));
  float g0 = (float)g0_acc;
  if (s->flags & ORC_OPT_SGD) {
    orc_sgd_scatter(s->V, d, indices + base, nnz, gV, s->lr);
    orc_sgd_scatter(s->W, 1, indices + base, nnz, gW, s->lr);
    s->w0[0] = s->w0[0] - s->lr * g0;
  } else {
    int32_t *uq = (int32_t *)malloc((size_t)(nnz > 0 ? nnz : 1) * sizeof(int32_t));
    int32_t *idx = (int32_t *)malloc((size_t)(nnz > 0 ? nnz : 1) * sizeof(int32_t));
    float *gs = (float *)malloc((size_t)(nnz > 0 ? nnz : 1) * d * sizeof(float));
    float *gsw = (float *)malloc((size_t)(nnz > 0 ? nnz : 1) * sizeof(float));
    const float lr_t = orc_adam_lr_t(s->lr, s->beta1_power, s->beta2_power);
    int64_t n = orc_unique_first_occurrence(indices + base, nnz, uq, idx);
    orc_segment_sum(gV, idx, nnz, d, n, gs);
    orc_adam_sparse(s->V, s->m_V, s->v_V, s->n_feat, d, uq, n, gs, lr_t, s->beta1, s->beta2, s->eps);
    orc_segment_sum(gW, idx, nnz, 1, n, gsw);
    orc_adam_sparse(s->W, s->m_W, s->v_W, s->n_feat, 1, uq, n, gsw, lr_t, s->beta1, s->beta2, s->eps);
    orc_adam_dense(s->w0, s->m_w0, s->v_w0, 1, &g0, s->lr, s->beta1_power, s->beta2_power, s->beta1, s->beta2, s->eps);
    s->beta1_power = s->beta1_power * s->beta1;
    s->beta2_power = s->beta2_power * s->beta2;
    free(uq); free(idx); free(gs); free(gsw);
  }
  s->global_step += 1;
  free(yhat); free(sums); free(gV); free(gW);
  return 0;
}

/* ---- all-pairs scoring: als3.py:110-113  M = U.V^T + W_user[:,None] + W_work[None,:] + bias -- */
/* numpy does this in float64 (als3.py arrays are float64); restated in double, cast on store.  */
ORC_API void orc_allpairs(const float *U, const float *V, const float *wu, const float *wi, float mu,
                          int64_t n_users, int64_t n_items, int32_t dim, float *M) {
#pragma omp parallel for schedule(static)
  for (int64_t u = 0; u < n_users; ++u)
    for (int64_t i = 0; i < n_items; ++i) {
      double acc = 0.0;
      for (int k = 0; k < dim; ++k) acc += (double)U[u * dim + k] * (double)V[i * dim + k];
      M[u * n_items + i] = (float)(acc + (double)wu[u] + (double)wi[i] + (double)mu);
    }
}

ORC_API int orc_abi_version(void) { return 1; }
