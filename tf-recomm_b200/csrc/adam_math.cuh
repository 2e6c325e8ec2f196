// Shared device code of the Adam kernels (adam.cu: LDG/STG pass, slice rows; adam_ring.cu: TMA-bulk ring pass):
// TF AdamOptimizer's per-element arithmetic in TF's rounding order (TF: adam.py::_apply_sparse_shared, SURVEY A.4) and
// the end-of-step scalar work (TF: training_ops.cc ApplyAdam on bias_global, A.5; adam.py::_finish).
#pragma once
#include "common.cuh"

namespace tfr {

struct AdamK {
  float b1, b2, lr_t, eps, omb1, omb2;
};
__device__ __forceinline__ AdamK load_k(const tfr_opt_scalars* opt) {
  AdamK k;
  k.b1 = opt->beta1; k.b2 = opt->beta2; k.lr_t = opt->lr_t; k.eps = opt->eps;
  k.omb1 = opt->one_minus_beta1; k.omb2 = opt->one_minus_beta2;
  return k;
}
__device__ __forceinline__ void adam_decay(float& var, float& m, float& v, const AdamK& k) {
  m = mul_rn(m, k.b1);
  v = mul_rn(v, k.b2);
  var = sub_rn(var, div_rn(mul_rn(k.lr_t, m), add_rn(sqrt_rn(v), k.eps)));
}
__device__ __forceinline__ void adam_grad(float& var, float& m, float& v, float g, const AdamK& k) {
  m = add_rn(mul_rn(m, k.b1), mul_rn(g, k.omb1));
  v = add_rn(mul_rn(v, k.b2), mul_rn(mul_rn(g, g), k.omb2));
  var = sub_rn(var, div_rn(mul_rn(k.lr_t, m), add_rn(sqrt_rn(v), k.eps)));
}

// end-of-step work folded into the pass (the last CTA to finish does it): dense Adam on bias_global from the
// forward's per-CTA partials + the step scalars (what finish_step_kernel does as a launch of its own)
struct FinishArgs {
  tfr_opt_scalars* opt;  // writable alias of the kernel's (read-only) scalars: written by ONE warp after every CTA
                         // has arrived, i.e. after every read of the step's scalars
  float *mu, *m_mu, *v_mu;
  const float* partials;
  const double* se_partials;
  int n_partials;  // 0 = no end-of-step work in this launch
};
// one warp: fold the per-CTA partials in a fixed order, update bias_global (TF: training_ops.cc ApplyAdam, A.5),
// advance beta powers / lr_t / counters (TF: adam.py::_finish), record the step's float64 squared-error sum
static __device__ __noinline__ void finish_step_scalars(float* mu, float* m_mu, float* v_mu, tfr_opt_scalars* opt,
                                                    const float* partials, const double* se_partials, int n_partials) {
  float a = 0.0f;
  double se = 0.0;
  const int ln = threadIdx.x & 31;
  for (int j = ln; j < n_partials; j += 32) { a = add_rn(a, partials[j]); se += se_partials[j]; }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    a = add_rn(a, __shfl_xor_sync(0xffffffffu, a, o));
    se += __shfl_xor_sync(0xffffffffu, se, o);
  }
  if (ln == 0) {
    const float g = a;  // d cost / d bias_global = sum_b e_b  (A.3)
    opt->g_mu = g;
    opt->se_sum = se;
    if (opt->se_ring && opt->se_ring_len > 0) opt->se_ring[opt->global_step % opt->se_ring_len] = se;
    const bool sgd = opt->flags & TFR_OPT_SGD;
    if (opt->var_mask & TFR_VAR_MU) {
      if (sgd) {
        *mu = sub_rn(*mu, mul_rn(opt->lr, g));
      } else {  // TF: training_ops.cc ApplyAdam (A.5)
        float alpha = sqrt_rn(sub_rn(1.0f, opt->beta2_power));
        alpha = mul_rn(opt->lr, alpha);
        alpha = div_rn(alpha, sub_rn(1.0f, opt->beta1_power));
        float mm = *m_mu, vv = *v_mu;
        mm = add_rn(mm, mul_rn(sub_rn(g, mm), opt->one_minus_beta1));
        vv = add_rn(vv, mul_rn(sub_rn(mul_rn(g, g), vv), opt->one_minus_beta2));
        *m_mu = mm;
        *v_mu = vv;
        *mu = sub_rn(*mu, div_rn(mul_rn(mm, alpha), add_rn(sqrt_rn(vv), opt->eps)));
      }
    }
    if (!sgd) {  // TF: adam.py::_finish
      opt->beta1_power = mul_rn(opt->beta1_power, opt->beta1);
      opt->beta2_power = mul_rn(opt->beta2_power, opt->beta2);
      // lr_t of the NEXT step (TF: _apply_sparse_shared recomputes it from the advanced powers), so that a step
      // needs no kernel in front of the forward; this step's stays for the two-step pass
      opt->lr_t_prev = opt->lr_t;
      float tt = sqrt_rn(sub_rn(1.0f, opt->beta2_power));
      opt->lr_t = div_rn(mul_rn(opt->lr, tt), sub_rn(1.0f, opt->beta1_power));
    }
    opt->global_step += 1;
    opt->batch_cursor += 1;
  }
}


}  // namespace tfr
