// C-ABI glue: error reporting, workspace carving, the full train step (the sequence that replaces one
// sess.run([train_op, logits, infer]) of svd_train_val.py:70-72) and CUDA-graph helpers.
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>

#include <chrono>
#include <map>
#include <mutex>

#include "common.cuh"

namespace tfr {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int sm_count() {  // of the CURRENT device (cached per device: a process may drive several)
  static int cached[64] = {0};
  int dev = 0, n = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return 148;
  if (dev >= 0 && dev < 64 && cached[dev] > 0) return cached[dev];
  if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) return 148;
  if (dev >= 0 && dev < 64) cached[dev] = n;
  return n;
}

namespace {
struct TuneEntry { const char* name; int dflt; };
const TuneEntry kTune[TUNE_COUNT] = {
    {"SMEM_CARVEOUT", 62},   // 141 KB of shared memory on every kernel of the step: four CTAs of the segment-sum kernel
                             // (32 KB each) per SM, and enough L1 for the LDG pass (100 %: pass 125 -> 149 us)
    {"TILES_CARVEOUT", -1}, {"SEG_MAX_UNITS", 0}, {"SEG_TILE", 0}, {"STREAM_COPY_ONLY", 0}, {"STREAM_LD", 2},
    {"STREAM_ST", 0}, {"STREAM_CTAS_PER_SM", 2}, {"STREAM_UNROLL", 2}, {"STREAM_THREADS", 448}, {"STREAM_DYNAMIC", 0},
    // the TMA-bulk ring pass is OFF by default: alone it matches the LDG pass (135 vs 137 us at the ML-25M shape), in
    // situ -- the next batch's id sort competing for issue slots with its 16 consumer warps per SM -- it loses (150-157
    // vs 125 us); profiles/r02_pass_ring_vs_ldg.md
    {"PASS_RING", 0},
    {"RING_STAGES", 4}, {"RING_STAGE_KB", 24}, {"RING_THREADS", 320}, {"RING_L2_HINT", 2}, {"RING_CTAS_PER_SM", 2},
    {"RING_SLOT_MODE", 1}, {"AP_STAGES", 7}, {"TL_EVERY_CTA", 0},
    // programmatic dependent launch along tiles -> fix-up -> pass: no gain at the ML-25M shape (178.2 vs 177.5 us per
    // step) and a loss at the ML-1M shape (the early-resident dependents delay the side stream's id sort: 53 vs 37 us)
    {"PDL", 0},
    {"SORT_SPLIT", 0},
    {"RANK_CHUNK", 4096}, {"RANK_STAGES", 7},
    // ALS item half-sweep at the ML-25M shape, d = 128 (NVIDIA B200, 1000 W, profiles/r06_als_ml25m.json): 112.3 / 111.1 /
    // 111.1 / 112.6 / 121.4 ms at 1024 / 2048 / 4096 / 8192 / 16384 ratings per chunk; 4096 ties the fastest with a 224 MB
    // workspace (2048: 491 MB)
    {"ALS_CHUNK", 4096},
    // 0: the fused segment sums take segsum_tiles_kernel<4, L, 4, true, false> where chain_tiles_kernel<L, T> would run;
    // the two compute the same bits, and the old kernel is the reference the tests hold the chain kernel to
    {"SEG_CHAIN", 1},
};
std::mutex g_tune_mu;
int g_tune_val[TUNE_COUNT];
bool g_tune_known[TUNE_COUNT];
}  // namespace

int tune(TuneKey k) {
  std::lock_guard<std::mutex> g(g_tune_mu);
  if (!g_tune_known[k]) {
    char env[64];
    snprintf(env, sizeof(env), "TFR_%s", kTune[k].name);
    const char* e = getenv(env);
    g_tune_val[k] = e ? atoi(e) : kTune[k].dflt;
    g_tune_known[k] = true;
  }
  return g_tune_val[k];
}

int fwd_err_n_partials(int dim, int64_t B);
int advance_prefetch_cursor(tfr_opt_scalars* opt, cudaStream_t st, bool prime);
int seg_tile(int64_t B, int dim);
int svd_segment_grads_impl(const tfr_svd_tables* t, const tfr_opt_scalars* opt, const int32_t* users,
                           const int32_t* items, int64_t B, const tfr_svd_step_ws* ws, int flags_host, void* stream);
int adam_pass_and_finish(const tfr_adam_table* tabs, int nt, const tfr_svd_tables* t, tfr_opt_scalars* opt,
                         const tfr_svd_step_ws* ws, int n_partials, int tl_slot, void* stream);
int adam_pair_pass_and_finish(const tfr_adam_table* tabs, const float* const* gsum0, int nt, const tfr_svd_tables* t,
                              tfr_opt_scalars* opt, const tfr_svd_step_ws* ws, int n_partials, void* stream);
int adam_bring_and_finish(const tfr_slice_update* sides, const int64_t* const* slot, int32_t width, int64_t n,
                          const tfr_svd_tables* t, tfr_opt_scalars* opt, const tfr_svd_step_ws* ws, int n_partials,
                          void* stream);

void prep_kernel(const void* fn) { prep_kernel_carveout(fn, 0); }

void prep_kernel_carveout(const void* fn, size_t smem_per_sm) {
  static std::mutex mu;
  static std::map<const void*, int> applied;  // the carve-out a kernel was last given
  int carve = tune(TUNE_SMEM_CARVEOUT);
  if (carve > 0 && smem_per_sm > 0) {
    const size_t need = smem_per_sm + 4096;  // + the per-CTA reserve
    const int pct = (int)((need * 100 + 228 * 1024 - 1) / (228 * 1024));
    if (pct > carve) carve = pct > 100 ? 100 : pct;
  }
  std::lock_guard<std::mutex> g(mu);
  auto it = applied.find(fn);
  if (it != applied.end() && it->second == carve) return;
  if (carve > 0) cudaFuncSetAttribute(fn, cudaFuncAttributePreferredSharedMemoryCarveout, carve);
  cudaGetLastError();
  applied[fn] = carve;
}

}  // namespace tfr

using namespace tfr;

extern "C" const char* tfr_last_error(void) { return g_err; }
extern "C" int tfr_abi_version(void) { return TFR_ABI_VERSION; }

extern "C" int tfr_tune_set(const char* name, int32_t value) {
  TFR_CHECK_ARG(name);
  for (int k = 0; k < TUNE_COUNT; ++k)
    if (!strcmp(name, kTune[k].name)) {
      std::lock_guard<std::mutex> g(g_tune_mu);
      g_tune_val[k] = value;
      g_tune_known[k] = true;
      return TFR_OK;
    }
  set_error("unknown tuning knob %s", name);
  return TFR_ERR_INVALID;
}

extern "C" int tfr_tune_get(const char* name, int32_t* value) {
  TFR_CHECK_ARG(name && value);
  for (int k = 0; k < TUNE_COUNT; ++k)
    if (!strcmp(name, kTune[k].name)) {
      *value = tune((TuneKey)k);
      return TFR_OK;
    }
  set_error("unknown tuning knob %s", name);
  return TFR_ERR_INVALID;
}

extern "C" int tfr_device_sm_count(void) {
  int dev = 0, n = 0;
  TFR_CUDA(cudaGetDevice(&dev));
  TFR_CUDA(cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev));
  return n;
}

__global__ void set_se_ring_kernel(tfr_opt_scalars* opt, double* ring, int64_t len) {
  opt->se_ring = ring;
  opt->se_ring_len = len;
}

__global__ void set_timeline_kernel(tfr_opt_scalars* opt, uint64_t* tl) { opt->timeline = tl; }

extern "C" int tfr_opt_set_timeline(tfr_opt_scalars* opt_dev, uint64_t* timeline, void* stream) {
  TFR_CHECK_ARG(opt_dev);
  set_timeline_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(opt_dev, timeline);
  TFR_LAUNCH_CHECK();
  return TFR_OK;
}

extern "C" int tfr_opt_set_se_ring(tfr_opt_scalars* opt_dev, double* se_ring, int64_t se_ring_len, void* stream) {
  TFR_CHECK_ARG(opt_dev && se_ring_len >= 0);
  set_se_ring_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(opt_dev, se_ring, se_ring_len);
  TFR_LAUNCH_CHECK();
  return TFR_OK;
}

// ---- step workspace ---------------------------------------------------------------------------------

static int64_t carve(char* base, int64_t B, int32_t dim, tfr_svd_step_ws* o) {
  int64_t off = 0;
  auto take = [&](int64_t bytes) {
    char* p = base ? base + off : nullptr;
    off += align_up(bytes, 256);
    return p;
  };
  const int kTile = seg_tile(B, dim);  // 32, 16 or 8 sorted entries per tile (segsum.cu)
  const int64_t n_tiles = (B + kTile - 1) / kTile;
  tfr_svd_step_ws w;
  memset(&w, 0, sizeof(w));
  w.err = (float*)take(B * 4);
  // + 1: [TFR_MAX_PARTIALS] receives the partials folded by the fix-up's last CTA (off the table pass's tail)
  w.partials = (float*)take((TFR_MAX_PARTIALS + 1) * 4);
  w.se_partials = (double*)take((TFR_MAX_PARTIALS + 1) * 8);
  w.su_ids = (int32_t*)take(B * 4);
  w.su_pos = (int32_t*)take(B * 4);
  w.si_ids = (int32_t*)take(B * 4);
  w.si_pos = (int32_t*)take(B * 4);
  w.gsum_uf = (float*)take(B * (int64_t)dim * 4);
  w.gsum_if = (float*)take(B * (int64_t)dim * 4);
  w.gsum_ub = (float*)take(B * 4);
  w.gsum_ib = (float*)take(B * 4);
  w.cont_uf = (float*)take(n_tiles * dim * 4);
  w.cont_if = (float*)take(n_tiles * dim * 4);
  w.tail_uf = (float*)take(n_tiles * dim * 4);
  w.tail_if = (float*)take(n_tiles * dim * 4);
  w.cont_ub = (float*)take(n_tiles * 4);
  w.cont_ib = (float*)take(n_tiles * 4);
  w.tail_ub = (float*)take(n_tiles * 4);
  w.tail_ib = (float*)take(n_tiles * 4);
  w.kind_u = (uint8_t*)take(n_tiles);
  w.kind_i = (uint8_t*)take(n_tiles);
  w.fix_list_u = (int32_t*)take(n_tiles * 4);
  w.fix_list_i = (int32_t*)take(n_tiles * 4);
  w.sort_ws_bytes = tfr_dedup_workspace_bytes(B);
  w.sort_ws = take(w.sort_ws_bytes);
  w.fix_count = base ? reinterpret_cast<uint32_t*>(reinterpret_cast<char*>(w.sort_ws) + 64) : nullptr;
  w.tile = kTile;
  w.n_tiles = (int32_t)n_tiles;
  if (o) *o = w;
  return off;
}

extern "C" int64_t tfr_svd_step_workspace_bytes(int64_t B, int32_t dim) {
  if (B <= 0 || dim <= 0) return TFR_ERR_INVALID;
  return carve(nullptr, B, dim, nullptr) + 256;
}

extern "C" int tfr_svd_step_carve(void* workspace, int64_t workspace_bytes, int64_t B, int32_t dim,
                                  tfr_svd_step_ws* out) {
  TFR_CHECK_ARG(workspace && out && B > 0 && dim > 0);
  if (workspace_bytes < tfr_svd_step_workspace_bytes(B, dim)) {
    set_error("step workspace too small: %lld < %lld", (long long)workspace_bytes,
              (long long)tfr_svd_step_workspace_bytes(B, dim));
    return TFR_ERR_WORKSPACE;
  }
  char* base = reinterpret_cast<char*>(align_up((int64_t)(uintptr_t)workspace, 256));
  carve(base, B, dim, out);
  return TFR_OK;
}

// ---- the step ------------------------------------------------------------------------------------------
//   SORT (side stream, optional): id sort (needs only the ids)   ||   S0: forward + d cost/d logits
//   S0: segment sums (need err + sorted pairs) -> fix-up  (write gsum and the row -> slot maps)
//   S0: Adam: ONE in-order pass over every row of every table  |  SGD: slice rows only (ops.py:145)
//   S0: finish
static int run_step(const tfr_svd_tables* t, tfr_opt_scalars* opt, const int32_t* users, const int32_t* items,
                    const float* rates, int64_t B, float* logits, float* infer, int32_t flags, int32_t var_mask,
                    void* workspace, int64_t workspace_bytes, void* stream, void* const* side_streams, int32_t n_side,
                    void* const* fj_events, bool presorted, int phases = 3) {
  TFR_CHECK_ARG(t && opt && users && items && rates && B > 0 && t->dim > 0);
  TFR_CHECK_ARG(n_side >= 0 && n_side <= 1 && (n_side == 0 || (side_streams && fj_events && fj_events[0] && fj_events[1])));
  cudaEvent_t ev_fork = n_side > 0 ? (cudaEvent_t)fj_events[0] : nullptr;
  cudaEvent_t ev_join = n_side > 0 ? (cudaEvent_t)fj_events[1] : nullptr;
  // flags / var_mask repeat what the caller gave tfr_opt_init: the device copy drives the kernels, the
  // host copy selects which launches are issued (var_list: untrained tables get no launch at all).
  const bool sgd = flags & TFR_OPT_SGD;
  // row-sharded mode trains with Adam only: the SGD slice update takes every run head of the sorted keys for a row,
  // the "not mine" run (key user_num / item_num) included, one row past the local tables
  TFR_CHECK_ARG(!(sgd && t->g_user_feat));
  TFR_CHECK_ARG(sgd || (t->m_uf && t->v_uf && t->m_if && t->v_if && t->m_ub && t->v_ub && t->m_ib && t->v_ib &&
                        t->m_mu && t->v_mu));
  tfr_svd_step_ws ws;
  int rc = tfr_svd_step_carve(workspace, workspace_bytes, B, t->dim, &ws);
  if (rc) return rc;
  cudaStream_t s0 = (cudaStream_t)stream;
  cudaStream_t sorts = (n_side > 0 && !presorted) ? (cudaStream_t)side_streams[0] : s0;
  const int dim = t->dim;
  // Single-table mode: the forward is fused into the segment sums.  Row-sharded mode (g_* set): every rank needs
  // every occurrence's error, the local tiles only visit the occurrences of local rows -> separate forward.
  const bool fused = t->g_user_feat == nullptr;
  // fused: the fix-up's last CTA has already folded the forward's per-CTA partial sums into [TFR_MAX_PARTIALS]
  tfr_svd_step_ws ws_fin = ws;
  int n_partials = fused ? 1 : fwd_err_n_partials(dim, B);
  if (fused) { ws_fin.partials = ws.partials + TFR_MAX_PARTIALS; ws_fin.se_partials = ws.se_partials + TFR_MAX_PARTIALS; }
  if (!(phases & 1)) goto phase2;
  if (sorts != s0) {
    TFR_CUDA(cudaEventRecord(ev_fork, s0));
    TFR_CUDA(cudaStreamWaitEvent(sorts, ev_fork, 0));
  }
  // + 1: in row-sharded mode the value user_num / item_num itself occurs (the "not mine" mark)
  if (!presorted && (rc = tfr_dedup_sort_pairs_tl(users, (int64_t)t->user_num + 1, ws.su_ids, ws.su_pos, items,
                                                  (int64_t)t->item_num + 1, ws.si_ids, ws.si_pos, B, ws.sort_ws,
                                                  ws.sort_ws_bytes, opt, sorts)))
    return rc;
  if (!fused && (rc = tfr_svd_fwd_err(t, opt, users, items, rates, B, logits, infer, &ws, s0))) return rc;
  if (sorts != s0) {
    TFR_CUDA(cudaEventRecord(ev_join, sorts));
    TFR_CUDA(cudaStreamWaitEvent(s0, ev_join, 0));
  }
  if (fused) {
    if ((rc = tfr_svd_fwd_segment_grads(t, opt, users, items, rates, B, logits, infer, flags, &ws, s0))) return rc;
  } else {
    if ((rc = svd_segment_grads_impl(t, opt, users, items, B, &ws, flags, s0))) return rc;
  }
phase2:
  if (!(phases & 2)) return TFR_OK;
  if (!sgd) {
    tfr_adam_table tabs[4];
    int nt = 0;
    // the small scalar-path tables first: their few trips overlap the start of the feature-table stream instead of
    // forming a tail after it
    if (var_mask & TFR_VAR_UB) tabs[nt++] = tfr_adam_table{t->user_bias, t->m_ub, t->v_ub, t->user_num, 1, t->user_slot, ws.gsum_ub, 0};
    if (var_mask & TFR_VAR_IB) tabs[nt++] = tfr_adam_table{t->item_bias, t->m_ib, t->v_ib, t->item_num, 1, t->item_slot, ws.gsum_ib, 0};
    if (var_mask & TFR_VAR_IF) tabs[nt++] = tfr_adam_table{t->item_feat, t->m_if, t->v_if, t->item_num, dim, t->item_slot, ws.gsum_if, t->feat_stride};
    if (var_mask & TFR_VAR_UF) tabs[nt++] = tfr_adam_table{t->user_feat, t->m_uf, t->v_uf, t->user_num, dim, t->user_slot, ws.gsum_uf, t->feat_stride};
    return adam_pass_and_finish(tabs, nt, t, opt, &ws_fin, n_partials, TFR_TL_STREAM_UF, s0);
  }
  {
    tfr_slice_update sides[2];
    int ns = 0;
    if (var_mask & (TFR_VAR_UF | TFR_VAR_UB))
      sides[ns++] = tfr_slice_update{(var_mask & TFR_VAR_UF) ? t->user_feat : nullptr, nullptr, nullptr,
                                     (var_mask & TFR_VAR_UB) ? t->user_bias : nullptr, nullptr, nullptr,
                                     ws.su_ids, ws.gsum_uf, ws.gsum_ub, t->feat_stride};
    if (var_mask & (TFR_VAR_IF | TFR_VAR_IB))
      sides[ns++] = tfr_slice_update{(var_mask & TFR_VAR_IF) ? t->item_feat : nullptr, nullptr, nullptr,
                                     (var_mask & TFR_VAR_IB) ? t->item_bias : nullptr, nullptr, nullptr,
                                     ws.si_ids, ws.gsum_if, ws.gsum_ib, t->feat_stride};
    if (ns && (rc = tfr_adam_slice_multi(sides, ns, dim, B, opt, 1, TFR_TL_TOUCHED_U, s0))) return rc;
  }
  return tfr_svd_finish_step(t, opt, users, items, B, &ws_fin, n_partials, s0);
}

extern "C" int tfr_svd_train_step(const tfr_svd_tables* t, tfr_opt_scalars* opt, const int32_t* users,
                                  const int32_t* items, const float* rates, int64_t B, float* logits, float* infer,
                                  int32_t flags, int32_t var_mask, void* workspace, int64_t workspace_bytes,
                                  void* stream, void* const* side_streams, int32_t n_side,
                                  void* const* fork_join_events) {
  return run_step(t, opt, users, items, rates, B, logits, infer, flags, var_mask, workspace, workspace_bytes, stream,
                  side_streams, n_side, fork_join_events, false);
}

extern "C" int tfr_svd_train_step_presorted(const tfr_svd_tables* t, tfr_opt_scalars* opt, const int32_t* users,
                                            const int32_t* items, const float* rates, int64_t B, float* logits,
                                            float* infer, int32_t flags, int32_t var_mask, int32_t phases,
                                            void* workspace, int64_t workspace_bytes, void* stream) {
  TFR_CHECK_ARG(phases >= 1 && phases <= 3);
  return run_step(t, opt, users, items, rates, B, logits, infer, flags, var_mask, workspace, workspace_bytes, stream,
                  nullptr, 0, nullptr, true, phases);
}

// ---- two steps per table pass (include/tfrecomm.h: tfr_svd_pair_bring / tfr_svd_pair_pass) ----------------------------
static int pair_args(const tfr_svd_tables* t, tfr_opt_scalars* opt, int64_t B, int32_t flags, void* ws_t,
                     int64_t ws_t_bytes, void* ws_next, int64_t ws_next_bytes, tfr_svd_step_ws* a, tfr_svd_step_ws* b) {
  TFR_CHECK_ARG(t && opt && B > 0 && t->dim > 0 && ws_t && ws_next && ws_t != ws_next);
  // Adam on single-table tables: SGD has no table-wide pass, the row-sharded step folds its partial sums elsewhere
  TFR_CHECK_ARG(!(flags & TFR_OPT_SGD) && t->g_user_feat == nullptr && t->user_slot && t->item_slot);
  TFR_CHECK_ARG(t->m_uf && t->v_uf && t->m_if && t->v_if && t->m_ub && t->v_ub && t->m_ib && t->v_ib && t->m_mu && t->v_mu);
  int rc = tfr_svd_step_carve(ws_t, ws_t_bytes, B, t->dim, a);
  if (rc) return rc;
  if ((rc = tfr_svd_step_carve(ws_next, ws_next_bytes, B, t->dim, b))) return rc;
  // the fused step: its fix-up's last CTA folded the partial sums into [TFR_MAX_PARTIALS]
  a->partials += TFR_MAX_PARTIALS; a->se_partials += TFR_MAX_PARTIALS;
  b->partials += TFR_MAX_PARTIALS; b->se_partials += TFR_MAX_PARTIALS;
  return TFR_OK;
}

extern "C" int tfr_svd_pair_bring(const tfr_svd_tables* t, tfr_opt_scalars* opt, int64_t B, int32_t flags,
                                  int32_t var_mask, void* ws_t, int64_t ws_t_bytes, void* ws_next, int64_t ws_next_bytes,
                                  void* stream) {
  tfr_svd_step_ws a, b;
  int rc = pair_args(t, opt, B, flags, ws_t, ws_t_bytes, ws_next, ws_next_bytes, &a, &b);
  if (rc) return rc;
  const bool uf = var_mask & TFR_VAR_UF, ub = var_mask & TFR_VAR_UB, itf = var_mask & TFR_VAR_IF, ib = var_mask & TFR_VAR_IB;
  const tfr_slice_update sides[2] = {
      {uf ? t->user_feat : nullptr, t->m_uf, t->v_uf, ub ? t->user_bias : nullptr, t->m_ub, t->v_ub, b.su_ids,
       a.gsum_uf, a.gsum_ub, t->feat_stride},
      {itf ? t->item_feat : nullptr, t->m_if, t->v_if, ib ? t->item_bias : nullptr, t->m_ib, t->v_ib, b.si_ids,
       a.gsum_if, a.gsum_ib, t->feat_stride}};
  const int64_t* slots[2] = {t->user_slot, t->item_slot};
  return adam_bring_and_finish(sides, slots, t->dim, B, t, opt, &a, 1, stream);
}

extern "C" int tfr_svd_pair_pass(const tfr_svd_tables* t, tfr_opt_scalars* opt, int64_t B, int32_t flags,
                                 int32_t var_mask, void* ws_t, int64_t ws_t_bytes, void* ws_next, int64_t ws_next_bytes,
                                 void* stream) {
  tfr_svd_step_ws a, b;
  int rc = pair_args(t, opt, B, flags, ws_t, ws_t_bytes, ws_next, ws_next_bytes, &a, &b);
  if (rc) return rc;
  const int dim = t->dim;
  tfr_adam_table tabs[4];
  const float* gsum0[4];
  int nt = 0;
  // the order of run_step's pass
  if (var_mask & TFR_VAR_UB) { gsum0[nt] = a.gsum_ub; tabs[nt++] = tfr_adam_table{t->user_bias, t->m_ub, t->v_ub, t->user_num, 1, t->user_slot, b.gsum_ub, 0}; }
  if (var_mask & TFR_VAR_IB) { gsum0[nt] = a.gsum_ib; tabs[nt++] = tfr_adam_table{t->item_bias, t->m_ib, t->v_ib, t->item_num, 1, t->item_slot, b.gsum_ib, 0}; }
  if (var_mask & TFR_VAR_IF) { gsum0[nt] = a.gsum_if; tabs[nt++] = tfr_adam_table{t->item_feat, t->m_if, t->v_if, t->item_num, dim, t->item_slot, b.gsum_if, t->feat_stride}; }
  if (var_mask & TFR_VAR_UF) { gsum0[nt] = a.gsum_uf; tabs[nt++] = tfr_adam_table{t->user_feat, t->m_uf, t->v_uf, t->user_num, dim, t->user_slot, b.gsum_uf, t->feat_stride}; }
  return adam_pair_pass_and_finish(tabs, gsum0, nt, t, opt, &b, 1, stream);
}

// The step from the sort on, for the all-to-all sharded exchange: keys and ws.err by arrival position are the caller's
// (tfr_shard_owner_prepare), the partner rows come from t->g_* by position, the step's d cost/d bias_global and squared
// error are the all-reduced scalars.
extern "C" int tfr_svd_train_step_gathered(const tfr_svd_tables* t, tfr_opt_scalars* opt, const int32_t* keys_u,
                                           const int32_t* keys_i, int64_t n, int32_t flags, int32_t var_mask,
                                           const float* sum_err, const double* sum_se, void* workspace,
                                           int64_t workspace_bytes, void* stream) {
  TFR_CHECK_ARG(t && opt && n >= 0 && t->dim > 0 && sum_err && sum_se && workspace);
  TFR_CHECK_ARG(!(flags & TFR_OPT_SGD));   // the sharded path trains with Adam (BASELINE configs[4])
  TFR_CHECK_ARG(n == 0 || (keys_u && keys_i && t->g_user_feat && t->g_item_feat));
  tfr_svd_step_ws ws;
  int rc = tfr_svd_step_carve(workspace, workspace_bytes, n > 0 ? n : 1, t->dim, &ws);
  if (rc) return rc;
  if (n > 0) {
    if ((rc = tfr_dedup_sort_pairs_tl(keys_u, (int64_t)t->user_num + 1, ws.su_ids, ws.su_pos, keys_i, (int64_t)t->item_num + 1,
                                      ws.si_ids, ws.si_pos, n, ws.sort_ws, ws.sort_ws_bytes, opt, stream)))
      return rc;
    if ((rc = svd_segment_grads_impl(t, opt, keys_u, keys_i, n, &ws, flags, stream))) return rc;
  }
  tfr_svd_step_ws ws_fin = ws;
  ws_fin.partials = const_cast<float*>(sum_err);
  ws_fin.se_partials = const_cast<double*>(sum_se);
  tfr_adam_table tabs[4];
  int nt = 0;
  const int dim = t->dim;
  if (var_mask & TFR_VAR_UB) tabs[nt++] = tfr_adam_table{t->user_bias, t->m_ub, t->v_ub, t->user_num, 1, t->user_slot, ws.gsum_ub, 0};
  if (var_mask & TFR_VAR_IB) tabs[nt++] = tfr_adam_table{t->item_bias, t->m_ib, t->v_ib, t->item_num, 1, t->item_slot, ws.gsum_ib, 0};
  if (var_mask & TFR_VAR_IF) tabs[nt++] = tfr_adam_table{t->item_feat, t->m_if, t->v_if, t->item_num, dim, t->item_slot, ws.gsum_if, t->feat_stride};
  if (var_mask & TFR_VAR_UF) tabs[nt++] = tfr_adam_table{t->user_feat, t->m_uf, t->v_uf, t->user_num, dim, t->user_slot, ws.gsum_uf, t->feat_stride};
  return adam_pass_and_finish(tabs, nt, t, opt, &ws_fin, 1, TFR_TL_STREAM_UF, stream);
}

extern "C" int tfr_svd_prefetch_batch(const tfr_svd_tables* t, tfr_opt_scalars* opt, const int32_t* col_user,
                                      const int32_t* col_item, const float* col_rate, const int64_t* row_index,
                                      int64_t batch_index, int64_t B, int32_t* users, int32_t* items, float* rates,
                                      void* workspace, int64_t workspace_bytes, void* stream) {
  TFR_CHECK_ARG(t && B > 0 && t->dim > 0 && batch_index >= -3);
  tfr_svd_step_ws ws;
  int rc = tfr_svd_step_carve(workspace, workspace_bytes, B, t->dim, &ws);
  if (rc) return rc;
  if ((rc = tfr_svd_batch_assemble(t, opt, col_user, col_item, col_rate, row_index, batch_index == -3 ? -1 : batch_index,
                                   B, users, items, rates, stream)))
    return rc;
  // stream-ordered after the assemble kernel has read it: the next assemble-ahead draws the following batch
  if (batch_index <= -2 && (rc = advance_prefetch_cursor(opt, (cudaStream_t)stream, batch_index == -3))) return rc;
  return tfr_dedup_sort_pairs_tl(users, (int64_t)t->user_num + 1, ws.su_ids, ws.su_pos, items,
                                 (int64_t)t->item_num + 1, ws.si_ids, ws.si_pos, B, ws.sort_ws, ws.sort_ws_bytes, opt,
                                 stream);
}

// ---- host side of the feed boundary ----------------------------------------------------------------------------
namespace {
// returns the number of values outside [0, bound) (bound <= 0: unchecked), judged on the SOURCE value so that an id
// that does not fit int32 cannot alias a valid one after the cast
template <typename Out, typename In>
int64_t pack_col(const char* src, int64_t stride, int64_t n, Out* dst, int64_t bound) {
  // a 65536-row batch is ~1.5 MB of float64 in, 0.75 MB out: split over a few host threads (memory-bound)
  const int nt = n >= 16384 ? 4 : 1;
  int64_t bad = 0;
#pragma omp parallel for num_threads(nt) schedule(static) reduction(+ : bad)
  for (int64_t c = 0; c < nt; ++c) {
    const int64_t k0 = n * c / nt, k1 = n * (c + 1) / nt;
    const In lo = (In)0, hi = (In)bound;
    if (stride == (int64_t)sizeof(In)) {
      const In* p = reinterpret_cast<const In*>(src);
      if (bound > 0) {
        for (int64_t k = k0; k < k1; ++k) { const In x = p[k]; bad += !(x >= lo && x < hi); dst[k] = (Out)x; }
      } else {
        for (int64_t k = k0; k < k1; ++k) dst[k] = (Out)p[k];  // contiguous: vectorised by the host compiler
      }
    } else {
      for (int64_t k = k0; k < k1; ++k) {
        const In x = *reinterpret_cast<const In*>(src + k * stride);
        if (bound > 0) bad += !(x >= lo && x < hi);
        dst[k] = (Out)x;
      }
    }
  }
  return bad;
}
template <typename Out>
int64_t pack_any(const void* src, int dtype, int64_t stride, int64_t n, Out* dst, int64_t bound = 0) {
  const char* p = static_cast<const char*>(src);
  switch (dtype) {
    case 0: return pack_col<Out, double>(p, stride, n, dst, bound);
    case 1: return pack_col<Out, float>(p, stride, n, dst, bound);
    case 2: return pack_col<Out, int32_t>(p, stride, n, dst, bound);
    case 3: return pack_col<Out, int64_t>(p, stride, n, dst, bound);
  }
  return -1;
}
}  // namespace

extern "C" int tfr_host_pack_feed_checked(const void* users_host, int32_t users_dtype, int64_t users_stride,
                                          const void* items_host, int32_t items_dtype, int64_t items_stride,
                                          const void* rates_host, int32_t rates_dtype, int64_t rates_stride, int64_t n,
                                          void* staging_host, int64_t user_num, int64_t item_num) {
  TFR_CHECK_ARG(n >= 0 && staging_host && (n == 0 || (users_host && items_host && rates_host)));
  TFR_CHECK_ARG(users_dtype >= 0 && users_dtype <= 3 && items_dtype >= 0 && items_dtype <= 3 && rates_dtype >= 0 &&
                rates_dtype <= 3);
  TFR_CHECK_ARG(user_num < ((int64_t)1 << 31) && item_num < ((int64_t)1 << 31));
  int32_t* ids = static_cast<int32_t*>(staging_host);
  float* rates = reinterpret_cast<float*>(ids + 2 * n);
  const int64_t bad_u = pack_any<int32_t>(users_host, users_dtype, users_stride, n, ids, user_num);
  const int64_t bad_i = pack_any<int32_t>(items_host, items_dtype, items_stride, n, ids + n, item_num);
  pack_any<float>(rates_host, rates_dtype, rates_stride, n, rates);
  if (bad_u || bad_i) {
    set_error("indices out of range: %lld user ids outside [0, %lld), %lld item ids outside [0, %lld)", (long long)bad_u,
              (long long)user_num, (long long)bad_i, (long long)item_num);
    return TFR_ERR_INVALID;
  }
  return TFR_OK;
}

extern "C" int tfr_host_pack_feed(const void* users_host, int32_t users_dtype, int64_t users_stride,
                                  const void* items_host, int32_t items_dtype, int64_t items_stride,
                                  const void* rates_host, int32_t rates_dtype, int64_t rates_stride, int64_t n,
                                  void* staging_host) {
  return tfr_host_pack_feed_checked(users_host, users_dtype, users_stride, items_host, items_dtype, items_stride,
                                    rates_host, rates_dtype, rates_stride, n, staging_host, 0, 0);
}

// ---- the feed path (include/tfrecomm.h: "the feed_dict step") -----------------------------------------------------------
extern "C" int tfr_svd_feed_stage(const tfr_svd_tables* t, tfr_feed_set* set, const void* users_host, int32_t users_dtype,
                                  int64_t users_stride, const void* items_host, int32_t items_dtype, int64_t items_stride,
                                  const void* rates_host, int32_t rates_dtype, int64_t rates_stride, int64_t B) {
  TFR_CHECK_ARG(t && set && B > 0 && t->dim > 0 && set->h_feed && set->ev_h2d);
  set->sorted = 0;
  set->staged = 0;
  if (set->used) {
    // The previous copy out of h_feed is done.  ev_h2d covers the eager path; a copy made by a step graph's fetch kernel is
    // only known to be over when the step that CONSUMED that batch has finished (ev_done, recorded eagerly behind its
    // graph: an event-record node inside a launched graph does not hold a host wait back before it has executed).
    TFR_CUDA(cudaEventSynchronize((cudaEvent_t)set->ev_h2d));
    if (set->ev_done) TFR_CUDA(cudaEventSynchronize((cudaEvent_t)set->ev_done));
  }
  const int rc = tfr_host_pack_feed_checked(users_host, users_dtype, users_stride, items_host, items_dtype, items_stride,
                                            rates_host, rates_dtype, rates_stride, B, set->h_feed, t->user_num, t->item_num);
  if (rc) return rc;
  set->used = 1;
  set->staged = 1;
  return TFR_OK;
}

// The two ends of the feed graph as kernels over zero-copy (pinned, device-mapped) host memory -- what the batch assembly is
// to the device-resident stream path; a graph of kernel nodes only (with memcpy nodes in the side branch nothing of that
// branch ran before the table pass had drained: profiles/r02_feed_path.md).
// fetch: [users | items | rates] of the staged batch, 3 * B 32-bit words; four independent 128-bit loads per thread keep
// enough PCIe reads in flight from the one CTA per SM that fits beside the table pass.
constexpr int FETCH_UNROLL = 4;
__global__ void __launch_bounds__(256) feed_fetch_kernel(const uint32_t* __restrict__ h_src, uint32_t* __restrict__ d_dst,
                                                         int64_t words) {
  const int64_t n16 = words / 4;
  const bool vec = (((uintptr_t)h_src | (uintptr_t)d_dst) & 15) == 0;
  if (vec) {
    const int64_t base = (int64_t)blockIdx.x * blockDim.x * FETCH_UNROLL + threadIdx.x;
    uint4 v[FETCH_UNROLL];
#pragma unroll
    for (int k = 0; k < FETCH_UNROLL; ++k) {
      const int64_t i = base + (int64_t)k * blockDim.x;
      if (i < n16) v[k] = reinterpret_cast<const uint4*>(h_src)[i];
    }
#pragma unroll
    for (int k = 0; k < FETCH_UNROLL; ++k) {
      const int64_t i = base + (int64_t)k * blockDim.x;
      if (i < n16) reinterpret_cast<uint4*>(d_dst)[i] = v[k];
    }
    if (blockIdx.x == 0 && threadIdx.x < (words & 3)) d_dst[n16 * 4 + threadIdx.x] = h_src[n16 * 4 + threadIdx.x];
  } else {
    for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < words; k += (int64_t)gridDim.x * blockDim.x)
      d_dst[k] = h_src[k];
  }
}

// Delivery of the predictions into the pinned (device-mapped) result buffer by a kernel; the last CTA then publishes the
// set's delivery count in *h_flag (system-scope fences: data before flag), which tfr_host_wait_flag polls -- no event, no
// API call on the host's critical path.
__global__ void __launch_bounds__(256) feed_deliver_kernel(const float* __restrict__ d_src, float* __restrict__ h_dst,
                                                           int64_t n, uint32_t* __restrict__ d_sync,
                                                           volatile uint32_t* __restrict__ h_flag) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t n4 = n / 4;
  const bool vec = (((uintptr_t)d_src | (uintptr_t)h_dst) & 15) == 0;
  if (vec) {
    if (i < n4) reinterpret_cast<float4*>(h_dst)[i] = reinterpret_cast<const float4*>(d_src)[i];
    const int64_t t = n4 * 4 + (i - n4);
    if (i >= n4 && t < n) h_dst[t] = d_src[t];
  } else {
    for (int64_t k = i; k < n; k += (int64_t)gridDim.x * blockDim.x) h_dst[k] = d_src[k];
  }
  __threadfence_system();
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned int arrived = atomicAdd(&d_sync[0], 1u);
    if (arrived == gridDim.x - 1) {   // every CTA's stores are fenced and counted
      d_sync[0] = 0u;
      const unsigned int seq = d_sync[1] + 1u;
      d_sync[1] = seq;
      __threadfence_system();
      *h_flag = seq;
    }
  }
}

// H2D copy of a staged set + the sort of its ids, on `side` (eager, or inside a capture: the copy's event is then recorded
// as an external node, for the host thread that repacks h_feed)
static int feed_copy_sort(const tfr_svd_tables* t, tfr_opt_scalars* opt, tfr_feed_set* set, int64_t B, cudaStream_t side,
                          bool capturing, cudaEvent_t before_sort) {
  tfr_svd_step_ws ws;
  int rc = tfr_svd_step_carve(set->workspace, set->workspace_bytes, B, t->dim, &ws);
  if (rc) return rc;
  if (capturing) {
    const int64_t words = 3 * B;
    TFR_PREP(feed_fetch_kernel);
    feed_fetch_kernel<<<(unsigned)((words / 4 + 256 * FETCH_UNROLL - 1) / (256 * FETCH_UNROLL) + 1), 256, 0, side>>>(
        static_cast<const uint32_t*>(set->h_feed), static_cast<uint32_t*>(set->d_feed), words);
    TFR_LAUNCH_CHECK();
    TFR_CUDA(cudaEventRecordWithFlags((cudaEvent_t)set->ev_h2d, side, cudaEventRecordExternal));
  } else {
    TFR_CUDA(cudaMemcpyAsync(set->d_feed, set->h_feed, 12 * (size_t)B, cudaMemcpyHostToDevice, side));
    TFR_CUDA(cudaEventRecord((cudaEvent_t)set->ev_h2d, side));
  }
  if (before_sort) TFR_CUDA(cudaStreamWaitEvent(side, before_sort, 0));
  const int32_t* ids = static_cast<const int32_t*>(set->d_feed);
  // inside the graph: the sort in its barrier-free form (one launch per phase): it runs in whatever room the table pass
  // leaves, and a CTA that has to wait for room holds up nobody
  return dedup_sort_pairs_impl(ids, (int64_t)t->user_num + 1, ws.su_ids, ws.su_pos, ids + B, (int64_t)t->item_num + 1,
                               ws.si_ids, ws.si_pos, B, ws.sort_ws, ws.sort_ws_bytes, opt, side, capturing);
}

extern "C" int tfr_svd_feed_sort(const tfr_svd_tables* t, tfr_opt_scalars* opt, tfr_feed_set* set, int64_t B,
                                 void* side_stream, void* after_event) {
  TFR_CHECK_ARG(t && opt && set && B > 0 && t->dim > 0 && side_stream && set->used && set->staged && !set->sorted);
  TFR_CHECK_ARG(set->h_feed && set->d_feed && set->workspace && set->ev_h2d && set->ev_sorted && set->ev_done);
  cudaStream_t side = (cudaStream_t)side_stream;
  // the step that last used this set's device buffers has finished (device-side wait; a no-op before the first record)
  TFR_CUDA(cudaStreamWaitEvent(side, (cudaEvent_t)set->ev_done, 0));
  const int rc = feed_copy_sort(t, opt, set, B, side, false, (cudaEvent_t)after_event);
  if (rc) return rc;
  TFR_CUDA(cudaEventRecord((cudaEvent_t)set->ev_sorted, side));
  set->staged = 0;
  set->sorted = 1;
  return TFR_OK;
}

extern "C" int tfr_svd_feed_prefetch(const tfr_svd_tables* t, tfr_opt_scalars* opt, tfr_feed_set* set, const void* users_host,
                                     int32_t users_dtype, int64_t users_stride, const void* items_host, int32_t items_dtype,
                                     int64_t items_stride, const void* rates_host, int32_t rates_dtype, int64_t rates_stride,
                                     int64_t B, void* side_stream) {
  TFR_CHECK_ARG(opt);
  int rc = tfr_svd_feed_stage(t, set, users_host, users_dtype, users_stride, items_host, items_dtype, items_stride, rates_host,
                              rates_dtype, rates_stride, B);
  return rc ? rc : tfr_svd_feed_sort(t, opt, set, B, side_stream, nullptr);
}

extern "C" int tfr_svd_feed_step(const tfr_svd_tables* t, tfr_opt_scalars* opt, tfr_feed_set* set, int64_t B, int32_t flags,
                                 int32_t var_mask, int32_t fetch, void* stream, void* copy_stream, tfr_feed_set* next_set,
                                 void* side_stream) {
  TFR_CHECK_ARG(t && opt && set && B > 0 && set->used && set->sorted && set->d_feed && set->d_out && set->ev_pred);
  TFR_CHECK_ARG(fetch >= 0 && fetch <= 2 && (fetch == 0 || (copy_stream && set->h_out && set->ev_d2h)));
  TFR_CHECK_ARG(!next_set || (next_set != set && side_stream));
  cudaStream_t s0 = (cudaStream_t)stream, sc = (cudaStream_t)copy_stream;
  TFR_CUDA(cudaStreamWaitEvent(s0, (cudaEvent_t)set->ev_sorted, 0));
  if (set->copied) TFR_CUDA(cudaStreamWaitEvent(s0, (cudaEvent_t)set->ev_d2h, 0));  // d_out is about to be overwritten
  const int32_t* ids = static_cast<const int32_t*>(set->d_feed);
  const float* rates = reinterpret_cast<const float*>(ids + 2 * B);
  int rc = run_step(t, opt, ids, ids + B, rates, B, set->d_out, set->d_out + B, flags, var_mask, set->workspace,
                    set->workspace_bytes, stream, nullptr, 0, nullptr, true, 1);
  if (rc) return rc;
  // end of forward + segment sums: the table pass starts here
  TFR_CUDA(cudaEventRecord((cudaEvent_t)set->ev_pred, s0));
  if (next_set && next_set->staged && !next_set->sorted &&
      (rc = tfr_svd_feed_sort(t, opt, next_set, B, side_stream, set->ev_pred)))
    return rc;
  if (fetch) {
    // the predictions come from the PRE-update tables (A.7): they go back while the table pass runs
    TFR_CUDA(cudaStreamWaitEvent(sc, (cudaEvent_t)set->ev_pred, 0));
    const size_t off = fetch == 1 ? (size_t)B : 0, cnt = fetch == 1 ? (size_t)B : 2 * (size_t)B;
    TFR_CUDA(cudaMemcpyAsync(set->h_out + off, set->d_out + off, cnt * sizeof(float), cudaMemcpyDeviceToHost, sc));
    TFR_CUDA(cudaEventRecord((cudaEvent_t)set->ev_d2h, sc));
    set->copied = 1;
  }
  if ((rc = run_step(t, opt, ids, ids + B, rates, B, set->d_out, set->d_out + B, flags, var_mask, set->workspace,
                     set->workspace_bytes, stream, nullptr, 0, nullptr, true, 2)))
    return rc;
  TFR_CUDA(cudaEventRecord((cudaEvent_t)set->ev_done, s0));
  return TFR_OK;
}

// The same step as ONE graph: [H2D + id sort of the staged next batch] beside [forward + segment sums -> {copy of the
// predictions, table pass}].  Eager launches on several streams do not run beside the table pass on this platform -- the
// side stream's sort and even the copy engine's D2H only start when the pass has drained (tools/timeline.py eager vs graph,
// profiles/r02_feed_path.md) -- the branches of a graph do.
namespace {
struct CaptureEvents {
  cudaEvent_t e[2] = {nullptr, nullptr};
  ~CaptureEvents() {
    for (cudaEvent_t x : e)
      if (x) cudaEventDestroy(x);
  }
};

int deliver(tfr_feed_set* set, int64_t B, int32_t fetch, cudaStream_t st) {
  const int64_t off = fetch == 1 ? B : 0, cnt = fetch == 1 ? B : 2 * B;
  TFR_PREP(feed_deliver_kernel);
  feed_deliver_kernel<<<(unsigned)((cnt / 4 + 255) / 256 + 1), 256, 0, st>>>(set->d_out + off, set->h_out + off, cnt,
                                                                           set->d_sync, set->h_flag);
  TFR_LAUNCH_CHECK();
  return TFR_OK;
}

int feed_graph_body(const tfr_svd_tables* t, tfr_opt_scalars* opt, tfr_feed_set* set, tfr_feed_set* next_set, int64_t B,
                    int32_t flags, int32_t var_mask, int32_t fetch, bool early_side, cudaStream_t c0, cudaStream_t cs,
                    CaptureEvents& ev) {
  cudaEvent_t e_fwd = ev.e[0], e_sorted = ev.e[1];
  const int32_t* ids = static_cast<const int32_t*>(set->d_feed);
  const float* rates = reinterpret_cast<const float*>(ids + 2 * B);
  int rc;
  // ONE branch of kernels beside the table pass: delivery of the predictions -> fetch of the staged next batch -> its id
  // sort in the barrier-free form.  (Measured, profiles/r02_feed_path.md: the one-launch sort with its grid barrier,
  // released next to the pass, sometimes only got part of its grid resident until the pass drained -- 45 -> 250 us instead
  // of 57 -> 125.)
  // Small tables (early_side): the pass is a few microseconds, the sort is the longest thing in the step -- the fetch + sort
  // branch forks at the very start, beside the forward, and the delivery sits on the step stream in front of the pass.
  const bool side = next_set || (fetch && !early_side);
  if (early_side && next_set) {
    TFR_CUDA(cudaEventRecord(e_fwd, c0));
    TFR_CUDA(cudaStreamWaitEvent(cs, e_fwd, 0));
    if ((rc = feed_copy_sort(t, opt, next_set, B, cs, true, nullptr))) return rc;
  }
  if ((rc = run_step(t, opt, ids, ids + B, rates, B, set->d_out, set->d_out + B, flags, var_mask, set->workspace,
                     set->workspace_bytes, c0, nullptr, 0, nullptr, true, 1)))
    return rc;
  if (early_side) {
    if (fetch && (rc = deliver(set, B, fetch, c0))) return rc;
  } else {
    TFR_CUDA(cudaEventRecord(e_fwd, c0));
    if (side) TFR_CUDA(cudaStreamWaitEvent(cs, e_fwd, 0));
    if (fetch && (rc = deliver(set, B, fetch, cs))) return rc;
    if (next_set && (rc = feed_copy_sort(t, opt, next_set, B, cs, true, nullptr))) return rc;
  }
  if (side) TFR_CUDA(cudaEventRecord(e_sorted, cs));
  if ((rc = run_step(t, opt, ids, ids + B, rates, B, set->d_out, set->d_out + B, flags, var_mask, set->workspace,
                     set->workspace_bytes, c0, nullptr, 0, nullptr, true, 2)))
    return rc;
  if (side) TFR_CUDA(cudaStreamWaitEvent(c0, e_sorted, 0));
  return TFR_OK;
}
}  // namespace

extern "C" int tfr_svd_feed_graph_create(const tfr_svd_tables* t, tfr_opt_scalars* opt, tfr_feed_set* set,
                                         tfr_feed_set* next_set, int64_t B, int32_t flags, int32_t var_mask, int32_t fetch,
                                         int32_t early_side, void* capture_stream, void* capture_side_stream,
                                         void** graph_exec_out) {
  TFR_CHECK_ARG(t && opt && set && B > 0 && t->dim > 0 && graph_exec_out && capture_stream);
  TFR_CHECK_ARG(set->d_feed && set->d_out && set->workspace && fetch >= 0 && fetch <= 2);
  TFR_CHECK_ARG((fetch == 0 && !next_set) || capture_side_stream);
  TFR_CHECK_ARG(fetch == 0 || (set->h_out && set->d_sync && set->h_flag));
  TFR_CHECK_ARG(!next_set || (next_set != set && next_set->h_feed && next_set->d_feed &&
                              next_set->workspace && next_set->ev_h2d));
  CaptureEvents ev;
  for (cudaEvent_t& x : ev.e) TFR_CUDA(cudaEventCreateWithFlags(&x, cudaEventDisableTiming));
  cudaStream_t c0 = (cudaStream_t)capture_stream;
  // relaxed: the feed worker thread may be inside cudaEventSynchronize while this thread captures
  TFR_CUDA(cudaStreamBeginCapture(c0, cudaStreamCaptureModeRelaxed));
  const int rc = feed_graph_body(t, opt, set, next_set, B, flags, var_mask, fetch, early_side != 0, c0,
                                 (cudaStream_t)capture_side_stream, ev);
  cudaGraph_t graph = nullptr;
  const cudaError_t e_end = cudaStreamEndCapture(c0, &graph);
  if (rc) {
    if (graph) cudaGraphDestroy(graph);
    cudaGetLastError();
    return rc;
  }
  if (e_end != cudaSuccess) {
    set_error("cudaStreamEndCapture -> %s", cudaGetErrorString(e_end));
    cudaGetLastError();
    return TFR_ERR_CUDA;
  }
  cudaGraphExec_t exec = nullptr;
  const cudaError_t e_inst = cudaGraphInstantiate(&exec, graph, 0);
  cudaGraphDestroy(graph);
  if (e_inst != cudaSuccess) {
    set_error("cudaGraphInstantiate -> %s", cudaGetErrorString(e_inst));
    cudaGetLastError();
    return TFR_ERR_CUDA;
  }
  *graph_exec_out = (void*)exec;
  return TFR_OK;
}

extern "C" int tfr_svd_feed_graph_launch(void* graph_exec, tfr_feed_set* set, tfr_feed_set* next_set, int32_t fetch,
                                         void* stream) {
  TFR_CHECK_ARG(graph_exec && set && set->used && set->sorted && set->ev_sorted && set->ev_done);
  TFR_CHECK_ARG(!next_set || (next_set != set && next_set->staged && !next_set->sorted));
  cudaStream_t s0 = (cudaStream_t)stream;
  // a sort of this set queued eagerly (the first steps); one inside the previous graph is ordered by the stream itself
  TFR_CUDA(cudaStreamWaitEvent(s0, (cudaEvent_t)set->ev_sorted, 0));
  TFR_CUDA(cudaGraphLaunch((cudaGraphExec_t)graph_exec, s0));
  TFR_CUDA(cudaEventRecord((cudaEvent_t)set->ev_done, s0));
  if (fetch) set->deliver_seq += 1;   // what *h_flag reads once this launch's predictions are on the host
  if (next_set) {
    next_set->staged = 0;
    next_set->sorted = 1;
  }
  return TFR_OK;
}

extern "C" int tfr_host_wait_flag(const void* flag_host, uint32_t at_least, int64_t timeout_us) {
  TFR_CHECK_ARG(flag_host && timeout_us > 0);
  const volatile uint32_t* f = static_cast<const volatile uint32_t*>(flag_host);
  const auto t0 = std::chrono::steady_clock::now();
  for (uint64_t spins = 1; (int32_t)(*f - at_least) < 0; ++spins) {
#if defined(__x86_64__) || defined(__i386__)
    __builtin_ia32_pause();
#endif
    if ((spins & 4095) == 0 &&
        std::chrono::duration_cast<std::chrono::microseconds>(std::chrono::steady_clock::now() - t0).count() > timeout_us) {
      set_error("tfr_host_wait_flag: %u not reached after %lld us (flag = %u)", at_least, (long long)timeout_us, *f);
      return TFR_ERR_CUDA;
    }
  }
  return TFR_OK;
}

extern "C" int tfr_event_synchronize(void* event) {
  TFR_CHECK_ARG(event);
  TFR_CUDA(cudaEventSynchronize((cudaEvent_t)event));
  return TFR_OK;
}

extern "C" int tfr_event_create(void** event_out) {
  TFR_CHECK_ARG(event_out);
  cudaEvent_t ev = nullptr;
  TFR_CUDA(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
  *event_out = (void*)ev;
  return TFR_OK;
}

extern "C" int tfr_event_destroy(void* event) {
  if (event) TFR_CUDA(cudaEventDestroy((cudaEvent_t)event));
  return TFR_OK;
}

// ---- CUDA graphs ------------------------------------------------------------------------------------------
extern "C" int tfr_graph_begin_capture(void* stream) {
  TFR_CUDA(cudaStreamBeginCapture((cudaStream_t)stream, cudaStreamCaptureModeRelaxed));
  return TFR_OK;
}

extern "C" int tfr_graph_end_capture(void* stream, void** graph_exec_out) {
  TFR_CHECK_ARG(graph_exec_out);
  cudaGraph_t graph = nullptr;
  TFR_CUDA(cudaStreamEndCapture((cudaStream_t)stream, &graph));
  cudaGraphExec_t exec = nullptr;
  cudaError_t e = cudaGraphInstantiate(&exec, graph, 0);
  cudaGraphDestroy(graph);
  if (e != cudaSuccess) {
    set_error("cudaGraphInstantiate -> %s", cudaGetErrorString(e));
    return TFR_ERR_CUDA;
  }
  *graph_exec_out = (void*)exec;
  return TFR_OK;
}

extern "C" int tfr_graph_launch(void* graph_exec, void* stream) {
  TFR_CHECK_ARG(graph_exec);
  TFR_CUDA(cudaGraphLaunch((cudaGraphExec_t)graph_exec, (cudaStream_t)stream));
  return TFR_OK;
}

extern "C" int tfr_graph_destroy(void* graph_exec) {
  if (graph_exec) TFR_CUDA(cudaGraphExecDestroy((cudaGraphExec_t)graph_exec));
  return TFR_OK;
}
