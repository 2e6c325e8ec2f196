/*
 * tfrecomm.h -- C ABI of libtfrecomm.so: the B200 (sm_100a) implementation of TF-recomm's
 * matrix-factorization train step.
 *
 * The reference (jilljenn/TF-recomm) has NO FFI/plugin boundary of its own: it is Python that
 * builds a TensorFlow 1.x graph (ops.py) and drives it with sess.run (svd_train_val.py:70-72).
 * The boundary a drop-in must honour is therefore that Python surface (kept by tf-recomm_b200/ops.py,
 * dataio.py, session.py); this C ABI is what sits directly below it and replaces the TensorFlow
 * runtime.  Each entry point cites the reference lines (into /root/reference) whose arithmetic it
 * replaces; "TF:" cites TensorFlow 1.x by file name (SURVEY.md Appendix A).
 *
 * Conventions
 *  - Plain pointers and sizes only. Every pointer is a DEVICE pointer unless its name ends in _host.
 *  - The caller owns all memory (tables, optimizer slots, workspaces); the library never allocates
 *    device memory.  `stream` is a cudaStream_t passed as void*.  All calls are asynchronous on
 *    `stream` and capturable in a CUDA graph (no host sync, no allocation).
 *  - Return 0 on success, negative tfr_status on error; tfr_last_error() gives the message
 *    (thread-local).  There is no CPU fallback anywhere: without a CUDA device every compute entry
 *    point returns TFR_ERR_CUDA.
 *  - ids are int32 row indices; tables are fp32, row-major, contiguous: feat[rows][dim].
 */
#ifndef TFRECOMM_H_
#define TFRECOMM_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TFR_ABI_VERSION 1

typedef enum {
  TFR_OK = 0,
  TFR_ERR_INVALID = -1, /* bad argument (null pointer, negative size, unsupported dim) */
  TFR_ERR_CUDA = -2,    /* a CUDA runtime call failed; see tfr_last_error()            */
  TFR_ERR_WORKSPACE = -3 /* workspace too small                                         */
} tfr_status;

/* Model-variant flags. 0 = README model (README.md:31-39, doc/graph_svd.png): plain dot, squared
 * error, L2 on the gathered embeddings, Adam.  The fork as written is all four bits set. */
enum {
  TFR_ABS_ITEM = 1,        /* ops.py:44     tf.abs(feat_items) in the dot                 */
  TFR_LOSS_SIGMOID_CE = 2, /* ops.py:125-126 summed sigmoid cross-entropy on the logits    */
  TFR_REG_BIAS = 4,        /* ops.py:85-89  L2 on the gathered biases as well              */
  TFR_OPT_SGD = 8,         /* ops.py:145    GradientDescentOptimizer (scatter_sub, no Adam) */
  /* host-side only (never stored in tfr_opt_scalars): the workspace already holds this batch's sorted
   * (feature id, position) pairs -- a fixed CSR batch that is stepped every epoch is sorted once */
  TFR_FM_PRESORTED = 256
};
/* var_list bits (ops.py:118,147-149; adaptive_test.py:28 trains the user side only) */
enum { TFR_VAR_MU = 1, TFR_VAR_UB = 2, TFR_VAR_UF = 4, TFR_VAR_IB = 8, TFR_VAR_IF = 16, TFR_VAR_ALL = 31 };

const char* tfr_last_error(void);
int tfr_abi_version(void);
/* Number of SMs of the current device (148 on B200), or negative status. */
int tfr_device_sm_count(void);
/* Tuning knobs -- the ONLY process-wide state of the library (everything else is caller-owned).  A knob's value is what
 * tfr_tune_set gave it, else the environment variable TFR_<NAME> at first use, else its default.  Names (csrc/capi.cu):
 * SMEM_CARVEOUT, SEG_TILE, SEG_MAX_UNITS, PASS_RING (1 = interleaved tables take the TMA-bulk ring pass, 0 = the
 * LDG/STG pass), RING_STAGES, RING_STAGE_KB, RING_THREADS, RING_L2_HINT, STREAM_THREADS, STREAM_CTAS_PER_SM, ...
 * What a knob may change:
 *  - bit for bit the same results: SMEM_CARVEOUT, TILES_CARVEOUT, STREAM_LD, STREAM_ST, STREAM_CTAS_PER_SM,
 *    STREAM_UNROLL, STREAM_THREADS, STREAM_DYNAMIC, TL_EVERY_CTA, PDL, SORT_SPLIT, PASS_RING, RING_STAGES,
 *    RING_STAGE_KB, RING_THREADS, RING_L2_HINT, RING_CTAS_PER_SM, RING_SLOT_MODE 0..2, RANK_CHUNK;
 *  - the fp32 rounding of the training step, within the oracle's 1e-5 bar: SEG_TILE (where runs of equal ids are
 *    regrouped into partial sums; its default depends on the batch size, the dim and the device's SM count) and
 *    SEG_MAX_UNITS (lanes per row, hence the order of the fused forward's dot products, and the default tile);
 *  - the float64 summation order of the ALS half-sweep's heavy rows, which keeps parity with the exact solution, not bits:
 *    ALS_CHUNK (ratings per Gram chunk; read once, by tfr_als_chunk, when a plan is built);
 *  - results, on purpose (debug and measurement only): STREAM_COPY_ONLY, RING_SLOT_MODE 3, AP_STAGES, RANK_STAGES. */
int tfr_tune_set(const char* name, int32_t value);
int tfr_tune_get(const char* name, int32_t* value);

/* ------------------------------------------------------------------------------------------
 * Optimizer scalars kept in DEVICE memory so that a captured graph can be replayed every step.
 * Replaces the non-table state of TF AdamOptimizer (TF: adam.py _create_slots/_prepare/_finish):
 * beta1_power/beta2_power advance by one fp32 multiply per step AFTER the applies; lr_t is
 * recomputed at the start of each step as lr*sqrt(1-beta2_power)/(1-beta1_power) (A.4).
 * The caller allocates sizeof(tfr_opt_scalars) device bytes and fills it with tfr_opt_init.
 * ---------------------------------------------------------------------------------------- */
typedef struct {
  float lr, reg, beta1, beta2, eps;
  float beta1_power, beta2_power, lr_t;
  float one_minus_beta1, one_minus_beta2; /* fp32(1)-fp32(beta), as TF computes them */
  int32_t flags, var_mask;
  int64_t global_step;   /* svd_train_val.py:48 tf.train.get_or_create_global_step()        */
  int64_t batch_cursor;  /* next batch index into a device-resident index stream (see below) */
  int64_t prefetch_cursor; /* next batch the ASSEMBLE-AHEAD path draws: advanced only by tfr_svd_prefetch_batch's own
                              kernels (side stream), never by the step -- the step's last CTA advances batch_cursor
                              while the side stream may be running, so the two must not share a counter */
  double se_sum;         /* sum over the last step's batch of (rate - infer)^2, float64 like
                            svd_train_val.py:104 (np.power(train_rates - train_infer, 2))   */
  float g_mu;            /* last step's d cost / d bias_global (sum_b e_b)                   */
  uint32_t ticket;       /* CTA arrival counter of the table pass (its last CTA ends the step); 0 between steps */
  double* se_ring;       /* optional device ring: se_ring[global_step % se_ring_len] = se_sum, so the
                            driver's trailing-window train RMSE (svd_train_val.py:59,104,108) needs one
                            read per epoch instead of one per step                            */
  int64_t se_ring_len;
  uint32_t chunk_ctr[4]; /* per-table chunk counters of the table pass's dynamic scheduling; 0 between steps */
  uint64_t* timeline;    /* optional debug buffer [2][TFR_TL_SLOTS] of %globaltimer ns: earliest block entry and
                            latest warp exit of every kernel of the step (there is no nsys on the box); null = off */
} tfr_opt_scalars;
#define TFR_TL_SLOTS 16
enum { TFR_TL_ASSEMBLE = 0, TFR_TL_FWD = 1, TFR_TL_SORT = 2, TFR_TL_TILES = 3, TFR_TL_FIXUP = 4, TFR_TL_STREAM_UF = 5,
       TFR_TL_STREAM_IF = 6, TFR_TL_STREAM_UB = 7, TFR_TL_STREAM_IB = 8, TFR_TL_TOUCHED_U = 9, TFR_TL_TOUCHED_I = 10,
       TFR_TL_FINISH = 11 };

int tfr_opt_init(tfr_opt_scalars* opt_dev, float lr, float reg, float beta1, float beta2, float eps,
                 int32_t flags, int32_t var_mask, void* stream);
int tfr_opt_set_se_ring(tfr_opt_scalars* opt_dev, double* se_ring, int64_t se_ring_len, void* stream);
int tfr_opt_set_timeline(tfr_opt_scalars* opt_dev, uint64_t* timeline, void* stream);

/* ------------------------------------------------------------------------------------------
 * The five variables of ops.py:8-12,29-32 and their Adam slots (TF: adam.py zeros_like slots).
 * ---------------------------------------------------------------------------------------- */
typedef struct {
  int32_t user_num, item_num, dim;
  /* floats between consecutive rows of user_feat / item_feat AND of their Adam slots; 0 = dim (plain [rows][dim]
   * arrays).  3*dim with m_uf = user_feat + dim, v_uf = user_feat + 2*dim (likewise for items) is the INTERLEAVED
   * layout [rows][var | m | v][dim]: the table-wide Adam pass then reads and writes ONE stream instead of three
   * (measured on B200: 6.0 TB/s against 5.3 TB/s for three separate arrays), and a gathered row is still dim
   * contiguous floats. */
  int32_t feat_stride;
  float* mu;        /* bias_global   []      ops.py:8  */
  float* user_bias; /* user_bias     [U]     ops.py:9  */
  float* item_bias; /* item_bias     [I]     ops.py:11 */
  float* user_feat; /* user_features [U,dim] ops.py:29 */
  float* item_feat; /* item_features [I,dim] ops.py:31 */
  float *m_mu, *v_mu, *m_ub, *v_ub, *m_ib, *v_ib, *m_uf, *v_uf, *m_if, *v_if; /* null in SGD mode */
  /* row -> slot maps, initialised to -1 by the caller: (step stamp << 32 | k), stamp = low 32 bits of
   * opt->global_step when the entry was written, k = sorted index of the run head whose gsum[k] is the row's summed
   * gradient.  An entry counts only in the step that wrote it, so the maps are never reset (refill them with -1 if
   * global_step is ever set backwards, e.g. when restoring a checkpoint). */
  int64_t* user_slot; /* [U] */
  int64_t* item_slot; /* [I] */
  /* Row-sharded mode (tables hold only this rank's rows, id mod G == rank; SURVEY 8e).  When non-null, the
   * batch's gathered rows by BATCH POSITION ([B,dim] / [B], exchanged between ranks) replace the by-id gathers
   * of the forward and of the partner rows in the backward; the users/items arrays given to the step are then
   * LOCAL row indices, with the value user_num / item_num marking occurrences owned by another rank. */
  const float *g_user_feat, *g_item_feat, *g_user_bias, *g_item_bias;
  int64_t g_stride; /* floats between consecutive rows of g_user_feat / g_item_feat; 0 = dim */
} tfr_svd_tables;

/* ---- forward only: replaces sess.run([logits, infer]) at svd_train_val.py:121-122 -----------
 * gathers ops.py:13-14,37-38; logits = ((sum_k u*v' + mu) + b_u) + b_i ops.py:44-47;
 * head ops.py:76-78 (fork: infer = round(sigmoid(logits)); README: infer = logits).
 * logits / infer may be null.  B = 0 is a no-op. */
int tfr_svd_forward(const tfr_svd_tables* t, const int32_t* users, const int32_t* items, int64_t B,
                    int32_t flags, float* logits, float* infer, void* stream);

/* ---- batch assembly: replaces dataio.ShuffleIterator.next (dataio.py:114-117) on the device ---
 * cols_* are the training columns resident in HBM; row_index holds the pre-drawn MT19937
 * `np.random.randint(0, N, B)` stream for many steps (generated on the host so that it is the
 * reference's stream).  Batch k = rows row_index[k*B .. k*B+B).  batch_index >= 0 selects that batch;
 * -1 = the batch at opt->batch_cursor (this step's batch; call it on the step's own stream);
 * -2 = the batch at opt->prefetch_cursor (assemble-ahead on a side stream; tfr_svd_prefetch_batch then advances
 * that cursor with a kernel of its own, so nothing the concurrent step writes is read);
 * -3 (tfr_svd_prefetch_batch only) = the batch at batch_cursor, and prefetch_cursor := batch_cursor + 1: primes the
 * assemble-ahead path, on the step's own stream. */
int tfr_svd_batch_assemble(const tfr_svd_tables* t, tfr_opt_scalars* opt, const int32_t* col_user,
                           const int32_t* col_item, const float* col_rate, const int64_t* row_index,
                           int64_t batch_index, int64_t B, int32_t* users, int32_t* items, float* rates,
                           void* stream);

/* ---- dedup: replaces TF optimizer.py::_deduplicate_indexed_slices (tf.unique + unsorted_segment_sum)
 * Stable LSD radix sort of (id, position): sorted_ids ascending, sorted_pos = original positions,
 * ascending inside each run of equal ids (so a run lists one id's occurrences in BATCH ORDER).
 * Two independent problems (user ids, item ids) are sorted by ONE cooperative launch.
 * n may be 0.  max_id_* = number of rows of the table (exclusive upper bound of ids). */
int64_t tfr_dedup_workspace_bytes(int64_t n);
int tfr_dedup_sort_pairs(const int32_t* ids_a, int64_t max_id_a, int32_t* sorted_ids_a, int32_t* sorted_pos_a,
                         const int32_t* ids_b, int64_t max_id_b, int32_t* sorted_ids_b, int32_t* sorted_pos_b,
                         int64_t n, void* workspace, int64_t workspace_bytes, void* stream);
/* same, with the step's scalars so that the launch shows up in opt->timeline */
int tfr_dedup_sort_pairs_tl(const int32_t* ids_a, int64_t max_id_a, int32_t* sorted_ids_a, int32_t* sorted_pos_a,
                            const int32_t* ids_b, int64_t max_id_b, int32_t* sorted_ids_b, int32_t* sorted_pos_b,
                            int64_t n, void* workspace, int64_t workspace_bytes, const tfr_opt_scalars* opt,
                            void* stream);
/* tf.unique's own outputs from the sorted pairs (parity/debug API, not on the hot step):
 * uniq[0..n_uniq) in order of FIRST OCCURRENCE, idx[b] = position of ids[b] in uniq, *n_uniq_dev.
 * scratch: n int32. */
int tfr_unique_first_occurrence(const int32_t* sorted_ids, const int32_t* sorted_pos, int64_t n,
                                int32_t* uniq, int32_t* idx, int32_t* n_uniq_dev, int32_t* scratch,
                                void* stream);

/* ---- full train step: replaces sess.run([train_op, logits, infer]) at svd_train_val.py:70-72 ----
 * forward + d cost/d logits (ops.py:124-126) -> dedup -> per-row summed gradients (loss + reg*L2 on
 * the gathered rows, ops.py:81-89,140) -> TF sparse Adam over the WHOLE tables (A.4) / dense Adam on
 * bias_global (A.5), or scatter_sub SGD (ops.py:145).  logits/infer come from the PRE-update tables
 * (A.7).  users/items/rates are the assembled batch (device).  Advances opt->global_step,
 * beta powers and batch_cursor.  Launches: [id sort] -> forward fused into the segment sums -> fix-up of runs that
 * cross tiles -> ONE Adam pass whose last CTA ends the step. */
int64_t tfr_svd_step_workspace_bytes(int64_t B, int32_t dim);
/* Sets batch_cursor and prefetch_cursor (both to k): the next step / the next assemble-ahead draw batch k. */
int tfr_opt_set_cursor(tfr_opt_scalars* opt_dev, int64_t k, void* stream);
/* The id-only half of a step, for the NEXT batch, to be run on a side stream under the current step's table pass:
 * tfr_svd_batch_assemble(batch_index) into users/items/rates + tfr_dedup_sort_pairs into `workspace`'s sorted-pair
 * buffers.  tfr_svd_train_step_presorted then runs the rest (forward -> segment sums -> Adam pass -> finish) on
 * a workspace prepared that way. */
int tfr_svd_prefetch_batch(const tfr_svd_tables* t, tfr_opt_scalars* opt, const int32_t* col_user,
                           const int32_t* col_item, const float* col_rate, const int64_t* row_index,
                           int64_t batch_index, int64_t B, int32_t* users, int32_t* items, float* rates,
                           void* workspace, int64_t workspace_bytes, void* stream);
/* phases: 1 = forward + segment sums (read the tables), 2 = Adam pass / SGD slice + finish (write them), 3 = both.
 * A caller that prefetches the next batch forks its side stream between the two phases, so that the id-only work
 * runs under the bandwidth-bound pass instead of beside the latency-bound gathers. */
int tfr_svd_train_step_presorted(const tfr_svd_tables* t, tfr_opt_scalars* opt, const int32_t* users,
                                 const int32_t* items, const float* rates, int64_t B, float* logits, float* infer,
                                 int32_t flags, int32_t var_mask, int32_t phases, void* workspace,
                                 int64_t workspace_bytes, void* stream);
/* flags / var_mask must equal what tfr_opt_init was given (the host copy selects the launches, the
 * device copy drives the kernels).  side_streams (optional; n_side = 0..1): [0] runs the id sort next to the
 * forward.  Fork/join is by the two caller-owned events fork_join_events[0..1] (cudaEvent_t, created on the step's
 * device, e.g. by tfr_event_create; required when n_side > 0 -- the library keeps no events of its own), so the whole
 * step is still capturable as one graph from `stream`. */
int tfr_svd_train_step(const tfr_svd_tables* t, tfr_opt_scalars* opt, const int32_t* users,
                       const int32_t* items, const float* rates, int64_t B, float* logits, float* infer,
                       int32_t flags, int32_t var_mask, void* workspace, int64_t workspace_bytes, void* stream,
                       void* const* side_streams, int32_t n_side, void* const* fork_join_events);
/* cudaEvent_t (timing disabled) on the current device, for callers without CUDA bindings of their own. */
int tfr_event_create(void** event_out);
int tfr_event_destroy(void* event);

/* Pieces of the step, exported for parity tests and for callers that schedule them themselves. */
typedef struct { /* carved out of the step workspace by tfr_svd_step_carve */
  float* err;           /* [B] d cost / d logits                                     */
  float* partials;      /* [TFR_MAX_PARTIALS] per-CTA sums of err                    */
  double* se_partials;  /* [TFR_MAX_PARTIALS] per-CTA sums of (rate-infer)^2         */
  int32_t *su_ids, *su_pos, *si_ids, *si_pos; /* sorted (id,pos) for users / items   */
  float *gsum_uf, *gsum_if; /* [B,dim] summed gradient of the run whose head is at sorted index k */
  float *gsum_ub, *gsum_ib; /* [B]                                                  */
  float *cont_uf, *cont_if, *tail_uf, *tail_if; /* [n_tiles,dim] cross-tile partial sums */
  float *cont_ub, *cont_ib, *tail_ub, *tail_ib; /* [n_tiles]                          */
  uint8_t *kind_u, *kind_i;                     /* [n_tiles] tile classes for the fix-up */
  int32_t *fix_list_u, *fix_list_i;             /* [n_tiles] tiles whose last run goes on into later tiles (work list) */
  uint32_t* fix_count;  /* [4] list lengths (users, items), arrival ticket; lives in the first 256 bytes of sort_ws,
                           which every id sort zeroes */
  void* sort_ws; int64_t sort_ws_bytes;
  int32_t tile, n_tiles;
} tfr_svd_step_ws;
#define TFR_MAX_PARTIALS 1024
int tfr_svd_step_carve(void* workspace, int64_t workspace_bytes, int64_t B, int32_t dim, tfr_svd_step_ws* out);
/* forward + error: writes logits, infer, ws.err, partial sums (deterministic two-stage reduction). */
int tfr_svd_fwd_err(const tfr_svd_tables* t, const tfr_opt_scalars* opt, const int32_t* users,
                    const int32_t* items, const float* rates, int64_t B, float* logits, float* infer,
                    const tfr_svd_step_ws* ws, void* stream);
/* forward + d cost/d logits + segment sums in ONE launch pair (tiles + fix-up): each side recomputes the logit from
 * the rows it gathers for the gradient anyway.  Writes logits / infer (optional) and tfr_svd_fused_n_partials(dim, B)
 * partials for tfr_svd_finish_step; ws->err is not written.  Not for row-sharded tables (g_* set). */
int tfr_svd_fwd_segment_grads(const tfr_svd_tables* t, const tfr_opt_scalars* opt, const int32_t* users,
                              const int32_t* items, const float* rates, int64_t B, float* logits, float* infer,
                              int32_t flags, const tfr_svd_step_ws* ws, void* stream);
int tfr_svd_fused_n_partials(int32_t dim, int64_t B);
/* recomputes lr_t from the beta powers (after restoring a checkpoint; a step leaves the next step's lr_t behind) */
int tfr_svd_begin_step(tfr_opt_scalars* opt, void* stream);
/* ordered segment sums of the per-occurrence gradients (never materialised): for every run of equal
 * ids in the sorted pairs, gsum[head k] = sum in batch order of (e_b*partner_row + reg*own_row). */
int tfr_svd_segment_grads(const tfr_svd_tables* t, const tfr_opt_scalars* opt, const int32_t* users,
                          const int32_t* items, int64_t B, const tfr_svd_step_ws* ws, void* stream);
/* TF sparse Adam (A.4) as ONE streaming pass over every table, all tables in ONE launch: each parameter is
 * read and written exactly once per step (24 B/param), in address order.  A row that is in this step's slice
 * (slot[row] = k >= 0) takes its summed gradient from gsum[k]; every other row gets the pure decay + step.
 * slot may be null (no row has a gradient). */
typedef struct {
  float *var, *m, *v;  /* [rows*width], 16-byte aligned */
  int64_t rows;
  int32_t width;
  const int64_t* slot; /* [rows] row -> (stamp << 32 | run-head index into gsum); counts if stamp == step */
  const float* gsum;   /* [n, width] */
  int64_t stride;      /* floats between consecutive rows of var (and of m, of v); 0 = width */
} tfr_adam_table;
int tfr_adam_stream_multi(const tfr_adam_table* tables, int32_t n_tables /* 1..4 */, const tfr_opt_scalars* opt,
                          int32_t tl_slot, void* stream);
/* The slice rows alone: var/m/v[sorted_ids[k]] for every run head k with the summed gradient gsum[k]; feature
 * rows and bias entries of both tables in ONE launch.  Used for SGD (ops.py:145: var -= gsum, no table pass)
 * and by callers that schedule the slice separately. */
typedef struct {
  float *var, *m, *v;        /* feature table [rows, width]; null = not in var_list          */
  float *bvar, *bm, *bv;     /* bias table [rows] sharing the row ids; null = not in var_list  */
  const int32_t* sorted_ids; /* [n]                                                           */
  const float* gsum;         /* [n, width] valid at run heads                                  */
  const float* bgsum;        /* [n]                                                            */
  int64_t stride;            /* floats between consecutive rows of var / m / v; 0 = width      */
} tfr_slice_update;
int tfr_adam_slice_multi(const tfr_slice_update* sides, int32_t n_sides /* 1..2 */, int32_t width, int64_t n,
                         const tfr_opt_scalars* opt, int32_t sgd, int32_t tl_slot, void* stream);
int tfr_adam_touched(float* var, float* m, float* v, int32_t width, const int32_t* sorted_ids, int64_t n,
                     const float* gsum, const tfr_opt_scalars* opt, void* stream);
int tfr_sgd_apply(float* var, int32_t width, const int32_t* sorted_ids, int64_t n, const float* gsum,
                  void* stream);
/* end of step as a launch of its own: dense Adam/SGD on bias_global from the err partials (A.5), advance beta powers
 * and counters (TF: adam.py::_finish).  tfr_svd_train_step folds this into the Adam pass.  users/items/B: unused. */
int tfr_svd_finish_step(const tfr_svd_tables* t, tfr_opt_scalars* opt, const int32_t* users,
                        const int32_t* items, int64_t B, const tfr_svd_step_ws* ws, int32_t n_partials,
                        void* stream);

/* ---- row-sharded tables: the owner's half of the id -> row exchange (SURVEY 8e) ------------------------------
 * For every batch position b: if ids[b] mod n_ranks == rank, copy the local row ids[b] / n_ranks (and its bias)
 * to out_feat[b] / out_bias[b] and set local_keys[b] = ids[b] / n_ranks; otherwise write zeros and
 * local_keys[b] = rows_local (the "not mine" mark).  Summing out_* over ranks (NCCL all-reduce, exact: one
 * non-zero term per element) gives every rank the batch's gathered rows. */
int tfr_shard_gather_rows(const float* feat_local, const float* bias_local, int64_t rows_local, int32_t dim,
                          int64_t feat_stride /* floats between rows of feat_local; 0 = dim */, const int32_t* ids,
                          int64_t B, int32_t n_ranks, int32_t rank, float* out_feat, float* out_bias,
                          int32_t* local_keys, void* stream);

/* ---- row-sharded tables, the all-to-all exchange north_star names (ids -> rows back -> gradient records to the owners) ----
 * Per step every rank holds a slice of the global batch (contiguous in global batch order).  Records are dim + 4 floats:
 * [row | bias or e | pad].  The NCCL all-to-alls between these calls are the caller's (torch.distributed).
 *  tfr_shard_bucket: the slice's ids bucketed by owner (id mod n_ranks), stably -> counts [2 * n_ranks] (users to rank g,
 *    then items to rank g), send_ids [2n] = local row ids (id / n_ranks) in the combined layout [dst 0: users | items]
 *    [dst 1: ...], slot_u / slot_i [n] = index of occurrence p's user / item entry in that layout.
 *  tfr_shard_gather_records: owner side -- the rows asked for (recv_ids in the combined layout by SOURCE rank, the per-
 *    source counts cnt_u_host / cnt_i_host on the host) packed as records.
 *  tfr_shard_fwd_records: requester side -- forward (ops.py:44-47) + d cost/d logits (ops.py:124-126) on the slice from
 *    the records that came back; for every occurrence one outgoing record per table, at the same index: [PARTNER row | e].
 *    logits / infer [n] of the slice; sums2 (device, 2 doubles) = this rank's [sum e, sum (rate - infer)^2], to be
 *    all-reduced (sum) over the ranks.
 *  tfr_shard_owner_prepare: owner side -- sort keys of both tables over the received records (the other table's entries
 *    get the "not mine" mark users_local / items_local), err [total] by arrival position, and the all-reduced sums as
 *    the fp32 / float64 scalars the step's finish takes.
 *  tfr_svd_train_step_gathered: the single-GPU step from the sort on, on tables with g_* set (partner rows by arrival
 *    position, stride g_stride) and ws.err prefilled: stable sort, ordered segment sums, ONE Adam pass, finish.
 *    Arrival position ascends with (source rank, position in its slice) = global batch order. */
int64_t tfr_shard_bucket_workspace_bytes(int64_t n);
int tfr_shard_bucket(const int32_t* users, const int32_t* items, int64_t n, int32_t n_ranks, int32_t* counts,
                     int32_t* send_ids, int32_t* slot_u, int32_t* slot_i, void* workspace, int64_t workspace_bytes,
                     void* stream);
int tfr_shard_gather_records(const tfr_svd_tables* t, const int32_t* recv_ids, const int32_t* cnt_u_host,
                             const int32_t* cnt_i_host, int32_t n_ranks, float* records, void* stream);
int tfr_shard_fwd_records(const tfr_svd_tables* t, const tfr_opt_scalars* opt, const float* records_in,
                          const int32_t* slot_u, const int32_t* slot_i, const float* rates, int64_t n, float* records_out,
                          float* logits, float* infer, float* partials /* [TFR_MAX_PARTIALS] scratch */,
                          double* se_partials /* [TFR_MAX_PARTIALS] scratch */, double* sums2, void* stream);
int tfr_shard_owner_prepare(const int32_t* recv_ids, const float* records, const int32_t* cnt_u_host,
                            const int32_t* cnt_i_host, int32_t n_ranks, int32_t dim, int64_t users_local, int64_t items_local,
                            int32_t* keys_u, int32_t* keys_i, float* err, const double* sums2_allreduced, float* sum_err,
                            double* sum_se, void* stream);
int tfr_svd_train_step_gathered(const tfr_svd_tables* t, tfr_opt_scalars* opt, const int32_t* keys_u, const int32_t* keys_i,
                                int64_t n, int32_t flags, int32_t var_mask, const float* sum_err, const double* sum_se,
                                void* workspace, int64_t workspace_bytes, void* stream);

/* ---- FM forward: replaces forward.py:21-22 `fma` ---------------------------------------------
 * yhat[r] = w0 + sum_i W_i x_i + 0.5 * sum_f ((sum_i V_if x_i)^2 - sum_i V_if^2 x_i^2) on CSR rows
 * (indptr int64 [n+1], indices int32, data fp32).  sums (optional) receives sum_i V_if x_i [n,dim].
 * dim is 1..512; any other dim is TFR_ERR_INVALID. */
int tfr_fm_forward(int64_t n_rows, const int64_t* indptr, const int32_t* indices, const float* data,
                   const float* w0, const float* W, const float* V, int32_t dim, float* yhat, float* sums,
                   void* stream);

/* ---- FM train step (BASELINE configs[2]): the SVD step's structure on CSR rows -- forward (sums kept), d cost/d yhat
 * (squared error, or sigmoid-CE with TFR_LOSS_SIGMOID_CE), tf.unique-style dedup of the batch's feature ids, ordered
 * segment sums of the per-non-zero gradients  g_V = e*(x*(sum - V*x)) + reg*V,  g_W = e*x (+ reg*W with TFR_REG_BIAS),
 * ONE TF-Adam pass over V and W (or SGD), dense update of w0.  The reference trains its FM with libFM's MCMC sampler
 * (fm.py:104-110,154-155: external binary, out of scope); this is the step north_star asks for instead.
 * indptr[0] must be 0 (a batch is its own CSR matrix).  Caller-allocated scratch: rowof [nnz] (filled by the step:
 * CSR row of every non-zero), sums [n_rows, dim], err [n_rows]; workspace: tfr_svd_step_workspace_bytes(nnz, dim).
 * yhat comes from the PRE-update tables.  Rows without non-zeros are allowed (yhat = w0).  t->dim is 1..512; any
 * other dim is TFR_ERR_INVALID before anything is launched. */
typedef struct {
  int32_t n_feat, dim;
  float *w0, *W, *V;                         /* [1], [n_feat], [n_feat, dim] */
  float *m_w0, *v_w0, *m_W, *v_W, *m_V, *v_V; /* Adam slots; null in SGD mode  */
  int64_t* slot;                             /* [n_feat], as tfr_svd_tables' maps */
} tfr_fm_tables;
int tfr_fm_segment_grads(const float* V, const float* W, int64_t* slot, int32_t n_feat, int32_t dim,
                         const tfr_opt_scalars* opt, const float* sums, const float* err, const float* xval,
                         const int32_t* rowof, int64_t nnz, const tfr_svd_step_ws* ws, void* stream);
int tfr_fm_train_step(const tfr_fm_tables* t, tfr_opt_scalars* opt, int64_t n_rows, const int64_t* indptr,
                      const int32_t* indices, const float* data, int32_t* rowof, int64_t nnz, const float* y,
                      float* yhat, float* sums, float* err, int32_t flags, void* workspace, int64_t workspace_bytes,
                      void* stream);

/* ---- all-pairs scoring: replaces als3.py:110-113  M = U.V^T + W_user[:,None] + W_work[None,:] + bias -----------
 * (and the per-user ranking of forward.py:47-61 for k = 1).  Outputs, each optional: scores [n_users, n_items]
 * (row-major), best_score [n_users] / best_item [n_users] = the highest-scoring item of every user (lowest index on
 * ties), computed in the GEMM epilogue so that the score matrix need not exist.  use_tensor_cores = 1: tcgen05
 * (kind::tf32, TMEM accumulator, TMA loads), dim % 32 == 0 and dim <= 128; = 0: exact-fp32 CUDA-core kernel, any dim
 * (needs tfr_allpairs_workspace_bytes of workspace when best_* are requested). */
int64_t tfr_allpairs_workspace_bytes(int64_t n_users, int64_t n_items, int32_t dim, int32_t use_tensor_cores);
int tfr_allpairs(const float* user_feat, const float* item_feat, const float* user_bias, const float* item_bias,
                 const float* mu, int64_t n_users, int64_t n_items, int32_t dim,
                 int64_t user_stride, int64_t item_stride /* floats between rows; 0 = dim */, int32_t use_tensor_cores,
                 float* scores, float* best_score, int32_t* best_item, void* workspace, int64_t workspace_bytes,
                 void* stream);

/* ---- all-pairs CONSUMERS in the GEMM epilogue (tcgen05 path: dim % 32 == 0, dim <= 128): the score matrix is never written.
 *  k > 0: per-user ranking over ALL items -- forward.py:47-61 get_ranking (score every item for a user, sort, keep the
 *    first 50) for every user at once.  The tensor cores (tf32 operands) keep each row's n_cand >= k best candidates
 *    (n_cand <= 128; 64 for k = 50 is plenty); the candidates are then rescored in float64 -- the reference's own
 *    precision, als3.py:112 is numpy float64 -- ranked (score descending, lowest item index on ties) and CERTIFIED: the
 *    first k are the exact top-k of the whole row if the k-th exact score exceeds the worst candidate's tensor-core score
 *    by more than a bound on the tensor-core score's error, (2^-9 + dim * 2^-22) * ||u|| * max||v|| + 2^-22 * (||u|| *
 *    max||v|| + |b_u| + max|fl(b_i + mu)|) (tf32 operands, fp32 accumulation and bias additions).  n_cand below 11 keeps
 *    11 candidates (the workspace query accounts for them).  Rows that cannot be certified (near-ties) are redone over
 *    all items in float64 on CUDA cores.  Result: topk_val (float64) / topk_idx [n_users, k], identical to ranking the
 *    float64 score matrix; *n_uncertified = how many rows took the exact path.  Missing ranks (k > n_items): (-inf, -1).
 *  obs_indptr != null: the squared error on the OBSERVED pairs, als3.py:110-120,139-143 (predict = M[user_ids, work_ids],
 *    compute_rmse): pairs as CSR by user (obs_indptr int64 [n_users + 1], obs_item ascending inside a user, obs_rate);
 *    row_se[u] = sum over u's pairs of (score - rating)^2 in float64, scores as the tensor cores produce them (tf32
 *    operands: relative error <= 2^-9 on the dot product; tfr_svd_forward on the pairs is the exact alternative).
 * Both consumers can be requested in one sweep.  workspace: tfr_allpairs_topk_workspace_bytes (k > 0 only). */
int64_t tfr_allpairs_topk_workspace_bytes(int64_t n_users, int64_t n_items, int32_t k, int32_t n_cand);
int tfr_allpairs_consume(const float* user_feat, const float* item_feat, const float* user_bias, const float* item_bias,
                         const float* mu, int64_t n_users, int64_t n_items, int32_t dim, int64_t user_stride,
                         int64_t item_stride, int32_t k, int32_t n_cand, double* topk_val, int32_t* topk_idx,
                         int32_t* n_uncertified, const int64_t* obs_indptr, const int32_t* obs_item, const float* obs_rate,
                         double* row_se, void* workspace, int64_t workspace_bytes, void* stream);
/* The same top-k ranking over the items each user has NOT already rated: excl_indptr int64 [n_users + 1] / excl_item int32
 * list, per user, the item ids that must never be returned (ascending inside a user, duplicates allowed; excl_indptr = null:
 * nothing excluded, the result of tfr_allpairs_consume).  The tensor-core sweep skips them when it keeps candidates and the
 * certificate is over the rankable items: a user ranks min(k, rankable_u) items, rankable_u = n_items - (distinct excluded
 * ids of u), the ranks past that are (-inf, -1) (a user with every item excluded: all (-inf, -1), certified).  Any dim <=
 * 512: a dim the tcgen05 sweep cannot take (dim % 32 != 0 or dim > 128) sends EVERY row through the exact float64 path
 * (*n_uncertified = n_users), O(n_users * n_items * (dim + k)) on CUDA cores -- meant for ML-1M-sized tables.
 * workspace: tfr_allpairs_topk_workspace_bytes. */
int tfr_allpairs_rank_excluding(const float* user_feat, const float* item_feat, const float* user_bias,
                                const float* item_bias, const float* mu, int64_t n_users, int64_t n_items, int32_t dim,
                                int64_t user_stride, int64_t item_stride, int32_t k, int32_t n_cand,
                                const int64_t* excl_indptr, const int32_t* excl_item, double* topk_val, int32_t* topk_idx,
                                int32_t* n_uncertified, void* workspace, int64_t workspace_bytes, void* stream);

/* ---- top-k ranking for a batch of QUERY users: forward.py:47-61 get_ranking for the users asked about -------------------
 * Row q of topk_val (float64) / topk_idx [n_queries, k] is the ranking of user query_users[q], identical in ids and bits to
 * that user's row of tfr_allpairs_rank_excluding with the same tables, k and exclusion list:
 *  - score = ((acc + (double)b_u) + (double)b_i) + (double)mu, acc = sum over d = 0 .. dim-1, in that order from 0.0, of
 *    (double)u[d] * (double)v[d]; flags & TFR_ABS_ITEM: v = |v| (the fork model's u.|v|; no other flag changes the score);
 *  - score descending, lowest item id on ties; excluded items are never returned; a user with fewer than k rankable items
 *    gets (-inf, -1) past the last one.
 * excl_indptr int64 [n_users + 1] / excl_item: the exclusion CSR indexed by USER ID (not by query; ascending inside a user,
 * duplicates allowed), e.g. the training pairs built once; null = nothing excluded.  query_users (device) may repeat and
 * come in any order; an id outside [0, n_users) gives a row of (-inf, -1) and is never read through.  n_queries = 0 is a
 * no-op.  1 <= dim <= 512, 1 <= k <= 1024, n_items < 2^31, else TFR_ERR_INVALID before any CUDA call.
 * Float64 on CUDA cores: O(n_queries * n_items * dim), no tensor-core candidates.  The item axis is split into chunks
 * (knob RANK_CHUNK, items per chunk) that are scored and selected in parallel, then merged per query: any chunking gives the
 * same result.  workspace: tfr_rank_users_workspace_bytes (a function of its arguments only; needs no device). */
int64_t tfr_rank_users_workspace_bytes(int64_t n_queries, int64_t n_items, int32_t k);
int tfr_rank_users(const float* user_feat, const float* item_feat, const float* user_bias, const float* item_bias,
                   const float* mu, int64_t n_users, int64_t n_items, int32_t dim,
                   int64_t user_stride, int64_t item_stride /* floats between rows; 0 = dim */, int32_t flags,
                   const int32_t* query_users, int64_t n_queries, int32_t k, const int64_t* excl_indptr,
                   const int32_t* excl_item, double* topk_val, int32_t* topk_idx, void* workspace, int64_t workspace_bytes,
                   void* stream);

/* ---- fold-in of users that were not trained: exact least-squares user rows against the fixed item side -----------------
 * With item_feat, item_bias and mu fixed, the training loss (ops.py:81-89,124-126: squared error + reg * L2 on the gathered
 * rows, biases too with TFR_REG_BIAS) restricted to one user is a ridge regression in theta = [p_u ; b_u].  Its per-occurrence
 * gradients summed over the user's n ratings vanish exactly at the solution of
 *   (sum_j x_j x_j^T + reg * n * D) theta = sum_j (r_j - mu - b_{i_j}) x_j,   x_j = [v~_{i_j} ; 1],
 *   D = diag(1, ..., 1, REG_BIAS ? 1 : 0),   v~ = |v| with TFR_ABS_ITEM (ops.py:44), else v,
 * duplicates counted as in training.  Row r's ratings are items / rates [indptr[r] .. indptr[r + 1]) (indptr int64 [n + 1]);
 * out_feat [n, dim] / out_bias [n] receive theta rounded to fp32.  Float64 throughout, one CTA per row: Gram and right-hand
 * side summed in the row's CSR order from 0.0 (no atomics: a row's bits depend on its own ratings only, whatever the batch),
 * reg * n added to the diagonal, Cholesky + forward / back substitution in shared memory.  info [n] (int32): 0 = ok; j + 1 =
 * pivot j was not > 0 (reachable only with reg = 0); -1 = an item id outside [0, n_items), never read through; a row with
 * info != 0 is written as NaN.  A row without ratings gets p = 0, b = 0, info 0 (the model then scores it by mu + b_i).
 * reg is used as (double)reg.  Asynchronous, no workspace, capturable in a CUDA graph; n = 0 is a no-op.  TFR_ERR_INVALID
 * before any CUDA call for dim outside [1, 128], flags & TFR_LOSS_SIGMOID_CE (the fork's loss makes the problem
 * nonlinear), reg negative, NaN or infinite, and null pointers when n > 0.  The output goes straight into tfr_rank_users
 * as an n-row user table. */
int tfr_fold_in_users(const float* item_feat, const float* item_bias, const float* mu, int64_t n_items, int32_t dim,
                      int64_t item_stride /* floats between rows; 0 = dim */, int32_t flags, float reg,
                      const int64_t* indptr, const int32_t* items, const float* rates, int64_t n, float* out_feat,
                      float* out_bias, int32_t* info, void* stream);

/* ---- alternating least squares: exact user and item half-sweeps on the device --------------------------------------------
 * The objective is the training loss of the squared-error model, summed over every training occurrence (duplicates count):
 *   L = sum_(u,i,r) [ 1/2 (r - mu - b_u - b_i - p_u.q_i)^2 + 1/2 reg (|p_u|^2 + |q_i|^2) (+ 1/2 reg (b_u^2 + b_i^2) with
 *       TFR_REG_BIAS) ]
 * A sweep is three exact block minimisations of L, each of which can only lower it in exact arithmetic:
 *   1. users: tfr_als_half_sweep with the item side fixed (fixed = item_feat / item_bias, CSR by user of the item ids);
 *   2. items: tfr_als_half_sweep with the user side fixed (fixed = the fp32 user rows of step 1, CSR by item of the user ids);
 *   3. mu <- mu + sum e / N: tfr_svd_objective with mu_out = mu.
 * tfr_als_half_sweep: every row r of the solved side listed in light_rows or heavy_rows gets the (feat, bias) that solves
 * fold-in's system (tfr_fold_in_users) over its ratings partner / rates [indptr[r] .. indptr[r + 1]) against the fixed side,
 * in float64, rounded to fp32 and written to out_feat + r * out_stride / out_bias[r] (the m / v rows of an interleaved
 * table are never touched).  The plan (built once per training set by the caller):
 *   - light_rows [n_light]: rows with <= chunk ratings, solved one CTA per row with fold-in's code (same bits as
 *     tfr_fold_in_users of the same CSR);
 *   - heavy_rows [n_heavy], heavy_ptr int64 [n_heavy + 1], chunk_heavy [n_chunks]: rows with > chunk ratings; heavy row h owns
 *     chunks [heavy_ptr[h], heavy_ptr[h + 1]) of `chunk` consecutive ratings (the last one shorter), chunk_heavy[c] = h.
 *     One CTA per chunk writes its float64 Gram + right-hand side to the workspace (tfr_als_workspace_bytes(n_chunks, dim):
 *     (D (D + 1) / 2 + D) * 8 bytes per chunk, D = dim + 1), one CTA per heavy row sums them in chunk order and solves.
 *     chunk is the plan's: tfr_als_chunk() (knob ALS_CHUNK, clamped to [32, 2^20] and rounded up to a multiple of 32) at
 *     the time the plan was built.
 * A row without ratings gets zeros.  A row whose pivot is not > 0 (unreachable with reg > 0) or that names a partner id
 * outside [0, n_fixed) keeps its previous values and adds 1 to *n_failed (device int32, never reset here).  Asynchronous,
 * no host synchronisation, capturable in a CUDA graph; n_light = n_heavy = 0 is a no-op.  TFR_ERR_INVALID before any CUDA
 * call for dim outside [1, 128], flags & (TFR_LOSS_SIGMOID_CE | TFR_ABS_ITEM) (not least squares / not quadratic in q_i),
 * var_mask != TFR_VAR_ALL, reg <= 0, NaN or infinite (with reg > 0 every system is SPD) and null pointers.
 * tfr_svd_objective: over the CSR by user of the training ratings (user_items / user_rates, in range) and the item CSR's
 * indptr (for the item rows' occurrence counts), e = r - mu - b_u - b_i - p_u.q~_i per occurrence in float64 from the fp32
 * tables (q~ = |q| with TFR_ABS_ITEM); out6 (device, 6 doubles, optional) = (L, sum e^2, sum e, sum n_row |row|^2,
 * sum n_row b_row^2, N); mu_out (optional) = fl32(mu + sum e / N) when N > 0 (step 3).  Fixed-order reduction, no
 * floating-point atomics: the same bits every run.  workspace: tfr_svd_objective_workspace_bytes. */
int32_t tfr_als_chunk(void);
int64_t tfr_als_workspace_bytes(int64_t n_chunks, int32_t dim);
int tfr_als_half_sweep(const float* fixed_feat, const float* fixed_bias, const float* mu, int64_t n_fixed, int32_t dim,
                       int64_t fixed_stride /* floats between rows; 0 = dim */, int32_t flags, int32_t var_mask, float reg,
                       const int64_t* indptr, const int32_t* partner, const float* rates, const int32_t* light_rows,
                       int64_t n_light, const int32_t* heavy_rows, const int64_t* heavy_ptr, int64_t n_heavy,
                       const int32_t* chunk_heavy, int64_t n_chunks, int32_t chunk, float* out_feat,
                       int64_t out_stride /* 0 = dim */, float* out_bias, int32_t* n_failed, void* workspace,
                       int64_t workspace_bytes, void* stream);
int64_t tfr_svd_objective_workspace_bytes(int64_t n_users, int64_t n_items);
int tfr_svd_objective(const float* user_feat, const float* user_bias, const float* item_feat, const float* item_bias,
                      const float* mu, int64_t n_users, int64_t n_items, int32_t dim, int64_t user_stride,
                      int64_t item_stride /* 0 = dim */, int32_t flags, float reg, const int64_t* user_indptr,
                      const int32_t* user_items, const float* user_rates, const int64_t* item_indptr, double* out6,
                      float* mu_out, void* workspace, int64_t workspace_bytes, void* stream);

/* ---- host side of the feed_dict boundary: the columns a reference iterator yields (dataio.py:114-117: float64 views
 * of one [B, ncols] matrix, ids included) packed into a pinned staging buffer in the device's types -- int32 ids
 * (value cast, like TF feeding an int32 placeholder, A.7) followed by float32 rates: [users B | items B | rates B].
 * HOST pointers; dtype codes: 0 = float64, 1 = float32, 2 = int32, 3 = int64; strides in BYTES.  No device work.
 * user_num / item_num > 0: ids outside [0, num) are an error (TFR_ERR_INVALID, like TF's embedding_lookup raising
 * InvalidArgumentError on the CPU) -- nothing out of range ever reaches a gather; <= 0: unchecked. */
int tfr_host_pack_feed_checked(const void* users_host, int32_t users_dtype, int64_t users_stride,
                               const void* items_host, int32_t items_dtype, int64_t items_stride,
                               const void* rates_host, int32_t rates_dtype, int64_t rates_stride, int64_t n,
                               void* staging_host /* 12 * n bytes */, int64_t user_num, int64_t item_num);
int tfr_host_pack_feed(const void* users_host, int32_t users_dtype, int64_t users_stride, const void* items_host,
                       int32_t items_dtype, int64_t items_stride, const void* rates_host, int32_t rates_dtype,
                       int64_t rates_stride, int64_t n, void* staging_host /* 12 * n bytes */);

/* ---- the feed_dict step (what Session.prefetch / Session.run issue) -----------------------------------------------------
 * One staging set of the feed path; all memory and the five events (cudaEvent_t, tfr_event_create) are the caller's.
 * Four or five sets are used round-robin.  Every reuse is ordered by the set's events (or by the step stream itself): the
 * pinned buffer is never repacked while a copy out of it is queued, the device buffers never overwritten while a step
 * still reads them. */
typedef struct {
  void* h_feed;      /* pinned host, 12 * B bytes: [users int32 | items int32 | rates float32]                 */
  void* d_feed;      /* device, same layout                                                                    */
  float* d_out;      /* device, 2 * B floats: [logits | infer]                                                 */
  float* h_out;      /* pinned host, 2 * B floats                                                              */
  void* workspace;   /* tfr_svd_step_workspace_bytes(B, dim)                                                   */
  int64_t workspace_bytes;
  void *ev_h2d, *ev_sorted, *ev_pred, *ev_d2h, *ev_done;
  int32_t used;      /* set by the library: the set has been staged before (its events have a history)        */
  int32_t copied;    /* set by the library: a copy out of d_out has been issued                               */
  int32_t sorted;    /* set by the library: the batch's ids are sorted (or their sort is queued)               */
  int32_t staged;    /* set by the library: h_feed holds a packed batch that has not gone to the device        */
  uint32_t* d_sync;  /* device, 2 words, zero-initialised by the caller (graph steps: CTA counter, delivery count)  */
  uint32_t* h_flag;  /* pinned host, 1 word, zero-initialised by the caller (graph steps: the delivery count)       */
  uint32_t deliver_seq; /* set by the library: *h_flag >= deliver_seq once the last graph step's predictions are in h_out */
  uint32_t reserved;
} tfr_feed_set;
/* tfr_svd_feed_stage: HOST ONLY -- pack (tfr_host_pack_feed_checked: value cast + range check) into h_feed.  Needs nothing of
 * the model, blocks only on ev_h2d / ev_done of the set's previous use (the pinned buffer must be free to repack: its copy
 * to the device is over, and so is the step that consumed it), touches no stream: it may run on any host thread (the
 * engine's feed worker).
 * tfr_svd_feed_sort: H2D copy of the staged batch + the sort of its ids on side_stream, behind after_event when one is
 * given (NULL: as soon as the set's previous step has finished). */
int tfr_svd_feed_stage(const tfr_svd_tables* t, tfr_feed_set* set, const void* users_host, int32_t users_dtype,
                       int64_t users_stride, const void* items_host, int32_t items_dtype, int64_t items_stride,
                       const void* rates_host, int32_t rates_dtype, int64_t rates_stride, int64_t B);
int tfr_svd_feed_sort(const tfr_svd_tables* t, tfr_opt_scalars* opt, tfr_feed_set* set, int64_t B, void* side_stream,
                      void* after_event);
/* stage + sort (after_event = NULL) in one call. */
int tfr_svd_feed_prefetch(const tfr_svd_tables* t, tfr_opt_scalars* opt, tfr_feed_set* set, const void* users_host,
                          int32_t users_dtype, int64_t users_stride, const void* items_host, int32_t items_dtype,
                          int64_t items_stride, const void* rates_host, int32_t rates_dtype, int64_t rates_stride,
                          int64_t B, void* side_stream);
/* forward + segment sums -> [copy of the predictions to h_out on copy_stream, beside the table pass] -> Adam pass / SGD.
 * fetch: 0 = nothing, 1 = infer only (B floats into h_out[B..2B); the README head has logits == infer), 2 = logits and
 * infer.  Asynchronous: the caller waits on set->ev_d2h (tfr_event_synchronize) before reading h_out.
 * next_set (optional): a STAGED set -- its tfr_svd_feed_sort is queued on side_stream behind this step's forward
 * (after_event = this set's ev_pred). */
int tfr_svd_feed_step(const tfr_svd_tables* t, tfr_opt_scalars* opt, tfr_feed_set* set, int64_t B, int32_t flags,
                      int32_t var_mask, int32_t fetch, void* stream, void* copy_stream, tfr_feed_set* next_set,
                      void* side_stream);
/* The same step as ONE CUDA graph of kernels only: forward + segment sums -> { table pass | delivery of the predictions ->
 * fetch + id sort of next_set }.  The staged batch is read, and the predictions are written, by kernels over the pinned
 * buffers (zero-copy; h_feed / h_out / h_flag must be device-mapped pinned memory, cudaHostAlloc or torch pin_memory):
 * the shape of the device-resident stream path, whose batch assembly + sort are known to run beside the table pass.
 * Measured on B200 (profiles/r02_feed_path.md): launched eagerly on other streams, neither the sort nor the copy of the
 * predictions gets going before the pass has drained.
 * early_side != 0 (small tables, where the sort is longer than the pass): the fetch + sort branch forks at the start of the
 * step instead, and the delivery sits on the step stream in front of the pass.
 * create: captures on the two given streams (used for nothing else; relaxed mode) and instantiates; the executable graph
 * is bound to this (set, next_set, B, flags, var_mask, fetch) and to the tables' addresses; tfr_graph_destroy frees it.
 * launch: set must be sorted, next_set (if the graph was created with one) staged.  The predictions are in h_out when
 * *h_flag has reached set->deliver_seq (tfr_host_wait_flag); ev_h2d (next_set) is recorded inside the graph, ev_done (set)
 * behind it. */
int tfr_svd_feed_graph_create(const tfr_svd_tables* t, tfr_opt_scalars* opt, tfr_feed_set* set, tfr_feed_set* next_set,
                              int64_t B, int32_t flags, int32_t var_mask, int32_t fetch, int32_t early_side,
                              void* capture_stream, void* capture_side_stream, void** graph_exec_out);
int tfr_svd_feed_graph_launch(void* graph_exec, tfr_feed_set* set, tfr_feed_set* next_set, int32_t fetch, void* stream);
int tfr_event_synchronize(void* event);
/* spins (HOST) until *flag_host, a 32-bit counter in pinned memory, has reached at_least (wrap-around safe); TFR_ERR_CUDA
 * after timeout_us. */
int tfr_host_wait_flag(const void* flag_host, uint32_t at_least, int64_t timeout_us);

/* ---- DISCRETE-branch metrics on the device: replaces the host code of svd_train_val.py:94-98,138-143 -------------------
 * out4 (device, 4 doubles) = [ sum_b sigmoid_cross_entropy(labels_b, logits_b)   (cost_nll, ops.py:125-126),
 *                              #{b : round(sigmoid(logits_b)) == labels_b}         (:96,140),
 *                              roc_auc_score(labels, sigmoid(logits))              (:97,141; NaN if one class only),
 *                              #{b : labels_b > 0.5} ]
 * AUC by the rank statistic with tied scores averaged (what sklearn's trapezoids give): the fp32 probabilities are sorted
 * with the step's stable radix sort, runs of equal scores found by flags + prefix sums.  Deterministic. */
int64_t tfr_binary_metrics_workspace_bytes(int64_t n);
int tfr_binary_metrics(const float* logits, const float* labels, int64_t n, void* workspace, int64_t workspace_bytes,
                       double* out4, void* stream);

/* ---- top-k ranking metrics on the device --------------------------------------------------------------------------------
 * topk_idx [n_rows, k]: any ranking (tfr_allpairs_rank_excluding, tfr_topk_rows; -1 = no item, never a hit); relevant set
 * as CSR: rel_indptr int64 [n_rows + 1], rel_item int32 strictly ascending inside a row.  Per row u with R_u its relevant
 * items and h_r = [topk_idx[u, r] in R_u]:  HR = [sum h_r >= 1], precision = sum h_r / k, recall = sum h_r / |R_u|,
 * NDCG = sum_r h_r / log2(r + 2) over sum_{r < min(k, |R_u|)} 1 / log2(r + 2), in float64.  Rows with |R_u| = 0 are not
 * evaluated.  sums (device, 5 doubles) = (sum HR, sum precision, sum recall, sum NDCG, rows evaluated); row_metrics
 * (device, [n_rows, 4] = HR, precision, recall, NDCG; NaN for rows not evaluated) only when not null.  Fixed-order
 * reduction, no floating-point atomics: the same bits every run. */
int64_t tfr_ranking_metrics_workspace_bytes(int64_t n_rows, int32_t k);
int tfr_ranking_metrics(const int32_t* topk_idx, int64_t n_rows, int32_t k, const int64_t* rel_indptr, const int32_t* rel_item,
                        double* row_metrics, double* sums, void* workspace, int64_t workspace_bytes, void* stream);

/* ---- KTM design matrix on the device: replaces fm.py:61-93 df_to_sparse (scipy coo / hstack / tocsr on the host) ---------
 * One block per active agent, hstacked in the order given: agents_host[g] in 0..7 = users, items, skills, attempts, wins,
 * fails, item_wins, item_fails; col0_host[g] = first column of block g.  users / items: one-hot; skills: qmatrix[item];
 * wins / fails: the per-skill counters of the event (skill_wins / skill_fails CSR rows, explicit zeros kept);
 * attempts = skill_wins + skill_fails as scipy adds them (union pattern, zero sums dropped); item_wins / item_fails: the
 * item one-hot scaled by the event's wins / fails column.  Two steps: indptr (count + scan; indptr[n] = nnz), then fill.
 * Device pointers except agents_host / col0_host. */
int64_t tfr_ktm_workspace_bytes(int64_t n);
int tfr_ktm_csr_indptr(const int32_t* user, const int32_t* item, const float* wins_col, const float* fails_col,
                       const int64_t* q_indptr, const int32_t* q_indices, const float* q_data, const int64_t* sw_indptr,
                       const int32_t* sw_indices, const float* sw_data, const int64_t* sf_indptr, const int32_t* sf_indices,
                       const float* sf_data, int64_t n, const int32_t* agents_host, const int32_t* col0_host,
                       int32_t n_agents, int64_t* indptr, void* workspace, int64_t workspace_bytes, void* stream);
int tfr_ktm_csr_fill(const int32_t* user, const int32_t* item, const float* wins_col, const float* fails_col,
                     const int64_t* q_indptr, const int32_t* q_indices, const float* q_data, const int64_t* sw_indptr,
                     const int32_t* sw_indices, const float* sw_data, const int64_t* sf_indptr, const int32_t* sf_indices,
                     const float* sf_data, int64_t n, const int32_t* agents_host, const int32_t* col0_host,
                     int32_t n_agents, const int64_t* indptr, int32_t* indices, float* data, void* stream);

/* ---- ranking consumer: replaces forward.py:47-61 get_ranking (score every item for a user, sort, keep the first 50) ---
 * The k best entries of every row of scores [n_rows, n_cols] (row_stride floats between rows, 0 = n_cols), in rank
 * order: out_val / out_idx [n_rows, k].  Ties go to the lowest index, NaN is never ranked, missing ranks (k > number of
 * rankable entries) are (-inf, -1).  Scores come from tfr_svd_forward / tfr_fm_forward / tfr_allpairs. */
int tfr_topk_rows(const float* scores, int64_t n_rows, int64_t n_cols, int64_t row_stride, int32_t k, float* out_val,
                  int32_t* out_idx, void* stream);

/* ---- CUDA-graph helpers (thin wrappers so that a ctypes host needs no CUDA bindings) ------------ */
int tfr_graph_begin_capture(void* stream);
int tfr_graph_end_capture(void* stream, void** graph_exec_out);
int tfr_graph_launch(void* graph_exec, void* stream);
int tfr_graph_destroy(void* graph_exec);

#ifdef __cplusplus
}
#endif
#endif /* TFRECOMM_H_ */
