// K4: TF AdamOptimizer's IndexedSlices semantics (TF: adam.py::_apply_sparse_shared, SURVEY A.4; the
// optimizer north_star names, selected at ops.py:144/148):
//     m   = m*beta1                (WHOLE table)      m[uq]  += g*(1-beta1)
//     v   = v*beta2                (WHOLE table)      v[uq]  += (g*g)*(1-beta2)
//     var = var - (lr_t*m)/(sqrt(v)+eps)  (WHOLE table)
// TF runs this as ~8 unfused table-wide kernels; here each parameter is read and written exactly once
// per step (24 B/param): adam_stream_kernel is the streaming pass over the rows NOT in this step's
// slice (g = 0), adam_touched_kernel updates the slice rows with their summed gradient.  Every
// operation keeps TF's rounding order (separate mul/add, correctly rounded sqrt and divide).
// Also: dense ApplyAdam for bias_global (TF: training_ops.cc, A.5), scatter_sub SGD (ops.py:145) and
// the end-of-step bookkeeping (TF: adam.py::_finish).
#include <stdlib.h>
#include <string.h>

#include "adam_math.cuh"

namespace tfr {

// cache hints of the streaming accesses (TFR_STREAM_LD / TFR_STREAM_ST: 0 = .cs, 1 = default, 2 = .cg, 3 = .lu / .wt).
// Measured on B200 at the ML-25M shape (tools/pass_bench.py): loads .cg or .lu 131.5 us per pass against 140 us with
// .cs and 135-138 us with the default; the store hint makes no difference (.cs kept: evict-first, so the pass does not
// push the batch's gathered rows out of L2).  Default: ld = .cg, st = .cs.
__device__ __forceinline__ float4 ld_hint_f4(const float4* p, int h) {
  float4 r;
  if (h == 0) return ld_stream_f4(p);
  if (h == 1) asm volatile("ld.global.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p));
  else if (h == 2) asm volatile("ld.global.cg.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p));
  else asm volatile("ld.global.lu.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p));
  return r;
}
__device__ __forceinline__ void st_hint_f4(float4* p, const float4& v, int h) {
  if (h == 0) { st_stream_f4(p, v); return; }
  if (h == 1) asm volatile("st.global.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
  else if (h == 2) asm volatile("st.global.cg.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
  else asm volatile("st.global.wt.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}

// ---- the whole-table pass: every row of every table, in address order, ONE launch ----------------------
// Each parameter is read and written exactly once per step (24 B/param).  The concatenated tables are cut
// into units of 4 floats; a persistent grid strides over them, UNROLL units per thread and trip (6*UNROLL
// 16-byte requests in flight per thread), .cs (evict-first) accesses because nothing is reused.  A row of
// this step's slice (slot[row] = k >= 0) adds its summed gradient gsum[k]; all other rows get g = 0, for
// which m*b1 + 0*(1-b1), v*b2 + 0 reduce to TF's pure decay bit for bit.  Splitting the slice rows into a
// separate scattered kernel was measured slower: both halves lose DRAM page locality (4.9 and 3.7 TB/s
// against 6.0 TB/s for the in-order pass).
struct StreamTab {
  float *var, *m, *v;
  const int64_t* slot;  // (step stamp << 32 | run-head index); valid only if the stamp is this step's
  const float* gsum;
  const float* gsum0;  // two-step pass: the previous step's summed gradients (rows stamped with that step)
  uint32_t n;        // floats (rows * width)
  uint32_t width;    // floats per row
  uint32_t stride;   // floats between consecutive rows of var (and of m, of v): width, or 3*width when var | m | v of a
                     // row are interleaved (m = var + width, v = var + 2*width) -- then ONE stream is read and written
  uint32_t unit_end; // exclusive end of this table's units in the concatenated unit space
};
struct StreamArgs {
  StreamTab t[4];
  int n_tabs;
  uint32_t total_units;
  FinishArgs fin;
  // small tables (a few trips in all): the grid is PARTITIONED over the tables -- CTAs [cta_begin[i], cta_begin[i+1])
  // stream table i -- instead of every CTA walking table after table, which costs one round of latencies per table
  int partition;
  uint32_t cta_begin[5];
  int ld_hint, st_hint;
  int tl_every;   // debug timeline: every CTA stamps its exit (the true end of the pass, not a sample)
  int dynamic;    // 1: warps take chunks off opt->chunk_ctr[table] (needs fin: the last CTA resets the counters)
  int copy_only;  // experiment (TFR_STREAM_COPY_ONLY=1): same loads and stores, no arithmetic -- the memory ceiling
};

constexpr uint32_t DYN_TRIPS = 8;

// STEPS = 2: the pass applies two steps, t = global_step - 1 (already ended: tfr_svd_pair_bring) and t+1 = global_step,
// in registers.  Rows of batch t+1 (stamp t+1) were brought to the end of step t before step t+1's forward and take
// step t+1's gradient; rows of batch t only (stamp t) take step t's gradient, then step t+1's decay; all others decay
// twice.  Per element that is the fp32 sequence two one-step passes run, so the state is the same bit for bit.
template <int UNROLL, bool DYNAMIC, int STEPS>
__global__ void __launch_bounds__(512, 2) adam_stream_multi_kernel(const __grid_constant__ StreamArgs a,
                                                                const tfr_opt_scalars* __restrict__ opt, int tl_slot) {
  static_assert(STEPS == 1 || (STEPS == 2 && !DYNAMIC), "two-step pass: static schedule only");
  pdl_wait();                // the fix-up's summed gradients and slot maps are complete
  pdl_launch_dependents();   // the next step's segment sums may become resident as this grid drains
  TlScope tl_scope(opt, tl_slot, a.tl_every != 0);
  const AdamK k = load_k(opt);
  AdamK k0 = k;              // STEPS = 2: step t's scalars (only lr_t differs between two steps)
  if (STEPS == 2) k0.lr_t = opt->lr_t_prev;
  const uint32_t stamp = (uint32_t)opt->global_step;
  uint32_t stride = gridDim.x * blockDim.x;
  uint32_t gtid = blockIdx.x * blockDim.x + threadIdx.x;
  int tb0 = 0, tb1 = a.n_tabs;
  if (a.partition) {
    int mine = 0;
#pragma unroll
    for (int i = 1; i < 4; ++i)
      if (i < a.n_tabs && blockIdx.x >= a.cta_begin[i]) mine = i;
    tb0 = mine;
    tb1 = mine + 1;
    gtid = (blockIdx.x - a.cta_begin[mine]) * blockDim.x + threadIdx.x;
    stride = (a.cta_begin[mine + 1] - a.cta_begin[mine]) * blockDim.x;
  }
  // Table after table (no barrier in between: a thread that runs out of units of one table moves on to the next), so
  // that everything about the table -- pointers, row width, slot map -- is loop-invariant.
#pragma unroll 1
  for (int tb = tb0; tb < tb1; ++tb) {
    const StreamTab& t = a.t[tb];
    if ((t.width & 3u) == 0u) {
      // rows of whole 16-byte units: a unit lies in one row, so one slot-map lookup decides between TF's two cases --
      // a row of this step's slice (scatter-added gradient) or a row that only decays (m*b1, v*b2: exactly what TF's
      // table-wide assign computes; adam_grad with g = 0 would differ in the sign of a zero)
      const uint32_t n4 = t.n >> 2;
      const uint32_t upr = t.width >> 2;  // units per row
      const int sh = (upr & (upr - 1u)) == 0u ? 31 - __clz(upr) : -1;
      const uint32_t spr = t.stride >> 2;   // units between consecutive rows
      const bool dense = spr == upr;        // plain [rows][width] arrays: unit q is at offset q
      float4* const pv = reinterpret_cast<float4*>(t.var);
      float4* const pm = reinterpret_cast<float4*>(t.m);
      float4* const pz = reinterpret_cast<float4*>(t.v);
      // one trip: UNROLL units per thread, `us` units apart, the first at q0
      auto trip = [&](uint32_t q0, uint32_t us) {

        float4 x[UNROLL], y[UNROLL], z[UNROLL], g[UNROLL];
        bool has[UNROLL], has0[UNROLL];  // has: a row of this step's slice; has0 (STEPS = 2): of step t's only
        size_t at[UNROLL];
        uint32_t row[UNROLL];
#pragma unroll
        for (int u = 0; u < UNROLL; ++u) {
          const uint32_t q = q0 + u * us;
          if (q < n4) {
            row[u] = sh >= 0 ? (q >> sh) : (q / upr);
            at[u] = dense ? (size_t)q : (size_t)row[u] * spr + (q - row[u] * upr);
            x[u] = ld_hint_f4(pv + at[u], a.ld_hint);
            y[u] = ld_hint_f4(pm + at[u], a.ld_hint);
            z[u] = ld_hint_f4(pz + at[u], a.ld_hint);
          }
        }
#pragma unroll
        for (int u = 0; u < UNROLL; ++u) {
          const uint32_t q = q0 + u * us;
          has[u] = false;
          has0[u] = false;
          if (q < n4 && t.slot) {
            const int64_t sl = t.slot[row[u]];
            has[u] = (uint32_t)(sl >> 32) == stamp;
            if (STEPS == 2) has0[u] = (uint32_t)(sl >> 32) == stamp - 1u;
            if (has[u] || has0[u])
              g[u] = *reinterpret_cast<const float4*>((has[u] ? t.gsum : t.gsum0) + (size_t)(uint32_t)sl * t.width +
                                                      ((q - row[u] * upr) << 2));
          }
        }
#pragma unroll
        for (int u = 0; u < UNROLL; ++u) {
          const uint32_t q = q0 + u * us;
          if (q >= n4) continue;
          if (a.copy_only) {
          } else if (has[u]) {
            adam_grad(x[u].x, y[u].x, z[u].x, g[u].x, k);
            adam_grad(x[u].y, y[u].y, z[u].y, g[u].y, k);
            adam_grad(x[u].z, y[u].z, z[u].z, g[u].z, k);
            adam_grad(x[u].w, y[u].w, z[u].w, g[u].w, k);
          } else {
            if (STEPS == 2) {
              if (has0[u]) {
                adam_grad(x[u].x, y[u].x, z[u].x, g[u].x, k0);
                adam_grad(x[u].y, y[u].y, z[u].y, g[u].y, k0);
                adam_grad(x[u].z, y[u].z, z[u].z, g[u].z, k0);
                adam_grad(x[u].w, y[u].w, z[u].w, g[u].w, k0);
              } else {
                adam_decay(x[u].x, y[u].x, z[u].x, k0);
                adam_decay(x[u].y, y[u].y, z[u].y, k0);
                adam_decay(x[u].z, y[u].z, z[u].z, k0);
                adam_decay(x[u].w, y[u].w, z[u].w, k0);
              }
            }
            adam_decay(x[u].x, y[u].x, z[u].x, k);
            adam_decay(x[u].y, y[u].y, z[u].y, k);
            adam_decay(x[u].z, y[u].z, z[u].z, k);
            adam_decay(x[u].w, y[u].w, z[u].w, k);
          }
          st_hint_f4(pv + at[u], x[u], a.st_hint);
          st_hint_f4(pm + at[u], y[u], a.st_hint);
          st_hint_f4(pz + at[u], z[u], a.st_hint);
        }
      };
      if constexpr (!DYNAMIC) {
#pragma unroll 1
        for (uint32_t q0 = gtid; q0 < n4; q0 += stride * UNROLL) trip(q0, stride);
      } else {
        // dynamic: a WARP takes the next chunk of DYN_TRIPS * 32 * UNROLL consecutive units off a per-table counter, so
        // that the persistent grid's warps finish together whatever their SM's share of the memory system was
        constexpr uint32_t CHUNK = DYN_TRIPS * 32u * UNROLL;
        const uint32_t lane = threadIdx.x & 31u;
#pragma unroll 1
        for (;;) {
          uint32_t c = 0;
          if (lane == 0) c = atomicAdd(&a.fin.opt->chunk_ctr[tb], 1u);
          c = __shfl_sync(0xffffffffu, c, 0);
          if ((uint64_t)c * CHUNK >= n4) break;
          const uint32_t base = c * CHUNK + lane;
#pragma unroll 1
          for (uint32_t t_ = 0; t_ < DYN_TRIPS; ++t_) {
            const uint32_t q0 = base + t_ * 32u * UNROLL;
            if (q0 < n4) trip(q0, 32u);
          }
        }
      }
    } else {
      // dim 15 rows, bias tables (width 1): every float has its own row -- small tables, scalar path
#pragma unroll 1
      for (uint32_t e = gtid; e < t.n; e += stride) {
        const uint32_t row = t.width == 1u ? e : e / t.width;
        const size_t at = (size_t)row * t.stride + (e - row * t.width);
        float p = ld_stream_f1(t.var + at), q = ld_stream_f1(t.m + at), r = ld_stream_f1(t.v + at);
        bool hs = false, hs0 = false;
        float gg = 0.0f;
        if (t.slot) {
          const int64_t sl = t.slot[row];
          hs = (uint32_t)(sl >> 32) == stamp;
          if (STEPS == 2) hs0 = (uint32_t)(sl >> 32) == stamp - 1u;
          if (hs || hs0) gg = (hs ? t.gsum : t.gsum0)[(size_t)(uint32_t)sl * t.width + (e - row * t.width)];
        }
        if (hs) {
          adam_grad(p, q, r, gg, k);
        } else {
          if (STEPS == 2) {
            if (hs0) adam_grad(p, q, r, gg, k0); else adam_decay(p, q, r, k0);
          }
          adam_decay(p, q, r, k);
        }
        st_stream_f1(t.var + at, p);
        st_stream_f1(t.m + at, q);
        st_stream_f1(t.v + at, r);
      }
    }
  }
  if (a.fin.n_partials > 0) {  // the last CTA to get here ends the step (every CTA has read lr_t and the stamp by now)
    __shared__ int s_last;
    __syncthreads();
    if (threadIdx.x == 0) {
      __threadfence();
      s_last = atomicAdd(&a.fin.opt->ticket, 1u) == gridDim.x - 1;
    }
    __syncthreads();
    if (s_last && threadIdx.x < 32) {
      finish_step_scalars(a.fin.mu, a.fin.m_mu, a.fin.v_mu, a.fin.opt, a.fin.partials, a.fin.se_partials,
                          a.fin.n_partials);
      if (threadIdx.x == 0) {
        a.fin.opt->ticket = 0;
        for (int i = 0; i < 4; ++i) a.fin.opt->chunk_ctr[i] = 0;
      }
    }
  }
}

// ---- slice rows: one lane group per ENT consecutive sorted entries; run heads act --------------------------
// Both tables' slices (users, items) in ONE launch (blockIdx.y).  A group first decides which of its ENT
// entries are run heads, then issues the loads of all of them together (up to 4*ENT 16-byte requests per
// lane in flight) before any arithmetic: the kernel is a chain of dependent latencies otherwise.
struct SliceSide {
  float *var, *m, *v;        // feature table (null = not trained)
  float *bvar, *bm, *bv;     // bias table sharing the row ids (null = not trained)
  const int32_t* sid;        // sorted ids
  const float* gsum;         // [n, width] summed gradient at run heads
  const float* bgsum;        // [n]
  int64_t stride;            // floats between consecutive rows of var / m / v
};
constexpr int SLICE_ENT = 4;

template <int VEC, int L>
__global__ void __launch_bounds__(256) adam_slice_kernel(SliceSide s0, SliceSide s1, int width, int64_t n,
                                                         const tfr_opt_scalars* __restrict__ opt, int sgd, int tl_slot) {
  TlScope tl_scope(opt, tl_slot);
  const SliceSide s = blockIdx.y ? s1 : s0;
  const int lane = threadIdx.x & (L - 1);
  const int64_t kk0 = (((int64_t)blockIdx.x * blockDim.x + threadIdx.x) / L) * SLICE_ENT;
  if (kk0 >= n) return;
  int32_t id[SLICE_ENT];
  bool head[SLICE_ENT];
  int32_t prev = kk0 > 0 ? s.sid[kk0 - 1] : -1;
#pragma unroll
  for (int e = 0; e < SLICE_ENT; ++e) {
    const int64_t kk = kk0 + e;
    id[e] = kk < n ? s.sid[kk] : -1;
    head[e] = kk < n && id[e] != prev;
    prev = id[e];
  }
  AdamK k;
  if (!sgd) k = load_k(opt);
  if (s.bvar && lane == 0) {  // the rows' bias entries (a width-1 table sharing the row ids)
    float a[SLICE_ENT], b[SLICE_ENT], d[SLICE_ENT], g[SLICE_ENT];
#pragma unroll
    for (int e = 0; e < SLICE_ENT; ++e)
      if (head[e]) {
        a[e] = s.bvar[id[e]];
        g[e] = s.bgsum[kk0 + e];
        if (!sgd) { b[e] = s.bm[id[e]]; d[e] = s.bv[id[e]]; }
      }
#pragma unroll
    for (int e = 0; e < SLICE_ENT; ++e)
      if (head[e]) {
        if (sgd) {
          s.bvar[id[e]] = sub_rn(a[e], g[e]);
        } else {
          adam_grad(a[e], b[e], d[e], g[e], k);
          s.bvar[id[e]] = a[e]; s.bm[id[e]] = b[e]; s.bv[id[e]] = d[e];
        }
      }
  }
  if (!s.var) return;
  const int n_units = width / VEC;
  for (int unit = lane; unit < n_units; unit += L) {
    float a[SLICE_ENT][VEC], b[SLICE_ENT][VEC], d[SLICE_ENT][VEC], g[SLICE_ENT][VEC];
#pragma unroll
    for (int e = 0; e < SLICE_ENT; ++e) {
      if (!head[e]) continue;
      const size_t off = (size_t)id[e] * s.stride + (size_t)unit * VEC;
      const size_t goff = (size_t)(kk0 + e) * width + (size_t)unit * VEC;
      if constexpr (VEC == 4) {
        const float4 av = *reinterpret_cast<const float4*>(s.var + off);
        const float4 gv = *reinterpret_cast<const float4*>(s.gsum + goff);
        a[e][0] = av.x; a[e][1] = av.y; a[e][2] = av.z; a[e][3] = av.w;
        g[e][0] = gv.x; g[e][1] = gv.y; g[e][2] = gv.z; g[e][3] = gv.w;
        if (!sgd) {
          const float4 bv4 = *reinterpret_cast<const float4*>(s.m + off);
          const float4 dv4 = *reinterpret_cast<const float4*>(s.v + off);
          b[e][0] = bv4.x; b[e][1] = bv4.y; b[e][2] = bv4.z; b[e][3] = bv4.w;
          d[e][0] = dv4.x; d[e][1] = dv4.y; d[e][2] = dv4.z; d[e][3] = dv4.w;
        }
      } else {
        a[e][0] = s.var[off]; g[e][0] = s.gsum[goff];
        if (!sgd) { b[e][0] = s.m[off]; d[e][0] = s.v[off]; }
      }
    }
#pragma unroll
    for (int e = 0; e < SLICE_ENT; ++e) {
      if (!head[e]) continue;
      const size_t off = (size_t)id[e] * s.stride + (size_t)unit * VEC;
#pragma unroll
      for (int c = 0; c < VEC; ++c) {
        if (sgd) a[e][c] = sub_rn(a[e][c], g[e][c]);  // ops.py:145 scatter_sub; gsum holds the sum of lr*g
        else adam_grad(a[e][c], b[e][c], d[e][c], g[e][c], k);
      }
      if constexpr (VEC == 4) {
        *reinterpret_cast<float4*>(s.var + off) = make_float4(a[e][0], a[e][1], a[e][2], a[e][3]);
        if (!sgd) {
          *reinterpret_cast<float4*>(s.m + off) = make_float4(b[e][0], b[e][1], b[e][2], b[e][3]);
          *reinterpret_cast<float4*>(s.v + off) = make_float4(d[e][0], d[e][1], d[e][2], d[e][3]);
        }
      } else {
        s.var[off] = a[e][0];
        if (!sgd) { s.m[off] = b[e][0]; s.v[off] = d[e][0]; }
      }
    }
  }
}

// ---- two steps per table pass: bring the rows of batch t+1 to the end of step t -------------------------------
// Runs after step t's segment sums and before step t+1's forward, one lane group per SLICE_ENT sorted entries of batch
// t+1, both sides in one launch (blockIdx.y).  A run head's row (and its bias entry) takes step t's summed gradient if
// the slot map carries step t's stamp (the row is in both batches), step t's decay otherwise; written back in place.
// The two-step pass then owes these rows step t+1 only.  The last CTA ends step t.
struct BringSide {
  float *var, *m, *v;        // feature table (null = not trained)
  float *bvar, *bm, *bv;     // bias table sharing the row ids (null = not trained)
  const int32_t* sid;        // batch t+1's sorted ids
  const int64_t* slot;       // row -> slot map as step t's fix-up left it
  const float* gsum;         // step t's summed gradients [n, width], by run head
  const float* bgsum;        // [n]
  int64_t stride;            // floats between consecutive rows of var / m / v
};

template <int VEC, int L>
__global__ void __launch_bounds__(256) adam_bring_kernel(BringSide s0, BringSide s1, int width, int64_t n,
                                                         const tfr_opt_scalars* __restrict__ opt, FinishArgs fin) {
  {
    TlScope tl_scope(opt, TFR_TL_BRING);
    const BringSide s = blockIdx.y ? s1 : s0;
    const AdamK k = load_k(opt);
    const uint32_t stamp = (uint32_t)opt->global_step;
    const int lane = threadIdx.x & (L - 1);
    const int64_t kk0 = (((int64_t)blockIdx.x * blockDim.x + threadIdx.x) / L) * SLICE_ENT;
    if (kk0 < n && (s.var || s.bvar)) {
      int32_t id[SLICE_ENT];
      bool head[SLICE_ENT], in[SLICE_ENT];
      uint32_t gi[SLICE_ENT];
      int32_t prev = kk0 > 0 ? s.sid[kk0 - 1] : -1;
#pragma unroll
      for (int e = 0; e < SLICE_ENT; ++e) {
        const int64_t kk = kk0 + e;
        id[e] = kk < n ? s.sid[kk] : -1;
        head[e] = kk < n && id[e] != prev;
        prev = id[e];
        in[e] = false;
        gi[e] = 0;
        if (head[e]) {
          const int64_t sl = s.slot[id[e]];
          in[e] = (uint32_t)(sl >> 32) == stamp;
          gi[e] = (uint32_t)sl;
        }
      }
      if (s.bvar && lane == 0) {
        float a[SLICE_ENT], b[SLICE_ENT], d[SLICE_ENT], g[SLICE_ENT];
#pragma unroll
        for (int e = 0; e < SLICE_ENT; ++e)
          if (head[e]) {
            a[e] = s.bvar[id[e]]; b[e] = s.bm[id[e]]; d[e] = s.bv[id[e]];
            if (in[e]) g[e] = s.bgsum[gi[e]];
          }
#pragma unroll
        for (int e = 0; e < SLICE_ENT; ++e)
          if (head[e]) {
            if (in[e]) adam_grad(a[e], b[e], d[e], g[e], k); else adam_decay(a[e], b[e], d[e], k);
            s.bvar[id[e]] = a[e]; s.bm[id[e]] = b[e]; s.bv[id[e]] = d[e];
          }
      }
      if (s.var) {
        const int n_units = width / VEC;
        for (int unit = lane; unit < n_units; unit += L) {
          float a[SLICE_ENT][VEC], b[SLICE_ENT][VEC], d[SLICE_ENT][VEC], g[SLICE_ENT][VEC];
#pragma unroll
          for (int e = 0; e < SLICE_ENT; ++e) {
            if (!head[e]) continue;
            const size_t off = (size_t)id[e] * s.stride + (size_t)unit * VEC;
            const size_t goff = (size_t)gi[e] * width + (size_t)unit * VEC;
            if constexpr (VEC == 4) {
              const float4 av = *reinterpret_cast<const float4*>(s.var + off);
              const float4 bv4 = *reinterpret_cast<const float4*>(s.m + off);
              const float4 dv4 = *reinterpret_cast<const float4*>(s.v + off);
              a[e][0] = av.x; a[e][1] = av.y; a[e][2] = av.z; a[e][3] = av.w;
              b[e][0] = bv4.x; b[e][1] = bv4.y; b[e][2] = bv4.z; b[e][3] = bv4.w;
              d[e][0] = dv4.x; d[e][1] = dv4.y; d[e][2] = dv4.z; d[e][3] = dv4.w;
              if (in[e]) {
                const float4 gv = *reinterpret_cast<const float4*>(s.gsum + goff);
                g[e][0] = gv.x; g[e][1] = gv.y; g[e][2] = gv.z; g[e][3] = gv.w;
              }
            } else {
              a[e][0] = s.var[off]; b[e][0] = s.m[off]; d[e][0] = s.v[off];
              if (in[e]) g[e][0] = s.gsum[goff];
            }
          }
#pragma unroll
          for (int e = 0; e < SLICE_ENT; ++e) {
            if (!head[e]) continue;
            const size_t off = (size_t)id[e] * s.stride + (size_t)unit * VEC;
#pragma unroll
            for (int c = 0; c < VEC; ++c) {
              if (in[e]) adam_grad(a[e][c], b[e][c], d[e][c], g[e][c], k);
              else adam_decay(a[e][c], b[e][c], d[e][c], k);
            }
            if constexpr (VEC == 4) {
              *reinterpret_cast<float4*>(s.var + off) = make_float4(a[e][0], a[e][1], a[e][2], a[e][3]);
              *reinterpret_cast<float4*>(s.m + off) = make_float4(b[e][0], b[e][1], b[e][2], b[e][3]);
              *reinterpret_cast<float4*>(s.v + off) = make_float4(d[e][0], d[e][1], d[e][2], d[e][3]);
            } else {
              s.var[off] = a[e][0]; s.m[off] = b[e][0]; s.v[off] = d[e][0];
            }
          }
        }
      }
    }
  }
  // the last CTA to get here ends step t (every CTA has read lr_t and the stamp by now)
  __shared__ int s_last;
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    s_last = atomicAdd(&fin.opt->ticket, 1u) == gridDim.x * gridDim.y - 1;
  }
  __syncthreads();
  if (s_last && threadIdx.x < 32) {
    finish_step_scalars(fin.mu, fin.m_mu, fin.v_mu, fin.opt, fin.partials, fin.se_partials, fin.n_partials);
    if (threadIdx.x == 0) fin.opt->ticket = 0;
  }
}

// ---- end of step (as a launch of its own: SGD mode, no trained table, the piecewise API) ---------------------
// The row -> slot maps carry the step's stamp, so nothing has to be reset between steps.
__global__ void __launch_bounds__(32) finish_step_kernel(tfr_svd_tables t, tfr_opt_scalars* opt,
                                                         const float* __restrict__ partials,
                                                         const double* __restrict__ se_partials, int n_partials) {
  TlScope tl_scope(opt, TFR_TL_FINISH);
  finish_step_scalars(t.mu, t.m_mu, t.v_mu, opt, partials, se_partials, n_partials);
}

__global__ void opt_init_kernel(tfr_opt_scalars* opt, float lr, float reg, float beta1, float beta2, float eps,
                                int flags, int var_mask) {
  opt->lr = lr; opt->reg = reg; opt->beta1 = beta1; opt->beta2 = beta2; opt->eps = eps;
  opt->beta1_power = beta1; opt->beta2_power = beta2;  // TF: adam.py _create_slots
  opt->one_minus_beta1 = sub_rn(1.0f, beta1);
  opt->one_minus_beta2 = sub_rn(1.0f, beta2);
  float tt = sqrt_rn(sub_rn(1.0f, beta2));
  opt->lr_t = div_rn(mul_rn(lr, tt), sub_rn(1.0f, beta1));
  opt->lr_t_prev = opt->lr_t;
  opt->flags = flags; opt->var_mask = var_mask;
  opt->global_step = 0; opt->batch_cursor = 0; opt->prefetch_cursor = 0;
  opt->se_sum = 0.0; opt->g_mu = 0.0f; opt->ticket = 0u;
  for (int i = 0; i < 4; ++i) opt->chunk_ctr[i] = 0u;
  opt->se_ring = nullptr; opt->se_ring_len = 0; opt->timeline = nullptr;
}

}  // namespace tfr

using namespace tfr;

extern "C" int tfr_opt_init(tfr_opt_scalars* opt_dev, float lr, float reg, float beta1, float beta2, float eps,
                            int32_t flags, int32_t var_mask, void* stream) {
  TFR_CHECK_ARG(opt_dev);
  opt_init_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(opt_dev, lr, reg, beta1, beta2, eps, flags, var_mask);
  TFR_LAUNCH_CHECK();
  return TFR_OK;
}

static int launch_stream_chunks(const StreamTab* chunks, int n_chunks, const tfr_opt_scalars* opt, int tl_slot,
                                cudaStream_t st, const FinishArgs* fin, int steps) {
  StreamArgs a;
  memset(&a, 0, sizeof(a));
  if (fin) a.fin = *fin;
  uint64_t units = 0;
  for (int i = 0; i < n_chunks; ++i) {
    a.t[i] = chunks[i];
    units += ((uint64_t)chunks[i].n + 3) / 4;
    a.t[i].unit_end = (uint32_t)units;
  }
  a.n_tabs = n_chunks;
  a.total_units = (uint32_t)units;
  a.copy_only = tune(TUNE_STREAM_COPY_ONLY);
  a.dynamic = (fin && steps == 1 && tune(TUNE_STREAM_DYNAMIC)) ? 1 : 0;
  a.tl_every = tune(TUNE_TL_EVERY_CTA);
  a.ld_hint = tune(TUNE_STREAM_LD);
  a.st_hint = tune(TUNE_STREAM_ST);
  // persistent grid: 2 CTAs x 448 threads x 64 registers per SM, 2 units per thread and trip.  448, not 512: two
  // CTAs of 512 threads take the whole register file, and the id sort of the NEXT batch (8K registers per CTA,
  // forked under this pass) could then only start when the pass drains -- which puts it on the critical path.
  // (3 x 256 also leaves room but measures 7 % slower: TFR_STREAM_* to experiment.)
  const int cfg_ctas = tune(TUNE_STREAM_CTAS_PER_SM);
  int cfg_unroll = tune(TUNE_STREAM_UNROLL);
  if (cfg_unroll < 1) cfg_unroll = 2;
  int cfg_threads = tune(TUNE_STREAM_THREADS);
  if (cfg_threads < 32 || cfg_threads > 512) cfg_threads = 448;
  cfg_threads &= ~31;  // whole warps: the dynamic variant's warp-wide shuffle needs every lane
  int64_t grid = ((int64_t)units + cfg_threads * cfg_unroll - 1) / (cfg_threads * cfg_unroll);
  const int64_t cap = (int64_t)sm_count() * cfg_ctas;
  if (cfg_ctas > 0 && grid > cap) grid = cap;
  // small tables: one slice of the grid per table (work counted in thread-trips: a vector table does 4 floats per
  // thread and trip, a scalar-path table one)
  uint64_t total_floats = 0;
  for (int i = 0; i < n_chunks; ++i) total_floats += chunks[i].n;
  if (n_chunks > 1 && total_floats * 12 < ((uint64_t)32 << 20)) {
    uint64_t work[4], total_work = 0;
    for (int i = 0; i < n_chunks; ++i) {
      work[i] = (chunks[i].width % 4 == 0) ? ((uint64_t)chunks[i].n + 3) / 4 : chunks[i].n;
      total_work += work[i];
    }
    int64_t want = (int64_t)((total_work + cfg_threads - 1) / cfg_threads);
    if (want > cap && cfg_ctas > 0) want = cap;
    if (want < n_chunks) want = n_chunks;
    uint32_t at = 0;
    for (int i = 0; i < n_chunks; ++i) {
      a.cta_begin[i] = at;
      uint64_t share = (work[i] * (uint64_t)want + total_work - 1) / total_work;
      if (share < 1) share = 1;
      at += (uint32_t)share;
    }
    a.cta_begin[n_chunks] = at;
    a.partition = 1;
    grid = at;
  }
  const bool pdl = tune(TUNE_PDL) != 0;
  if (steps == 2) {  // UNROLL 2 only: at 4 the kernel spills at 64 registers
    TFR_PREP((adam_stream_multi_kernel<2, false, 2>));
    TFR_CUDA(launch_kernel(adam_stream_multi_kernel<2, false, 2>, dim3((unsigned)grid), dim3(cfg_threads), 0, st, pdl, a, opt, tl_slot));
  } else if (a.dynamic) {
    TFR_PREP((adam_stream_multi_kernel<2, true, 1>));
    TFR_CUDA(launch_kernel(adam_stream_multi_kernel<2, true, 1>, dim3((unsigned)grid), dim3(cfg_threads), 0, st, pdl, a, opt, tl_slot));
  } else if (cfg_unroll >= 4) {
    TFR_PREP((adam_stream_multi_kernel<4, false, 1>));
    TFR_CUDA(launch_kernel(adam_stream_multi_kernel<4, false, 1>, dim3((unsigned)grid), dim3(cfg_threads), 0, st, pdl, a, opt, tl_slot));
  } else {
    TFR_PREP((adam_stream_multi_kernel<2, false, 1>));
    TFR_CUDA(launch_kernel(adam_stream_multi_kernel<2, false, 1>, dim3((unsigned)grid), dim3(cfg_threads), 0, st, pdl, a, opt, tl_slot));
  }
  return TFR_OK;
}

namespace tfr {
// adam_ring.cu: the TMA-bulk ring pass for interleaved feature tables (+ plain bias tables)
bool ring_pass_eligible(const tfr_adam_table* tabs, int n);
int ring_pass_launch(const tfr_adam_table* tabs, int n, const tfr_opt_scalars* opt, int tl_slot, cudaStream_t st,
                     const FinishArgs* fin);
// fin != null: the pass's last launch also ends the step (see FinishArgs); returns 1 if it did, 0 if no launch
// was issued (nothing to stream), negative on error.
// gsum0 (null: one step): the previous step's summed gradient of every table -- the two-step pass (always the LDG pass)
int adam_stream_multi_impl(const tfr_adam_table* tables, int32_t n_tables, tfr_opt_scalars* opt, int32_t tl_slot,
                           void* stream, const FinishArgs* fin, const float* const* gsum0 = nullptr);
}

extern "C" int tfr_adam_stream_multi(const tfr_adam_table* tables, int32_t n_tables, const tfr_opt_scalars* opt,
                                     int32_t tl_slot, void* stream) {
  const int rc = adam_stream_multi_impl(tables, n_tables, const_cast<tfr_opt_scalars*>(opt), tl_slot, stream, nullptr);
  return rc < 0 ? rc : TFR_OK;
}

int tfr::adam_stream_multi_impl(const tfr_adam_table* tables, int32_t n_tables, tfr_opt_scalars* opt, int32_t tl_slot,
                                void* stream, const FinishArgs* fin, const float* const* gsum0) {
  TFR_CHECK_ARG(tables && n_tables >= 1 && n_tables <= 4 && opt && tl_slot >= 0 && tl_slot < TFR_TL_SLOTS);
  for (int i = 0; i < n_tables; ++i) {
    TFR_CHECK_ARG(tables[i].rows >= 0 && tables[i].width > 0);
    TFR_CHECK_ARG(tables[i].rows == 0 || (tables[i].var && tables[i].m && tables[i].v && (!tables[i].slot || tables[i].gsum)));
  }
  const int steps = gsum0 ? 2 : 1;
  for (int i = 0; gsum0 && i < n_tables; ++i)
    TFR_CHECK_ARG(tables[i].rows == 0 || (tables[i].slot && gsum0[i] && (tables[i].width % 4 != 0 || (uintptr_t)gsum0[i] % 16 == 0)));
  if (steps == 1 && ring_pass_eligible(tables, n_tables)) {
    const int rc = ring_pass_launch(tables, n_tables, opt, tl_slot, (cudaStream_t)stream, fin);
    return rc < 0 ? rc : 1;
  }
  // The kernel indexes floats with 32 bits: a table of >= 2^32 floats (the 50M x 128 user shard of configs[4] at
  // G = 2) is cut into row ranges, and launches are split so that one launch covers < 2^32 units.
  const uint64_t kMaxFloats = ((uint64_t)1 << 32) - 8;
  StreamTab pending[4];
  int np = 0;
  uint64_t pending_units = 0;
  cudaStream_t st = (cudaStream_t)stream;
  for (int i = 0; i < n_tables; ++i) {
    const tfr_adam_table& t = tables[i];
    TFR_CHECK_ARG(t.rows >= 0 && t.width > 0);
    if (t.rows == 0) continue;
    TFR_CHECK_ARG(t.var && t.m && t.v && (!t.slot || t.gsum));
    // rows of whole 16-byte units are streamed with 128-bit accesses; other widths (dim 15, biases) go scalar
    TFR_CHECK_ARG(t.width % 4 != 0 ||
                  (((uintptr_t)t.var % 16 == 0) && ((uintptr_t)t.m % 16 == 0) && ((uintptr_t)t.v % 16 == 0)));
    const uint64_t rstride = t.stride ? (uint64_t)t.stride : (uint64_t)t.width;
    TFR_CHECK_ARG(rstride >= (uint64_t)t.width && rstride < ((uint64_t)1 << 31) && (t.width % 4 != 0 || rstride % 4 == 0));
    TFR_CHECK_ARG(!t.gsum || t.width % 4 != 0 || (uintptr_t)t.gsum % 16 == 0);
    uint64_t rows_per_chunk = kMaxFloats / (uint64_t)t.width;
    rows_per_chunk -= rows_per_chunk % 4;  // keeps every chunk's first float 16-byte aligned for any width
    for (uint64_t r0 = 0; r0 < (uint64_t)t.rows; r0 += rows_per_chunk) {
      const uint64_t nr = ((uint64_t)t.rows - r0 < rows_per_chunk) ? (uint64_t)t.rows - r0 : rows_per_chunk;
      StreamTab c;
      const uint64_t off = r0 * rstride;
      c.var = t.var + off; c.m = t.m + off; c.v = t.v + off;
      c.stride = (uint32_t)rstride;
      c.slot = t.slot ? t.slot + r0 : nullptr;
      c.gsum = t.gsum;
      c.gsum0 = gsum0 ? gsum0[i] : nullptr;
      c.n = (uint32_t)(nr * (uint64_t)t.width);
      c.width = (uint32_t)t.width;
      c.unit_end = 0;
      const uint64_t cu = ((uint64_t)c.n + 3) / 4;
      if (np == 4 || pending_units + cu >= ((uint64_t)1 << 32)) {
        int rc = launch_stream_chunks(pending, np, opt, tl_slot, st, nullptr, steps);
        if (rc) return rc;
        np = 0;
        pending_units = 0;
      }
      pending[np++] = c;
      pending_units += cu;
    }
  }
  if (np) {
    const int rc = launch_stream_chunks(pending, np, opt, tl_slot, st, fin, steps);
    return rc < 0 ? rc : 1;
  }
  return 0;
}

extern "C" int tfr_adam_slice_multi(const tfr_slice_update* sides, int32_t n_sides, int32_t width, int64_t n,
                                    const tfr_opt_scalars* opt, int32_t sgd, int32_t tl_slot, void* stream) {
  TFR_CHECK_ARG(sides && n_sides >= 1 && n_sides <= 2 && width > 0 && n >= 0 && tl_slot >= 0 && tl_slot < TFR_TL_SLOTS);
  if (n == 0) return TFR_OK;
  TFR_CHECK_ARG(sgd || opt);
  SliceSide ss[2];
  memset(ss, 0, sizeof(ss));
  for (int i = 0; i < n_sides; ++i) {
    const tfr_slice_update& u = sides[i];
    TFR_CHECK_ARG(u.sorted_ids);
    TFR_CHECK_ARG(!u.var || (u.gsum && (sgd || (u.m && u.v))));
    TFR_CHECK_ARG(!u.bvar || (u.bgsum && (sgd || (u.bm && u.bv))));
    ss[i].var = u.var; ss[i].m = u.m; ss[i].v = u.v; ss[i].bvar = u.bvar; ss[i].bm = u.bm; ss[i].bv = u.bv;
    ss[i].sid = u.sorted_ids; ss[i].gsum = u.gsum; ss[i].bgsum = u.bgsum;
    ss[i].stride = u.stride ? u.stride : width;
  }
  const RowGeom g = row_geom(width);
  const int64_t groups = (n + SLICE_ENT - 1) / SLICE_ENT;
  const int groups_per_cta = 256 / g.lanes;
  dim3 grid((unsigned)((groups + groups_per_cta - 1) / groups_per_cta), (unsigned)n_sides);
  cudaStream_t st = (cudaStream_t)stream;
#define TFR_SLICE_CASE(V, LL)                                                                        \
  if (g.vec == V && g.lanes == LL) {                                                                 \
    TFR_PREP((adam_slice_kernel<V, LL>));                                                            \
    adam_slice_kernel<V, LL><<<grid, 256, 0, st>>>(ss[0], ss[1], width, n, opt, sgd, tl_slot);       \
    TFR_LAUNCH_CHECK();                                                                               \
    return TFR_OK;                                                                                    \
  }
  TFR_SLICE_CASE(4, 1) TFR_SLICE_CASE(4, 2) TFR_SLICE_CASE(4, 4) TFR_SLICE_CASE(4, 8) TFR_SLICE_CASE(4, 16)
  TFR_SLICE_CASE(4, 32) TFR_SLICE_CASE(1, 1) TFR_SLICE_CASE(1, 2) TFR_SLICE_CASE(1, 4) TFR_SLICE_CASE(1, 8)
  TFR_SLICE_CASE(1, 16) TFR_SLICE_CASE(1, 32)
#undef TFR_SLICE_CASE
  set_error("unsupported width %d", width);
  return TFR_ERR_INVALID;
}

extern "C" int tfr_adam_touched(float* var, float* m, float* v, int32_t width, const int32_t* sorted_ids, int64_t n,
                                const float* gsum, const tfr_opt_scalars* opt, void* stream) {
  tfr_slice_update u{var, m, v, nullptr, nullptr, nullptr, sorted_ids, gsum, nullptr, 0};
  return tfr_adam_slice_multi(&u, 1, width, n, opt, 0, TFR_TL_SLOTS - 1, stream);
}

extern "C" int tfr_sgd_apply(float* var, int32_t width, const int32_t* sorted_ids, int64_t n, const float* gsum,
                             void* stream) {
  tfr_slice_update u{var, nullptr, nullptr, nullptr, nullptr, nullptr, sorted_ids, gsum, nullptr, 0};
  return tfr_adam_slice_multi(&u, 1, width, n, nullptr, 1, TFR_TL_SLOTS - 1, stream);
}

extern "C" int tfr_svd_finish_step(const tfr_svd_tables* t, tfr_opt_scalars* opt, const int32_t* users,
                                   const int32_t* items, int64_t B, const tfr_svd_step_ws* ws, int32_t n_partials,
                                   void* stream) {
  (void)users; (void)items; (void)B;  // kept in the signature: the slot maps are stamped, nothing to reset per id
  TFR_CHECK_ARG(t && opt && ws && n_partials > 0 && n_partials <= TFR_MAX_PARTIALS && t->mu);
  TFR_PREP(finish_step_kernel);
  finish_step_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(*t, opt, ws->partials, ws->se_partials, n_partials);
  TFR_LAUNCH_CHECK();
  return TFR_OK;
}

namespace tfr {
// the Adam pass of a step with the end-of-step work folded into its last CTA (falls back to the finish launch when
// there is nothing to stream)
int adam_pass_and_finish(const tfr_adam_table* tabs, int nt, const tfr_svd_tables* t, tfr_opt_scalars* opt,
                         const tfr_svd_step_ws* ws, int n_partials, int tl_slot, void* stream) {
  TFR_CHECK_ARG(n_partials > 0 && n_partials <= TFR_MAX_PARTIALS);
  int rc = 0;
  if (nt > 0) {
    const FinishArgs fin{opt, t->mu, t->m_mu, t->v_mu, ws->partials, ws->se_partials, n_partials};
    rc = adam_stream_multi_impl(tabs, nt, opt, tl_slot, stream, &fin);
    if (rc < 0) return rc;
  }
  if (rc == 0) return tfr_svd_finish_step(t, opt, nullptr, nullptr, 0, ws, n_partials, stream);
  return TFR_OK;
}

// the two-step pass of steps t (ended, summed gradients gsum0[i] of table i) and t+1 (ws), which it ends
int adam_pair_pass_and_finish(const tfr_adam_table* tabs, const float* const* gsum0, int nt, const tfr_svd_tables* t,
                              tfr_opt_scalars* opt, const tfr_svd_step_ws* ws, int n_partials, void* stream) {
  TFR_CHECK_ARG(n_partials > 0 && n_partials <= TFR_MAX_PARTIALS);
  int rc = 0;
  if (nt > 0) {
    const FinishArgs fin{opt, t->mu, t->m_mu, t->v_mu, ws->partials, ws->se_partials, n_partials};
    rc = adam_stream_multi_impl(tabs, nt, opt, TFR_TL_STREAM_UF, stream, &fin, gsum0);
    if (rc < 0) return rc;
  }
  if (rc == 0) return tfr_svd_finish_step(t, opt, nullptr, nullptr, 0, ws, n_partials, stream);
  return TFR_OK;
}

// sides[i].gsum / bgsum: step t's summed gradients; sorted_ids: batch t+1's; slot[i]: the side's row -> slot map
int adam_bring_and_finish(const tfr_slice_update* sides, const int64_t* const* slot, int32_t width, int64_t n,
                          const tfr_svd_tables* t, tfr_opt_scalars* opt, const tfr_svd_step_ws* ws, int n_partials,
                          void* stream) {
  TFR_CHECK_ARG(sides && slot && width > 0 && n > 0 && opt && n_partials > 0 && n_partials <= TFR_MAX_PARTIALS);
  BringSide ss[2];
  for (int i = 0; i < 2; ++i) {
    const tfr_slice_update& u = sides[i];
    TFR_CHECK_ARG(u.sorted_ids && slot[i]);
    TFR_CHECK_ARG(!u.var || (u.gsum && u.m && u.v));
    TFR_CHECK_ARG(!u.bvar || (u.bgsum && u.bm && u.bv));
    ss[i] = BringSide{u.var, u.m, u.v, u.bvar, u.bm, u.bv, u.sorted_ids, slot[i], u.gsum, u.bgsum,
                      u.stride ? u.stride : width};
  }
  const FinishArgs fin{opt, t->mu, t->m_mu, t->v_mu, ws->partials, ws->se_partials, n_partials};
  const RowGeom g = row_geom(width);
  const int64_t groups = (n + SLICE_ENT - 1) / SLICE_ENT;
  const int groups_per_cta = 256 / g.lanes;
  dim3 grid((unsigned)((groups + groups_per_cta - 1) / groups_per_cta), 2u);
  cudaStream_t st = (cudaStream_t)stream;
#define TFR_BRING_CASE(V, LL)                                                                        \
  if (g.vec == V && g.lanes == LL) {                                                                 \
    TFR_PREP((adam_bring_kernel<V, LL>));                                                            \
    adam_bring_kernel<V, LL><<<grid, 256, 0, st>>>(ss[0], ss[1], width, n, opt, fin);                \
    TFR_LAUNCH_CHECK();                                                                               \
    return TFR_OK;                                                                                    \
  }
  TFR_BRING_CASE(4, 1) TFR_BRING_CASE(4, 2) TFR_BRING_CASE(4, 4) TFR_BRING_CASE(4, 8) TFR_BRING_CASE(4, 16)
  TFR_BRING_CASE(4, 32) TFR_BRING_CASE(1, 1) TFR_BRING_CASE(1, 2) TFR_BRING_CASE(1, 4) TFR_BRING_CASE(1, 8)
  TFR_BRING_CASE(1, 16) TFR_BRING_CASE(1, 32)
#undef TFR_BRING_CASE
  set_error("unsupported width %d", width);
  return TFR_ERR_INVALID;
}
}  // namespace tfr
