// K3b: ordered segment sums of the per-occurrence gradients -- the "segment-reduce" half of the dedup
// (TF: tf.unsorted_segment_sum inside optimizer.py::_deduplicate_indexed_slices, SURVEY A.3), fused
// with the backward itself so the [B,dim] per-occurrence gradient rows of TF's IndexedSlices are never
// written to HBM.
//
// Backward restated (SURVEY 8a row a10; TF autodiff of ops.py:124-126,140 through ops.py:44-47,81-89):
//   user row u, occurrence b:  g = e_b * v'_b + reg * u        (v' = |v| if TFR_ABS_ITEM)
//   item row v, occurrence b:  g = (e_b * u_b) [* sign(v)] + reg * v
//   bias:                      g = e_b (+ reg * bias if TFR_REG_BIAS)
// each product and the add a separate fp32 rounding (separate TF kernels + AddN).  In SGD mode
// (ops.py:145) the summand is lr*g so that the apply is a single subtraction.
//
// Work decomposition: the sorted (id,pos) array is cut into tiles of 32 entries, one lane group per
// tile.  A group walks its tile in order, keeping the running sum of the current run of equal ids.
// Runs that begin and end inside the tile are final: gsum[head index] = sum.  A run that crosses a
// tile boundary leaves a partial (cont[t]: continues a run begun earlier; tail[t]: begins here, goes
// on) and the fix-up kernel adds the partials of consecutive tiles in order.  The result is a fixed
// function of the input (deterministic) and equals the in-order sum except for regrouping at the
// 32-entry tile boundaries.
#include <stdlib.h>

#include <map>
#include <mutex>

#include "segsum.cuh"

namespace tfr {

constexpr int SEG_TILE_MAX = 32;  // tiles of 32, 16 or 8 sorted entries: tfr::seg_tile(B, dim)

template <int VEC>
struct Acc {
  float v[VEC];
};

template <int VEC>
__device__ __forceinline__ Acc<VEC> load_units(const float* row, int unit) {
  Acc<VEC> a;
  if constexpr (VEC == 4) {
    const float4 x = ld_gather_f4(reinterpret_cast<const float4*>(row) + unit);
    a.v[0] = x.x; a.v[1] = x.y; a.v[2] = x.z; a.v[3] = x.w;
  } else {
    a.v[0] = ld_gather_f1(row + unit);
  }
  return a;
}

template <int VEC>
__device__ __forceinline__ void store_units(float* row, int unit, const Acc<VEC>& a) {
  if constexpr (VEC == 4) {
    reinterpret_cast<float4*>(row)[unit] = make_float4(a.v[0], a.v[1], a.v[2], a.v[3]);
  } else {
    row[unit] = a.v[0];
  }
}

// ---- asynchronous global -> shared copies (LDGSTS): the rows a tile needs are staged in shared memory without
// passing through registers, so that many rows are in flight per lane group while the consuming loop stays compact
template <int VEC>
__device__ __forceinline__ void cp_async_units(float* smem_dst, const float* gsrc) {
  const uint32_t d = (uint32_t)__cvta_generic_to_shared(smem_dst);
  if constexpr (VEC == 4) asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d), "l"(gsrc) : "memory");
  else asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(d), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

template <int VEC>
__device__ __forceinline__ Acc<VEC> lds_units(const float* row, int unit) {
  Acc<VEC> a;
  if constexpr (VEC == 4) {
    const float4 x = reinterpret_cast<const float4*>(row)[unit];
    a.v[0] = x.x; a.v[1] = x.y; a.v[2] = x.z; a.v[3] = x.w;
  } else {
    a.v[0] = row[unit];
  }
  return a;
}

#ifndef SEG_PBASE
#define SEG_PBASE 4
#endif
__host__ __device__ constexpr int seg_sub(int units, int lanes) {  // entries per staged sub-batch (<= lanes)
  int p = (SEG_PBASE / units) > 0 ? (SEG_PBASE / units) : 1;
  return p < lanes ? p : lanes;
}
// dynamic shared memory of the tiles kernel: per lane group 2 stages x P entries x (partner row + own row)
// (+ a pad that staggers the groups of a quarter-warp over the shared-memory banks)
__host__ __device__ constexpr int seg_region_floats(int dim, int lanes, int units, int vec) {
  const int base = 2 * seg_sub(units, lanes) * 2 * dim;
  return base + ((base % 32 == 0 && lanes * vec < 32) ? lanes * vec : 0);
}
inline size_t seg_smem_bytes(int dim, int lanes, int units, int vec) {
  return (size_t)(SEG_THREADS / lanes) * seg_region_floats(dim, lanes, units, vec) * sizeof(float);
}

// Sum of P per-lane partial values across the L lanes of a group, P <= L, in log2(L) exchange steps: the first
// log2(P) steps halve the number of values a lane carries (a lane whose bit `off` is set keeps the upper half),
// the rest are butterflies.  Afterwards v[0] of lane l is the complete sum of value number l >> (log2 L - log2 P).
// The order of the additions is a fixed function of (L, P): both tables' tiles reduce a dot product identically.
template <int L, int P>
__device__ __forceinline__ float reduce_transpose(float (&v)[P], int lane, unsigned gmask) {
  int n = P;
#pragma unroll
  for (int off = L / 2; off >= 1; off >>= 1) {
    if (n > 1) {
      n >>= 1;
      const bool upper = lane & off;
#pragma unroll
      for (int i = 0; i < P / 2; ++i) {
        if (i < n) {
          const float send = upper ? v[i] : v[i + n];
          const float keep = upper ? v[i + n] : v[i];
          v[i] = add_rn(keep, __shfl_xor_sync(gmask, send, off, L));
        }
      }
    } else {
      v[0] = add_rn(v[0], __shfl_xor_sync(gmask, v[0], off, L));
    }
  }
  return v[0];
}
__host__ __device__ constexpr int ilog2(int x) { return x <= 1 ? 0 : 1 + ilog2(x >> 1); }

// UNITS = per-lane units (of VEC floats) needed to cover a row with L lanes.  A lane group walks its tile in
// sub-batches of P entries, double-buffered in shared memory: while sub-batch i is consumed, the partner rows of
// sub-batch i+1 (and the own rows of its entries that open a run) are in flight -- otherwise a tile is a chain of 32
// dependent gather latencies.  Everything that is per ENTRY rather than per float (ids, ratings, biases, the logit,
// d cost/d logits) is computed lane-parallel -- lane j works for entry j of the chunk -- and only the error is
// broadcast: a warp spends its instructions on the rows, not on 32 copies of the scalar work.
// GENERIC = false: README model (plain dot, Adam); true: any flags (|v|, SGD scaling, FM rows).
template <int VEC, int L, int UNITS, bool FUSED, bool GENERIC>
__global__ void __launch_bounds__(SEG_THREADS) segsum_tiles_kernel(SegSide su, SegSide si, FwdArgs fw,
                                                                   const tfr_opt_scalars* __restrict__ opt,
                                                                   const float* __restrict__ err, int64_t B, int dim,
                                                                   int n_tiles, int tile) {
  pdl_wait();                // the previous step's table pass (tables, step scalars) is complete
  pdl_launch_dependents();   // the fix-up's CTAs may become resident as this grid drains
  TlScope tl_scope(opt, TFR_TL_TILES);
  constexpr int P = seg_sub(UNITS, L);
  constexpr int SH = ilog2(L) - ilog2(P);  // lane l ends up with the dot of entry l >> SH of the sub-batch
  extern __shared__ __align__(16) float s_rows[];
  const SegSide s = blockIdx.y ? si : su;
  const int lane = threadIdx.x & (L - 1);
  // sub-warp groups: all shuffles below are confined to the group (width = L) and use the group's own mask
  const int gshift = (threadIdx.x & 31) & ~(L - 1);
  const unsigned gmask = (L == 32) ? 0xffffffffu : (((1u << L) - 1u) << gshift);
  float* const stage = s_rows + (size_t)(threadIdx.x / L) * seg_region_floats(dim, L, UNITS, VEC);  // [2][P][partner | own][dim]
  const int n_units = dim / VEC;
  const int flags = opt->flags;
  const float reg = opt->reg;
  const bool abs_item = GENERIC && (flags & TFR_ABS_ITEM);
  const bool sgd = GENERIC && (flags & TFR_OPT_SGD);
  const bool fm = GENERIC && s.xval != nullptr;
  const bool reg_bias = flags & TFR_REG_BIAS;
  const float lr = opt->lr;
  const uint32_t stamp = (uint32_t)opt->global_step;
  float mu = 0.0f;
  if constexpr (FUSED) mu = *fw.mu;
  float err_acc = 0.0f;   // FUSED, user side: this lane's share of sum_b e_b and of the squared error
  double se_acc = 0.0;

  const int64_t n_groups = (int64_t)gridDim.x * (SEG_THREADS / L);
  for (int64_t t = (int64_t)blockIdx.x * (SEG_THREADS / L) + threadIdx.x / L; t < n_tiles; t += n_groups) {
    const int64_t k0 = t * tile;
    const int64_t k1 = min(k0 + tile, B);
    const int32_t prev_id = k0 > 0 ? s.sid[k0 - 1] : -1;
    const int32_t next_id = k1 < B ? s.sid[k1] : -1;
    if (s.sid[k0] >= s.n_rows) {  // the whole tile belongs to other ranks
      if (lane == 0) s.kind[t] = 0;
      continue;
    }

    Acc<VEC> acc[UNITS], own[UNITS], own_a[UNITS];  // own: run's row (gradient walk); own_a: same, dot walk
    float acc_b = 0.0f, own_b = 0.0f;
    int32_t cur = -1;
    int64_t run_start = k0;
    uint8_t kind = 0;

    auto flush = [&](int64_t k_end) {  // the run [run_start, k_end) of id `cur` is over (within this tile)
      const bool starts = run_start > k0 || cur != prev_id;
      const bool ends = k_end < k1 || cur != next_id;
      float* dst;
      float* dst_b;
      if (starts && ends) { dst = s.gsum + (size_t)run_start * dim; dst_b = s.gsum_b + run_start; }
      else if (!starts)   { dst = s.cont + (size_t)t * dim;         dst_b = s.cont_b + t; if (!ends) kind |= TILE_MID; }
      else                { dst = s.tail + (size_t)t * dim;         dst_b = s.tail_b + t; kind |= TILE_START; }
#pragma unroll
      for (int q = 0; q < UNITS; ++q) {
        const int unit = lane + q * L;
        if (unit < n_units) store_units<VEC>(dst, unit, acc[q]);
      }
      if (lane == 0) {
        *dst_b = acc_b;
        if (starts && ends) s.slot[cur] = pack_slot(stamp, run_start);
      }
    };

    int32_t carry_id = -1;  // id of the entry in front of the current chunk (inside this tile)
    bool done = false;
    for (int64_t kb = k0; kb < k1 && !done; kb += L) {
      // ---- lane j of the group works for entry kb + j: ids first (the row copies need them) ----
      const int64_t k = kb + lane;
      int32_t my_id = -1, my_partner = 0, my_b = 0;
      bool mine = false;
      if (k < k1) {
        my_id = s.sid[k];
        my_b = s.spos[k];
        mine = my_id < s.n_rows;
        if (mine) {
          if (fm) my_partner = s.rowof[my_b];  // FM: the "partner" of a non-zero is its CSR row's sums
          else my_partner = s.partner ? s.partner[my_b] : my_b;  // row-sharded mode: rows gathered by position
        }
      }
      int32_t before = __shfl_up_sync(gmask, my_id, 1, L);
      if (lane == 0) before = carry_id;
      // bit j: entry j opens a run (as far as this tile is concerned) / is a row of this rank
      const unsigned newmask = (__ballot_sync(gmask, my_id != before) >> gshift);
      const unsigned minemask = (__ballot_sync(gmask, mine) >> gshift) & (L == 32 ? 0xffffffffu : ((1u << L) - 1u));
      int cnt = (int)min((int64_t)L, k1 - kb);
      carry_id = __shfl_sync(gmask, my_id, cnt - 1, L);
      const int n_mine = __popc(minemask);  // sorted: the rows of other ranks are at the end
      if (n_mine < cnt) { cnt = n_mine; done = true; }

      // request the rows of sub-batch sb into stage sb & 1 (always commits a group, possibly an empty one)
      auto request = [&](int sb) {
        float* st = stage + (size_t)(sb & 1) * (P * 2) * dim;
#pragma unroll 1
        for (int jj = 0; jj < P; ++jj) {  // not unrolled: the copies need no registers, keep the code small
          const int j = sb * P + jj;
          if (j < cnt) {
            const int32_t pid = __shfl_sync(gmask, my_partner, j, L);
            const float* prow = s.partner_feat + (size_t)pid * s.partner_stride;
#pragma unroll
            for (int q = 0; q < UNITS; ++q) {
              const int unit = lane + q * L;
              if (unit < n_units) cp_async_units<VEC>(st + (size_t)(jj * 2) * dim + unit * VEC, prow + unit * VEC);
            }
            if ((newmask >> j) & 1u) {
              const int32_t id = __shfl_sync(gmask, my_id, j, L);
              const float* orow = s.own_feat + (size_t)id * s.own_stride;
#pragma unroll
              for (int q = 0; q < UNITS; ++q) {
                const int unit = lane + q * L;
                if (unit < n_units) cp_async_units<VEC>(st + (size_t)(jj * 2 + 1) * dim + unit * VEC, orow + unit * VEC);
              }
            }
          }
        }
        cp_async_commit();
      };
      const int n_sub = (cnt + P - 1) / P;
      request(0);
      if (n_sub > 1) request(1);
      // ---- the entries' scalars, fetched while the first rows are in flight ----
      float my_e = 0.0f, my_x = 1.0f, my_ob = 0.0f, my_pb = 0.0f, my_rate = 0.0f;
      if (mine) {
        if (fm) {
          my_e = err[my_partner];
          my_x = s.xval[my_b];
        } else if constexpr (FUSED) {
          my_rate = fw.rates[my_b];
          my_pb = ld_gather_f1(s.partner_bias + my_partner);
        } else {
          my_e = err[my_b];
        }
        if (FUSED || reg_bias) my_ob = ld_gather_f1(s.own_bias + my_id);
      }

      for (int sb = 0; sb < n_sub; ++sb) {
        if (sb + 1 < n_sub) cp_async_wait<1>(); else cp_async_wait<0>();
        __syncwarp(gmask);
        const float* st = stage + (size_t)(sb & 1) * (P * 2) * dim;
        const int jend = min(cnt, (sb + 1) * P);
        if constexpr (FUSED) {
          // ops.py:44-47 on the rows this tile holds anyway: P partial dot products per lane, one transposing
          // reduction, then lane j finishes the logit and d cost/d logits of ITS entry
          float part[P];
#pragma unroll
          for (int jj = 0; jj < P; ++jj) {
            part[jj] = 0.0f;
            const int j = sb * P + jj;
            if (j < jend) {
              if ((newmask >> j) & 1u) {
#pragma unroll
                for (int q = 0; q < UNITS; ++q) {
                  const int unit = lane + q * L;
                  if (unit < n_units) own_a[q] = lds_units<VEC>(st + (size_t)(jj * 2 + 1) * dim, unit);
                }
              }
#pragma unroll
              for (int q = 0; q < UNITS; ++q) {
                const int unit = lane + q * L;
                if (unit < n_units) {
                  const Acc<VEC> p = lds_units<VEC>(st + (size_t)(jj * 2) * dim, unit);
#pragma unroll
                  for (int c = 0; c < VEC; ++c) {
                    float vv = s.is_item ? own_a[q].v[c] : p.v[c];   // the item row (|v| in the fork's model)
                    const float uu = s.is_item ? p.v[c] : own_a[q].v[c];
                    if (abs_item) vv = fabsf(vv);
                    part[jj] = add_rn(part[jj], mul_rn(uu, vv));
                  }
                }
              }
            }
          }
          const float red = reduce_transpose<L, P>(part, lane, gmask);
          const int jm = lane - sb * P;  // my entry's index in this sub-batch, if it is in it
          const float dot = __shfl_sync(gmask, red, (jm & (P - 1)) << SH, L);
          if (jm >= 0 && jm < P && lane < jend) {
            float x = add_rn(dot, mu);                          // ops.py:45
            x = add_rn(x, s.is_item ? my_pb : my_ob);           // ops.py:46  + bias_users
            x = add_rn(x, s.is_item ? my_ob : my_pb);           // ops.py:47  + bias_items
            my_e = dloss(flags, x, my_rate);
            if (!s.is_item) {
              const float inf = (flags & TFR_LOSS_SIGMOID_CE) ? rintf(sigmoid_tf(x)) : x;
              if (fw.logits) fw.logits[my_b] = x;
              if (fw.infer) fw.infer[my_b] = inf;
              err_acc = add_rn(err_acc, my_e);
              const double dse = (double)my_rate - (double)inf;
              se_acc += dse * dse;
            }
          }
        }
        // ---- gradient walk: entries in order, runs flushed as they end ----
#pragma unroll 1
        for (int j = sb * P; j < jend; ++j) {
          const int jj = j - sb * P;
          const float e = __shfl_sync(gmask, my_e, j, L);
          if ((newmask >> j) & 1u) {
            if (cur >= 0) flush(kb + j);
            cur = __shfl_sync(gmask, my_id, j, L);
            run_start = kb + j;
#pragma unroll
            for (int q = 0; q < UNITS; ++q) {
              const int unit = lane + q * L;
              if (unit < n_units) own[q] = lds_units<VEC>(st + (size_t)(jj * 2 + 1) * dim, unit);
#pragma unroll
              for (int c = 0; c < VEC; ++c) acc[q].v[c] = 0.0f;
            }
            own_b = reg_bias ? __shfl_sync(gmask, my_ob, j, L) : 0.0f;
            acc_b = 0.0f;
          }
          float xv = 1.0f;
          if (fm) xv = __shfl_sync(gmask, my_x, j, L);
#pragma unroll
          for (int q = 0; q < UNITS; ++q) {
            const int unit = lane + q * L;
            if (unit < n_units) {
              const Acc<VEC> p = lds_units<VEC>(st + (size_t)(jj * 2) * dim, unit);
#pragma unroll
              for (int c = 0; c < VEC; ++c) {
                float g;
                if (fm) {
                  const float tt = sub_rn(p.v[c], mul_rn(own[q].v[c], xv));
                  g = mul_rn(e, mul_rn(xv, tt));
                } else if (!s.is_item) {
                  g = mul_rn(e, abs_item ? fabsf(p.v[c]) : p.v[c]);
                } else {
                  g = mul_rn(e, p.v[c]);
                  if (abs_item) {
                    const float o = own[q].v[c];
                    g = mul_rn(g, (o > 0.0f) ? 1.0f : ((o < 0.0f) ? -1.0f : 0.0f));
                  }
                }
                g = add_rn(g, mul_rn(reg, own[q].v[c]));
                if (sgd) g = mul_rn(lr, g);
                acc[q].v[c] = add_rn(acc[q].v[c], g);
              }
            }
          }
          float gb = fm ? mul_rn(e, xv) : e;
          if (reg_bias) gb = add_rn(gb, mul_rn(reg, own_b));
          if (sgd) gb = mul_rn(lr, gb);
          acc_b = add_rn(acc_b, gb);
        }
        __syncwarp(gmask);  // the stage is free again
        if (sb + 2 < n_sub) request(sb + 2);
      }
      if (done && cur >= 0) {  // the rest of the tile belongs to other ranks
        flush(kb + cnt);
        cur = -1;
      }
    }
    if (cur >= 0) flush(k1);
    if (lane == 0) {
      s.kind[t] = kind;
      if (kind & TILE_START) {  // a run begins here and goes on: queue its fix-up
        const uint32_t at = atomicAdd(s.fix_count, 1u);
        if (at < (uint32_t)n_tiles) s.fix_list[at] = (int32_t)t;
      }
    }
  }

  if constexpr (FUSED) {
    // fixed-order block reduction of the user side's sums (as svd_forward_kernel does)
    if (blockIdx.y == 0) {
      __shared__ float s_err[SEG_THREADS];
      __shared__ double s_se[SEG_THREADS];
      s_err[threadIdx.x] = err_acc;
      s_se[threadIdx.x] = se_acc;
      __syncthreads();
      if (threadIdx.x < 32) {
        float a = 0.0f;
        double d = 0.0;
        for (int j = threadIdx.x; j < SEG_THREADS; j += 32) { a = add_rn(a, s_err[j]); d += s_se[j]; }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
          a = add_rn(a, __shfl_xor_sync(0xffffffffu, a, o));
          d += __shfl_xor_sync(0xffffffffu, d, o);
        }
        if (threadIdx.x == 0) { fw.partials[blockIdx.x] = a; fw.se_partials[blockIdx.x] = d; }
      }
    }
  }
}

// Fix-up: a persistent grid walks the work list of TILE_START tiles.  A run that begins in tile t0 and ends in
// tile t1 has the partial sums tail[t0], cont[t0+1], ..., cont[t1]; tiles t0+1..t1-1 are TILE_MID.
//  * Short chains (t1 - t0 <= FIX_SHORT, almost all of them) are summed by ONE WARP each, in tile order, eight
//    partial rows in flight: no block barrier, thousands of chains side by side.
//  * Long chains (a hot row with thousands of occurrences) are parked in the CTA's shared list and summed afterwards
//    by the whole CTA: G thread groups add the cont rows j = g, g+G, g+2G, ... (each in increasing j), then
//    tail + p_0 + ... + p_{G-1}.
// Both are fixed functions of (t0, t1): the result does not depend on the order of the list or on which warp /
// CTA picked an entry up.
constexpr int FIX_THREADS = 256;
constexpr int FIX_SHORT = 32;      // partial rows one warp sums on its own
constexpr int FIX_LONG_CAP = 32;   // long chains a CTA can park (more: the warp sums them itself, slowly)

template <int VEC>
__global__ void __launch_bounds__(FIX_THREADS, 3) segsum_fixup_kernel(SegSide su, SegSide si, const tfr_opt_scalars* __restrict__ opt,
                                                                   uint32_t* counters, int64_t B, int dim, int n_tiles,
                                                                   int tile, int cw, float* fold_err, double* fold_se,
                                                                   int fold_n) {
  pdl_wait();                // the tiles kernel's partial rows and work lists are complete
  pdl_launch_dependents();   // the table pass's CTAs may become resident as this grid drains
  TlScope tl_scope(opt, TFR_TL_FIXUP, true);
  extern __shared__ float s_part[];  // [G][dim] (+ [G] bias partials)
  __shared__ int s_long[FIX_LONG_CAP][2];
  __shared__ int s_nlong;
  const SegSide s = blockIdx.y ? si : su;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int n_units = dim / VEC;
  const uint32_t stamp = (uint32_t)opt->global_step;
  const uint32_t n_fix = min(*s.fix_count, (uint32_t)n_tiles);
  if (threadIdx.x == 0) s_nlong = 0;
  __syncthreads();
  // One warp folds the fused forward's per-CTA partial sums (complete: the tiles kernel wrote them) into
  // [TFR_MAX_PARTIALS] -- in the order and with the adds of finish_step_scalars -- BESIDE the chains, so that the
  // step's end (the table pass's last CTA) reads one value instead of hundreds behind its tail.
  if (fold_n > 0 && blockIdx.y == 0 && blockIdx.x == gridDim.x - 1 && warp == FIX_THREADS / 32 - 1) {
    float a = 0.0f;
    double se = 0.0;
    for (int j = lane; j < fold_n; j += 32) { a = add_rn(a, fold_err[j]); se += fold_se[j]; }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      a = add_rn(a, __shfl_xor_sync(0xffffffffu, a, o));
      se += __shfl_xor_sync(0xffffffffu, se, o);
    }
    if (lane == 0) { fold_err[TFR_MAX_PARTIALS] = a; fold_se[TFR_MAX_PARTIALS] = se; }
  }

  // t1 = first tile after t0 that is not TILE_MID; head = sorted index of the run's first entry (ids are sorted:
  // the run is the suffix of tile t0)
  static_assert(SEG_TILE_MAX <= 32, "one warp looks at one tile");
  auto chain_of = [&](int t0, int& t1, int64_t& head) {
    const int64_t k0 = (int64_t)t0 * tile, k1 = min(k0 + tile, B);
    const int32_t last = s.sid[k1 - 1];
    const int64_t k = k0 + lane;
    const unsigned same = __ballot_sync(0xffffffffu, k < k1 && s.sid[k] == last);
    head = k0 + __ffs(same) - 1;
    t1 = -1;
    for (int base = t0 + 1; t1 < 0; base += 128) {  // four loads per lane in flight: a hot row's chain is hundreds of tiles
      bool stop[4];
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        const int tt = base + 32 * r + lane;
        stop[r] = tt >= n_tiles || !(s.kind[tt] & TILE_MID);
      }
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        const unsigned m = __ballot_sync(0xffffffffu, stop[r]);
        if (m && t1 < 0) t1 = base + 32 * r + __ffs(m) - 1;
      }
    }
    t1 = min(t1, n_tiles - 1);
  };
  // the chain's bias partials, summed by one warp: lane l adds cont_b[t0+1+l], cont_b[t0+1+l+32], ... then a
  // butterfly over the lanes -- a fixed function of (t0, t1), and 32 loads in flight instead of a serial chain
  auto warp_bias_sum = [&](int t0, int t1) {
    float part = 0.0f;
    for (int tt = t0 + 1 + lane; tt <= t1; tt += 32) part = add_rn(part, s.cont_b[tt]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) part = add_rn(part, __shfl_xor_sync(0xffffffffu, part, o));
    return add_rn(s.tail_b[t0], part);
  };
  // one warp: tail[t0] + cont[t0+1] + ... + cont[t1], in that order, four rows in flight
  auto warp_chain = [&](int t0, int t1, int64_t head) {
    for (int unit = lane; unit < n_units; unit += 32) {
      Acc<VEC> acc = load_units<VEC>(s.tail + (size_t)t0 * dim, unit);
      for (int tt = t0 + 1; tt <= t1; tt += 4) {
        Acc<VEC> x[4];
#pragma unroll
        for (int r = 0; r < 4; ++r)
          if (tt + r <= t1) x[r] = load_units<VEC>(s.cont + (size_t)(tt + r) * dim, unit);
#pragma unroll
        for (int r = 0; r < 4; ++r)
          if (tt + r <= t1) {
#pragma unroll
            for (int q = 0; q < VEC; ++q) acc.v[q] = add_rn(acc.v[q], x[r].v[q]);
          }
      }
      store_units<VEC>(s.gsum + (size_t)head * dim, unit, acc);
    }
    const float tot = warp_bias_sum(t0, t1);
    if (lane == 0) {
      s.gsum_b[head] = tot;
      s.slot[s.sid[head]] = pack_slot(stamp, head);
    }
  };

  const uint32_t n_warps = gridDim.x * (FIX_THREADS / 32);
  for (uint32_t w = blockIdx.x * (FIX_THREADS / 32) + warp; w < n_fix; w += n_warps) {
    const int t0 = s.fix_list[w];
    int t1;
    int64_t head;
    chain_of(t0, t1, head);
    if (t1 - t0 <= FIX_SHORT) {
      warp_chain(t0, t1, head);
    } else {
      int at = FIX_LONG_CAP;
      if (lane == 0) at = atomicAdd(&s_nlong, 1);
      at = __shfl_sync(0xffffffffu, at, 0);
      if (at < FIX_LONG_CAP) {
        if (lane == 0) { s_long[at][0] = t0; s_long[at][1] = t1; }
      } else {
        warp_chain(t0, t1, head);  // the CTA's list is full: correct, just not parallel
      }
    }
  }
  __syncthreads();

  // ---- the parked long chains, one after the other, by the whole CTA ----
  const int n_long = min(s_nlong, FIX_LONG_CAP);
  const int G = FIX_THREADS / cw;
  const int g = threadIdx.x / cw, c = threadIdx.x % cw;
  for (int e = 0; e < n_long; ++e) {
    const int t0 = s_long[e][0], t1 = s_long[e][1];
    for (int unit = c; unit < n_units; unit += cw) {
      Acc<VEC> acc;
#pragma unroll
      for (int q = 0; q < VEC; ++q) acc.v[q] = 0.0f;
      for (int tt = t0 + 1 + g; tt <= t1; tt += 8 * G) {  // eight rows in flight, added in increasing tile order
        Acc<VEC> x[8];
#pragma unroll
        for (int r = 0; r < 8; ++r)
          if (tt + r * G <= t1) x[r] = load_units<VEC>(s.cont + (size_t)(tt + r * G) * dim, unit);
#pragma unroll
        for (int r = 0; r < 8; ++r)
          if (tt + r * G <= t1) {
#pragma unroll
            for (int q = 0; q < VEC; ++q) acc.v[q] = add_rn(acc.v[q], x[r].v[q]);
          }
      }
#pragma unroll
      for (int q = 0; q < VEC; ++q) s_part[(size_t)g * dim + unit * VEC + q] = acc.v[q];
    }
    float bias_tot = 0.0f;
    if (warp == FIX_THREADS / 32 - 1) bias_tot = warp_bias_sum(t0, t1);  // the last warp, beside its row work
    __syncthreads();
    // head of the run inside t0 (every thread finds it for itself: the tile's ids are one cached line)
    const int64_t k0 = (int64_t)t0 * tile, k1 = min(k0 + tile, B);
    const int32_t id = s.sid[k1 - 1];
    int64_t a = k1 - 1;
    while (a > k0 && s.sid[a - 1] == id) --a;
    for (int col = threadIdx.x; col < dim; col += FIX_THREADS) {
      float tot = s.tail[(size_t)t0 * dim + col];
      for (int gg = 0; gg < G; ++gg) tot = add_rn(tot, s_part[(size_t)gg * dim + col]);
      s.gsum[(size_t)a * dim + col] = tot;
    }
    if (threadIdx.x == FIX_THREADS - 32) {  // lane 0 of the warp that summed the bias partials
      s.gsum_b[a] = bias_tot;
      s.slot[id] = pack_slot(stamp, a);
    }
    __syncthreads();  // s_part is reused by the next long chain
  }
  // the last CTA to finish empties the work lists for the next use of this workspace
  if (threadIdx.x == 0) {
    __threadfence();
    if (atomicAdd(counters + 2, 1u) == gridDim.x * gridDim.y - 1) { counters[0] = 0; counters[1] = 0; counters[2] = 0; }
  }
}

}  // namespace tfr

using namespace tfr;

namespace tfr {
// Lane-group geometry of the tiles kernel: few lanes per row, several units (of VEC floats) per lane -- a warp then
// walks 32/L tiles at once and everything that is per entry rather than per float (shuffles, branches, addresses) is
// paid once per warp instruction for 32/L entries.  UNITS is 1, 2, 4, 8 or 16 (rounded up; surplus units are masked);
// 8 and 16 only occur for rows of 129..511 floats with dim % 4 != 0 (32 lanes of one float each).
struct SegGeom {
  int vec, lanes, units;
};
// Every (VEC, L, UNITS) the tiles kernel is instantiated for: launch_segsum dispatches over this list, and for every dim
// of 1..512 seg_geom returns a member of it, whatever SEG_MAX_UNITS is (tests/test_geometry.py mirrors both).
#define TFR_SEG_CASES(X)                                                                                            \
  /* default geometry (<= 4 units per lane): L = 1 for rows of up to 4 units, then UNITS = 4 */                     \
  X(4, 1, 1) X(4, 1, 2) X(4, 1, 4) X(4, 2, 4) X(4, 4, 4) X(4, 8, 4) X(4, 16, 4) X(4, 32, 4)                         \
  X(1, 1, 1) X(1, 1, 2) X(1, 1, 4) X(1, 2, 4) X(1, 4, 4) X(1, 8, 4) X(1, 16, 4) X(1, 32, 4)                         \
  /* one unit per lane (rows of fewer than 32 units), two units (rows of 33..64 floats, dim % 4 != 0) */            \
  X(4, 2, 1) X(4, 4, 1) X(4, 8, 1) X(4, 16, 1) X(4, 32, 1)                                                          \
  X(1, 2, 1) X(1, 4, 1) X(1, 8, 1) X(1, 16, 1) X(1, 32, 1)                                                          \
  X(1, 32, 2) X(4, 16, 2) X(1, 8, 2)                                                                                \
  /* rows of 129..511 floats, dim % 4 != 0 */                                                                       \
  X(1, 32, 8) X(1, 32, 16)
static bool seg_case_exists(const SegGeom& g) {
#define TFR_SEG_HAS(V, LL, UU) if (g.vec == V && g.lanes == LL && g.units == UU) return true;
  TFR_SEG_CASES(TFR_SEG_HAS)
#undef TFR_SEG_HAS
  return false;
}
static SegGeom seg_geom_max_units(int dim, int forced) {
  SegGeom g;
  g.vec = (dim % 4 == 0) ? 4 : 1;
  const int n_units = dim / g.vec;
  // measured (B200): a tile is a chain of dependent latencies, so short rows want as many lanes as they have units
  // (ML-1M shape, dim 15: 25 us with 16 lanes against 42 us with 4); rows of >= 32 units do better with 4 units per
  // lane (dim 128: 48 us with 8 lanes against 54 us with 32)
  const int max_units = forced ? forced : (n_units >= 32 ? 4 : 1);
  int l = 1;
  while (l * max_units < n_units && l < 32) l <<= 1;
  g.lanes = l;
  const int u = (n_units + l - 1) / l;
  g.units = u <= 1 ? 1 : u <= 2 ? 2 : u <= 4 ? 4 : u <= 8 ? 8 : u <= 16 ? 16 : u;
  return g;
}
static SegGeom seg_geom(int dim) {
  int forced = tune(TUNE_SEG_MAX_UNITS);  // experiments: force 1, 2 or 4 units per lane
  if (forced != 1 && forced != 2 && forced != 4) forced = 0;
  const SegGeom g = seg_geom_max_units(dim, forced);
  // a forced unit count that has no instantiation for this dim falls back to the default geometry HERE, so that the
  // tile size, the fused forward's partial count (segsum_grid_x) and the launch all see the same geometry
  if (forced && !seg_case_exists(g)) return seg_geom_max_units(dim, 0);
  return g;
}
// Tile size: a lane group walks its tile entry by entry (a chain of dependent instructions), so the kernel's time is
// one tile's latency times the number of waves.  Pick the largest tile of 32 / 16 / 8 entries that still gives every SM
// a dozen warps; smaller tiles mean more runs crossing tiles, i.e. more fix-up work.
int seg_tile(int64_t B, int dim) {
  const int forced = tune(TUNE_SEG_TILE);
  if (forced == 8 || forced == 16 || forced == 32) return forced;
  const SegGeom g = seg_geom(dim);
  const int64_t groups_per_warp = 32 / g.lanes;
  const int64_t want = (int64_t)sm_count() * 12;
  for (int tile = 32; tile > 8; tile >>= 1) {
    const int64_t warps = (2 * ((B + tile - 1) / tile) + groups_per_warp - 1) / groups_per_warp;
    if (warps >= want) return tile;
  }
  return 8;
}
int segsum_grid_x(int dim, int64_t B) {  // CTAs per side = number of per-CTA partials of the fused forward
  const SegGeom g = seg_geom(dim);
  const int tile = seg_tile(B, dim);
  const int64_t n_tiles = (B + tile - 1) / tile;
  const int64_t groups_per_cta = SEG_THREADS / g.lanes;
  int64_t gx = (n_tiles + groups_per_cta - 1) / groups_per_cta;
  if (gx > TFR_MAX_PARTIALS) gx = TFR_MAX_PARTIALS;
  return (int)(gx < 1 ? 1 : gx);
}
}  // namespace tfr

// the tiles kernel stages rows in dynamic shared memory (32 KB per CTA at dim 128, up to 64 KB): opt in once per
// instantiation
int tfr::prep_tiles(const void* fn, size_t smem) {
  static std::mutex mu;
  static std::map<const void*, size_t> done;
  std::lock_guard<std::mutex> lock(mu);
  auto it = done.find(fn);
  if (it != done.end() && it->second >= smem) return TFR_OK;
  TFR_CUDA(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  // the same carve-out as every other kernel of the step (common.cuh: prep_kernel), so that no SM has to be
  // reconfigured between the pass, the tiles and the fix-up; TILES_CARVEOUT to experiment (100 = max shared)
  int carve = tune(TUNE_TILES_CARVEOUT);
  if (carve < 0) carve = tune(TUNE_SMEM_CARVEOUT);
  TFR_CUDA(cudaFuncSetAttribute(fn, cudaFuncAttributePreferredSharedMemoryCarveout, carve));
  done[fn] = smem;
  return TFR_OK;
}

// generic_flags: the HOST copy of the model flags has |v| or SGD set (the device copy drives the arithmetic, the host
// copy only selects the kernel variant: README model -> the lean one)
static int launch_segsum(const SegSide& su, const SegSide& si, int n_sides, const FwdArgs* fw,
                         const tfr_opt_scalars* opt, const float* err, int64_t B, int dim, bool generic_flags,
                         uint32_t* counters, cudaStream_t st) {
  const SegGeom g = seg_geom(dim);
  const int units = g.units;
  const int tile = seg_tile(B, dim);
  const int n_tiles = (int)((B + tile - 1) / tile);
  int cw = 1;
  while (cw < dim / g.vec && cw < FIX_THREADS) cw <<= 1;
  const int G = FIX_THREADS / cw;
  const size_t fix_smem = ((size_t)G * dim + G) * sizeof(float);
  // a warp per list entry: at most one entry per tile, so n_tiles / (warps per CTA) CTAs cover any list in one trip
  const int fix_warps = FIX_THREADS / 32;
  // (ncu: at 126 registers only two CTAs fit an SM and the grid ran in 3.5 waves; 64 registers spill and are slower;
  // bounded to 85 registers = three CTAs per SM, the grid capped at one resident wave for both sides)
  dim3 fix_grid((unsigned)min((n_tiles + fix_warps - 1) / fix_warps, 3 * sm_count() / n_sides), (unsigned)n_sides);
  dim3 grid((unsigned)segsum_grid_x(dim, B), (unsigned)n_sides);
  const FwdArgs none{};
  const bool pdl = tune(TUNE_PDL) != 0;
  const size_t smem = seg_smem_bytes(dim, g.lanes, units, g.vec);
  const bool generic = generic_flags || su.xval != nullptr;
#define TFR_SEG_LAUNCH(V, LL, UU, FU, GE)                                                                          \
  {                                                                                                                \
    if (int rc = prep_tiles((const void*)segsum_tiles_kernel<V, LL, UU, FU, GE>, smem)) return rc;                 \
    TFR_CUDA(launch_kernel(segsum_tiles_kernel<V, LL, UU, FU, GE>, grid, dim3(SEG_THREADS), smem, st, pdl, su, si,   \
                           fw ? *fw : none, opt, err, B, dim, n_tiles, tile));                                     \
  }
#define TFR_SEG_CASE(V, LL, UU)                                                                                   \
  if (g.vec == V && g.lanes == LL && units == UU) {                                                               \
    if (int rc = prep_tiles((const void*)segsum_fixup_kernel<V>, fix_smem)) return rc; /* same carve-out as the tiles */ \
    if (fw && generic) TFR_SEG_LAUNCH(V, LL, UU, true, true)                                                       \
    else if (fw && V == 4 && UU == 4 && chain_tiles_supported(LL, tile) && tune(TUNE_SEG_CHAIN)) {                  \
      if (int rc = launch_chain_tiles(su, si, *fw, opt, B, dim, n_tiles, tile, LL, grid, pdl, st)) return rc;      \
    } else if (fw) TFR_SEG_LAUNCH(V, LL, UU, true, false)                                                          \
    else if (generic) TFR_SEG_LAUNCH(V, LL, UU, false, true)                                                       \
    else TFR_SEG_LAUNCH(V, LL, UU, false, false)                                                                   \
    TFR_LAUNCH_CHECK();                                                                                            \
    TFR_CUDA(launch_kernel(segsum_fixup_kernel<V>, fix_grid, dim3(FIX_THREADS), fix_smem, st, pdl, su, si, opt, counters, \
                           B, dim, n_tiles, tile, cw, fw ? fw->partials : nullptr, fw ? fw->se_partials : nullptr,  \
                           fw ? (int)grid.x : 0));                                                                  \
    return TFR_OK;                                                                                                 \
  }
  TFR_SEG_CASES(TFR_SEG_CASE)
#undef TFR_SEG_CASE
#undef TFR_SEG_LAUNCH
  set_error("unsupported dim %d (vec %d lanes %d units %d): the segment sums take rows of 1 to 512 floats", dim, g.vec,
            g.lanes, units);
  return TFR_ERR_INVALID;
}

static void svd_sides(const tfr_svd_tables* t, const int32_t* users, const int32_t* items, const tfr_svd_step_ws* ws,
                      SegSide* su, SegSide* si) {
  const bool gathered = t->g_user_feat != nullptr;
  const int64_t fs = t->feat_stride ? t->feat_stride : t->dim;
  const int64_t ps = gathered ? (t->g_stride ? t->g_stride : (int64_t)t->dim) : fs;
  *su = SegSide{ws->su_ids, ws->su_pos, gathered ? nullptr : items, t->user_feat,
                gathered ? t->g_item_feat : t->item_feat, fs, ps, t->user_bias, gathered ? t->g_item_bias : t->item_bias,
                ws->gsum_uf, ws->gsum_ub, ws->cont_uf, ws->cont_ub, ws->tail_uf, ws->tail_ub, ws->kind_u, ws->fix_list_u,
                ws->fix_count, t->user_slot, t->user_num, nullptr, nullptr, 0};
  *si = SegSide{ws->si_ids, ws->si_pos, gathered ? nullptr : users, t->item_feat,
                gathered ? t->g_user_feat : t->user_feat, fs, ps, t->item_bias, gathered ? t->g_user_bias : t->user_bias,
                ws->gsum_if, ws->gsum_ib, ws->cont_if, ws->cont_ib, ws->tail_if, ws->tail_ib, ws->kind_i, ws->fix_list_i,
                ws->fix_count + 1, t->item_slot, t->item_num, nullptr, nullptr, 1};
}

namespace tfr {
// flags_host < 0: unknown -> the generic kernel variant
int svd_segment_grads_impl(const tfr_svd_tables* t, const tfr_opt_scalars* opt, const int32_t* users,
                           const int32_t* items, int64_t B, const tfr_svd_step_ws* ws, int flags_host, void* stream) {
  TFR_CHECK_ARG(t && opt && users && items && ws && B > 0 && t->dim > 0 && t->user_slot && t->item_slot);
  TFR_CHECK_ARG(!t->g_user_feat || t->g_item_feat);
  SegSide su, si;
  svd_sides(t, users, items, ws, &su, &si);
  const bool generic = flags_host < 0 || (flags_host & (TFR_ABS_ITEM | TFR_OPT_SGD));
  return launch_segsum(su, si, 2, nullptr, opt, ws->err, B, t->dim, generic, ws->fix_count, (cudaStream_t)stream);
}
}  // namespace tfr

extern "C" int tfr_svd_segment_grads(const tfr_svd_tables* t, const tfr_opt_scalars* opt, const int32_t* users,
                                     const int32_t* items, int64_t B, const tfr_svd_step_ws* ws, void* stream) {
  return svd_segment_grads_impl(t, opt, users, items, B, ws, -1, stream);
}

// forward + d cost/d logits + ordered segment sums in ONE launch (+ the fix-up of runs that cross tiles): the rows a
// tile gathers for the gradient are the rows the forward needs.  Writes logits / infer (optional) and
// tfr_svd_fused_n_partials(dim, B) partial sums for tfr_svd_finish_step; ws->err is NOT written.
extern "C" int tfr_svd_fwd_segment_grads(const tfr_svd_tables* t, const tfr_opt_scalars* opt, const int32_t* users,
                                         const int32_t* items, const float* rates, int64_t B, float* logits,
                                         float* infer, int32_t flags, const tfr_svd_step_ws* ws, void* stream) {
  TFR_CHECK_ARG(t && opt && users && items && rates && ws && B > 0 && t->dim > 0 && t->user_slot && t->item_slot);
  TFR_CHECK_ARG(t->mu && t->user_bias && t->item_bias);
  TFR_CHECK_ARG(!t->g_user_feat);  // row-sharded mode: every rank needs every occurrence's error -> separate forward
  SegSide su, si;
  svd_sides(t, users, items, ws, &su, &si);
  const FwdArgs fw{t->mu, rates, logits, infer, ws->partials, ws->se_partials};
  const bool generic = flags & (TFR_ABS_ITEM | TFR_OPT_SGD);
  return launch_segsum(su, si, 2, &fw, opt, nullptr, B, t->dim, generic, ws->fix_count, (cudaStream_t)stream);
}

extern "C" int tfr_svd_fused_n_partials(int32_t dim, int64_t B) {
  if (dim <= 0 || B <= 0) return TFR_ERR_INVALID;
  return segsum_grid_x(dim, B);
}

// FM: one table of feature rows V [n_feat, dim] (+ linear weights W [n_feat]); the "batch" of the segment sums is
// the batch's nnz non-zeros.  ws must be carved for B = nnz (the user-side buffers are used).
extern "C" int tfr_fm_segment_grads(const float* V, const float* W, int64_t* slot, int32_t n_feat, int32_t dim,
                                    const tfr_opt_scalars* opt, const float* sums, const float* err,
                                    const float* xval, const int32_t* rowof, int64_t nnz, const tfr_svd_step_ws* ws,
                                    void* stream) {
  TFR_CHECK_ARG(V && W && slot && opt && sums && err && xval && rowof && ws && nnz > 0 && dim > 0 && n_feat > 0);
  SegSide sf{ws->su_ids, ws->su_pos, nullptr, V, sums, dim, dim, W, nullptr, ws->gsum_uf, ws->gsum_ub, ws->cont_uf, ws->cont_ub,
             ws->tail_uf, ws->tail_ub, ws->kind_u, ws->fix_list_u, ws->fix_count, slot, n_feat, xval, rowof, 0};
  return launch_segsum(sf, sf, 1, nullptr, opt, err, nnz, dim, true, ws->fix_count, (cudaStream_t)stream);
}
