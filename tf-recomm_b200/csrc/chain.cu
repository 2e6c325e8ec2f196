// The tiles kernel of the step's default path: forward + d cost/d logits + ordered segment sums for the README model
// (plain dot, Adam) with rows of dim % 4 == 0 floats, four float4 units per lane.  It computes exactly what
// segsum_tiles_kernel<4, L, 4, true, false> computes -- the same tiles, the same in-order fold inside a tile, the same
// dot-product tree, the same per-CTA partial sums of e -- with fewer instructions per entry:
//  * the entries' scalars (row ids, batch position, biases, rating) are fetched lane-parallel once per tile and
//    parked in shared memory; every lane of the group then reads entry j's from there and finishes its logit and
//    d cost/d logits itself (the dot product reaches every lane anyway), so the walk broadcasts nothing but the dot;
//  * the walk is branch-free on run boundaries: the own row is copied for every entry (a repeated row is an L1 hit),
//    a run's sum restarts from +0 by a select, and only the store of a finished run is conditional;
//  * the gradient's adds are paired fp32 (FADD2), each half the same IEEE rounding as add_rn.
// Rows are staged as in segsum_tiles_kernel: cp.async into a two-slot ring per lane group, entry j + 1's in flight
// while j is consumed.  Partial rows, tile kinds and work lists are segsum.cu's: its fix-up finishes the runs that
// cross tiles.
#include "segsum.cuh"

namespace tfr {

__device__ __forceinline__ void cp_async_16(float4* smem_dst, const float* gsrc) {
  const uint32_t d = (uint32_t)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit_group() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait_group() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }
// paired fp32 add, each half one IEEE rounding like add_rn.  Only adds are paired: ptxas contracts a paired multiply
// (even one written as fma(a, b, -0)) into the paired add that consumes it, which would round once instead of twice;
// the scalar mul_rn is never contracted.
__device__ __forceinline__ float2 add2(float2 a, float2 b) {
  float2 r;
  asm("{.reg .b64 ra, rb, rd;\n\tmov.b64 ra, {%2, %3};\n\tmov.b64 rb, {%4, %5};\n\t"
      "add.rn.f32x2 rd, ra, rb;\n\tmov.b64 {%0, %1}, rd;}"
      : "=f"(r.x), "=f"(r.y) : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y));
  return r;
}
__device__ __forceinline__ float2 mul2(float2 a, float2 b) { return make_float2(mul_rn(a.x, b.x), mul_rn(a.y, b.y)); }

struct Row4 {  // one lane's four float4 units of a row, as pairs
  float2 v[4][2];
};

// L lanes per row, lane l holds the units l, l + L, l + 2L, l + 3L of 4 floats (units >= dim / 4 are absent);
// T entries per tile.  One lane group per tile, SEG_THREADS / L groups per CTA, tiles assigned as in segsum_tiles_kernel.
// per lane group: the row slots and the scalars of the tile's entries (written lane-parallel, then read by every lane of
// the group per entry: no shuffles inside the walk but the dot product's own)
template <int L, int T>
struct ChainSmem {
  float4 rows[SEG_THREADS / L][2][2][4 * L];  // [slot][partner row | own row][unit]
  int32_t ids[SEG_THREADS / L][6][T];  // partner row, own row, batch position; own bias, partner bias, rating (bits)
};

template <int L, int T, bool ITEM>
__device__ __forceinline__ void chain_tiles_side(const SegSide& s, const FwdArgs& fw,
                                                 const tfr_opt_scalars* __restrict__ opt, int64_t B, int dim,
                                                 int n_tiles, ChainSmem<L, T>& sm) {
  constexpr int NC = (T + L - 1) / L;  // chunks of L entries: lane l fetches the scalars of entries l, l + L, ...
  constexpr bool is_item = ITEM;
  const int lane = threadIdx.x & (L - 1);
  const int gshift = (threadIdx.x & 31) & ~(L - 1);
  const unsigned gmask = (L == 32) ? 0xffffffffu : (((1u << L) - 1u) << gshift);
  const int n_units = dim / 4;
  bool has[4];
#pragma unroll
  for (int q = 0; q < 4; ++q) has[q] = lane + q * L < n_units;
  const int flags = opt->flags;
  const float reg = opt->reg;
  const float2 reg2 = make_float2(reg, reg);
  const bool reg_bias = flags & TFR_REG_BIAS;
  const uint32_t stamp = (uint32_t)opt->global_step;
  const float mu = *fw.mu;
  float4 (&stage)[2][2][4 * L] = sm.rows[threadIdx.x / L];
  int32_t (&sc)[6][T] = sm.ids[threadIdx.x / L];
  float err_acc = 0.0f;  // user side: this lane's share of sum_b e_b and of the squared error (as segsum_tiles_kernel)
  double se_acc = 0.0;


  const int64_t n_groups = (int64_t)gridDim.x * (SEG_THREADS / L);
  for (int64_t t = (int64_t)blockIdx.x * (SEG_THREADS / L) + threadIdx.x / L; t < n_tiles; t += n_groups) {
    const int64_t k0 = t * T;
    const int n = (int)min((int64_t)T, B - k0);
    const int32_t prev_id = k0 > 0 ? s.sid[k0 - 1] : -1;
    const int32_t next_id = k0 + n < B ? s.sid[k0 + n] : -1;
    // (no rows of other ranks here: the fused step refuses row-sharded tables)

    __syncwarp(gmask);  // the group's previous tile has read its ids
    // ---- the entries' scalars, lane-parallel; bit j of newm: entry j opens a run (as far as this tile is concerned)
    unsigned newm = 0;
    int32_t carry = -1;  // id of the entry in front of the chunk
#pragma unroll
    for (int c = 0; c < NC; ++c) {
      const int j = c * L + lane;
      const bool valid = j < n;
      const int32_t id = valid ? s.sid[k0 + j] : -1;
      const int32_t pos = valid ? s.spos[k0 + j] : 0;
      int32_t before = __shfl_up_sync(gmask, id, 1, L);
      if (lane == 0) before = carry;
      carry = __shfl_sync(gmask, id, L - 1, L);
      const unsigned bits = (__ballot_sync(gmask, valid && id != before) >> gshift) &
                            (L == 32 ? 0xffffffffu : ((1u << L) - 1u));
      newm |= bits << (c * L);
      const int32_t part = valid ? s.partner[pos] : 0;
      if (j < T) {
        sc[0][j] = part;
        sc[1][j] = id;
        sc[2][j] = pos;
        sc[3][j] = __float_as_int(valid ? ld_gather_f1(s.own_bias + id) : 0.0f);
        sc[4][j] = __float_as_int(valid ? ld_gather_f1(s.partner_bias + part) : 0.0f);
        sc[5][j] = __float_as_int(valid ? fw.rates[pos] : 0.0f);
      }
    }
    __syncwarp(gmask);

    // entry j's rows are in the group's shared-memory slot j & 1, copied asynchronously; entry j + 1's are in flight
    // while j is consumed.  Each lane copies and reads only its own units: no barrier between the two.
    auto fetch = [&](int j) {
      const int32_t pid = sc[0][j], id = sc[1][j];
      const float* prow = s.partner_feat + (size_t)pid * s.partner_stride;
      const float* orow = s.own_feat + (size_t)id * s.own_stride;
#pragma unroll
      for (int q = 0; q < 4; ++q)
        if (has[q]) {
          cp_async_16(&stage[j & 1][0][lane + q * L], prow + (lane + q * L) * 4);
          cp_async_16(&stage[j & 1][1][lane + q * L], orow + (lane + q * L) * 4);
        }
      cp_async_commit_group();
    };
    fetch(0);

    float2 acc[4][2];
    float acc_b = 0.0f, own_b = 0.0f;
    int rs = 0;  // first entry of the current run
    uint8_t kind = 0;
#pragma unroll 2
    for (int j = 0; j < T; ++j) {
      // entries past the end of a short last tile are walked too (nothing of theirs is stored): every shuffle of the
      // walk stays in converged code
      const bool valid = j < n;
      if (j + 1 < n) {
        fetch(j + 1);
        cp_async_wait_group<1>();  // this lane's copies of entry j have landed
      } else {
        cp_async_wait_group<0>();
      }
      Row4 p, o;
#pragma unroll
      for (int q = 0; q < 4; ++q)
        if (has[q]) {
          const float4 x = stage[j & 1][0][lane + q * L], y = stage[j & 1][1][lane + q * L];
          p.v[q][0] = make_float2(x.x, x.y);
          p.v[q][1] = make_float2(x.z, x.w);
          o.v[q][0] = make_float2(y.x, y.y);
          o.v[q][1] = make_float2(y.z, y.w);
        }
      const bool nw = (newm >> j) & 1u;
      if (nw) rs = j;

      // ops.py:44-47: the lane's partial dot in unit order, the butterfly of reduce_transpose<L, 1>, lane 0's sum to
      // the group; every lane then finishes the logit and d cost/d logits of the entry (same operands: same bits)
      float part = 0.0f;
#pragma unroll
      for (int q = 0; q < 4; ++q)
        if (has[q]) {
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            const float2 m = mul2(o.v[q][h], p.v[q][h]);
            part = add_rn(part, m.x);
            part = add_rn(part, m.y);
          }
        }
#pragma unroll
      for (int off = L / 2; off >= 1; off >>= 1) part = add_rn(part, __shfl_xor_sync(gmask, part, off, L));
      const float dot = __shfl_sync(gmask, part, 0, L);
      const float ob = __int_as_float(sc[3][j]), pb = __int_as_float(sc[4][j]), rate = __int_as_float(sc[5][j]);
      float x = add_rn(dot, mu);                     // ops.py:45
      x = add_rn(x, is_item ? pb : ob);              // ops.py:46  + bias_users
      x = add_rn(x, is_item ? ob : pb);              // ops.py:47  + bias_items
      const float e = dloss(flags, x, rate);
      if (!is_item && valid && lane == (j & (L - 1))) {  // the lane that owns entry j's share of the sums
        const float inf = (flags & TFR_LOSS_SIGMOID_CE) ? rintf(sigmoid_tf(x)) : x;
        const int32_t pos = sc[2][j];
        if (fw.logits) fw.logits[pos] = x;
        if (fw.infer) fw.infer[pos] = inf;
        err_acc = add_rn(err_acc, e);
        const double dse = (double)rate - (double)inf;
        se_acc += dse * dse;
      }

      // ---- gradient: g = e * p + reg * own, added in entry order to the run's sum (which starts at +0)
      const float2 e2 = make_float2(e, e);
#pragma unroll
      for (int q = 0; q < 4; ++q)
        if (has[q]) {
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            const float2 g = add2(mul2(e2, p.v[q][h]), mul2(reg2, o.v[q][h]));
            acc[q][h] = add2(nw ? make_float2(0.0f, 0.0f) : acc[q][h], g);
          }
        }
      if (nw) own_b = ob;
      float gb = e;
      if (reg_bias) gb = add_rn(gb, mul_rn(reg, own_b));
      acc_b = add_rn(nw ? 0.0f : acc_b, gb);

      // ---- the run [rs, j] is over: write its sum where segsum_tiles_kernel's flush writes it
      const bool last = valid && (j + 1 >= n || ((newm >> (j + 1)) & 1u));
      if (last) {
        const int32_t cur = sc[1][j];
        const bool starts = rs > 0 || cur != prev_id;
        const bool ends = j + 1 < n || cur != next_id;
        float* dst;
        float* dst_b;
        if (starts && ends) { dst = s.gsum + (size_t)(k0 + rs) * dim; dst_b = s.gsum_b + k0 + rs; }
        else if (!starts)   { dst = s.cont + (size_t)t * dim;         dst_b = s.cont_b + t; if (!ends) kind |= TILE_MID; }
        else                { dst = s.tail + (size_t)t * dim;         dst_b = s.tail_b + t; kind |= TILE_START; }
#pragma unroll
        for (int q = 0; q < 4; ++q)
          if (has[q])
            reinterpret_cast<float4*>(dst)[lane + q * L] =
                make_float4(acc[q][0].x, acc[q][0].y, acc[q][1].x, acc[q][1].y);
        if (lane == 0) {
          *dst_b = acc_b;
          if (starts && ends) s.slot[cur] = pack_slot(stamp, k0 + rs);
        }
      }
    }
    if (lane == 0) {
      s.kind[t] = kind;
      if (kind & TILE_START) {  // a run begins here and goes on: queue its fix-up
        const uint32_t at = atomicAdd(s.fix_count, 1u);
        if (at < (uint32_t)n_tiles) s.fix_list[at] = (int32_t)t;
      }
    }
  }

  // fixed-order block reduction of the user side's sums (segsum_tiles_kernel's, thread for thread)
  if (!ITEM) {
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

// blockIdx.y selects the table; each side is its own inlined body, so that its arguments stay in the parameter bank
// instead of occupying registers
template <int L, int T>
__global__ void __launch_bounds__(SEG_THREADS, 4) chain_tiles_kernel(SegSide su, SegSide si, FwdArgs fw,
                                                                      const tfr_opt_scalars* __restrict__ opt,
                                                                      int64_t B, int dim, int n_tiles) {
  pdl_wait();                // the previous step's table pass (tables, step scalars) is complete
  pdl_launch_dependents();   // the fix-up's CTAs may become resident as this grid drains
  TlScope tl_scope(opt, TFR_TL_TILES);
  __shared__ ChainSmem<L, T> sm;
  if (blockIdx.y) chain_tiles_side<L, T, true>(si, fw, opt, B, dim, n_tiles, sm);
  else chain_tiles_side<L, T, false>(su, fw, opt, B, dim, n_tiles, sm);
}

#define TFR_CHAIN_CASES(X) X(8, 8) X(8, 16) X(16, 8) X(16, 16) X(16, 32) X(32, 8) X(32, 16) X(32, 32)

bool chain_tiles_supported(int lanes, int tile) {
#define TFR_CHAIN_HAS(LL, TT) if (lanes == LL && tile == TT) return true;
  TFR_CHAIN_CASES(TFR_CHAIN_HAS)
#undef TFR_CHAIN_HAS
  return false;
}

int launch_chain_tiles(const SegSide& su, const SegSide& si, const FwdArgs& fw, const tfr_opt_scalars* opt, int64_t B,
                       int dim, int n_tiles, int tile, int lanes, dim3 grid, bool pdl, cudaStream_t st) {
#define TFR_CHAIN_LAUNCH(LL, TT)                                                                                   \
  if (lanes == LL && tile == TT) {                                                                                 \
    if (int rc = prep_tiles((const void*)chain_tiles_kernel<LL, TT>, 0)) return rc;                                \
    TFR_CUDA(launch_kernel(chain_tiles_kernel<LL, TT>, grid, dim3(SEG_THREADS), 0, st, pdl, su, si, fw, opt, B, dim, \
                           n_tiles));                                                                              \
    return TFR_OK;                                                                                                 \
  }
  TFR_CHAIN_CASES(TFR_CHAIN_LAUNCH)
#undef TFR_CHAIN_LAUNCH
  set_error("launch_chain_tiles: no instantiation for %d lanes and tiles of %d", lanes, tile);
  return TFR_ERR_INVALID;
}

}  // namespace tfr
