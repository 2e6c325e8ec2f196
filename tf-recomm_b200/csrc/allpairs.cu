// K6: all-pairs scoring  M[u,i] = <U[u,:], V[i,:]> + W_user[u] + W_work[i] + bias
// Replaces als3.py:110-113 (`self.U.dot(self.V.T) + W_user.reshape(-1,1) + W_work.reshape(1,-1) + bias`, then
// indexing / ranking the rows; forward.py:47-61 ranks one user's row).  The only GEMM-shaped work of the path, so
// the only place tensor cores are used (north_star).
//
// tcgen05 path (dim a multiple of 32, <= 128): one CTA owns 128 users; their rows are loaded ONCE by TMA
// (cp.async.bulk.tensor, 128-byte swizzle) and stay in shared memory while the CTA sweeps the item table in tiles
// of 128 items, double-buffered by a TMA producer warp.  Per tile one elected thread issues dim/8 tcgen05.mma
// (kind::tf32: the fp32 tables are consumed as they are, no conversion pass) into one of two 128x128 fp32
// accumulators in TMEM; eight epilogue warps read the other one back with tcgen05.ld (thread = user row), add the
// biases and CONSUME the tile in registers: running best item per user (top-1 recommendation), and/or the scores
// themselves if the caller wants the matrix.  With the fused consumer the 40 GB score matrix of the ML-25M shape
// never exists.
//
// CUDA-core path (any dim): exact fp32, same outputs; also the reference for the tf32 tolerance in the tests.
//
// Ranking of UNSEEN items (tfr_allpairs_rank_excluding): the top-k consumer skips each user's excluded items (CSR walk in
// the epilogue, like the observed-pairs walk) and the certificate counts only rankable items.  For a dim the tcgen05
// sweep cannot take (dim % 32 != 0 or dim > 128, up to 512) there is no sweep: every row goes through the exact float64
// fallback, O(n_users * n_items * (dim + k)) -- fine at the ML-1M shape, not a path for ML-25M.
#include <cuda.h>
#include <string.h>

#include "common.cuh"

namespace tfr {

constexpr int AP_BM = 128, AP_BN = 128, AP_KC = 32;      // tile: 128 users x 128 items, K chunks of 32 floats (128 B)
constexpr int AP_CHUNK_BYTES = 128 * AP_KC * 4;           // one TMA box: 128 rows x 128 B = 16 KB

// ---- PTX wrappers ---------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "LAB_WAIT:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra LAB_DONE;\n\t"
      "bra LAB_WAIT;\n\t"
      "LAB_DONE:\n\t}" ::"r"(smem_u32(bar)), "r"(parity)
      : "memory");
}
// the same wait for the two single-thread roles (TMA producer, MMA issuer): they wait for the epilogue most of the time,
// and a bare try_wait loop takes issue slots from the epilogue warps that share their schedulers (ncu: SYNCS + YIELD + BRA
// were 40 % of the instructions the kernel executed) -- sleep between polls
__device__ __forceinline__ void mbar_wait_polite(uint64_t* bar, uint32_t parity) {
  uint32_t done;
  for (;;) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    if (done) break;
    __nanosleep(200);
  }
}
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* map, int c0, int c1, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
          smem_u32(dst)),
      "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
// K-major, 128-byte swizzle operand descriptor (cute/arch/mma_sm100_desc.hpp SmemDescriptor): start address >> 4 in
// bits [0,14); leading byte offset (unused for swizzled K-major) = 1 in [16,30); stride byte offset = 1024 B (one
// 8-row swizzle atom) >> 4 in [32,46); version = 1 in [46,48); layout SWIZZLE_128B = 2 in [61,64).
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t saddr) {
  return (uint64_t)((saddr & 0x3FFFFu) >> 4) | ((uint64_t)1 << 16) | ((uint64_t)(1024 >> 4) << 32) | ((uint64_t)1 << 46) |
         ((uint64_t)2 << 61);
}
// instruction descriptor (InstrDescriptor): D = F32 (1 @ [4,6)), A = B = TF32 (2 @ [7,10), [10,13)), both K-major,
// N >> 3 @ [17,23), M >> 4 @ [24,29)
__host__ __device__ constexpr uint32_t ap_idesc(int M, int N) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
      "l"(da), "l"(db), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, float* v) {
  uint32_t r[32];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}

// Warp roles (320 threads): warp 0 = TMA producer, warp 1 = MMA issuer (+ TMEM allocation), warps 2..9 = epilogue.
// An epilogue warp may only touch the TMEM lanes 32*(warp % 4) .. +31 (its quarter of the 128 user rows); two warps
// share each quarter and split the tile's 128 item columns in halves.  Pipelines: item tiles double-buffered in
// shared memory (full/empty mbarriers between TMA and MMA), accumulators double-buffered in TMEM (2 x 128 columns,
// full/empty mbarriers between MMA and epilogue), so TMA, tensor cores and the epilogue of consecutive tiles overlap.
//
// Consumers of a tile, all in the epilogue's registers (the score matrix never exists unless `scores` is asked for):
//   * top-1: running best item per user (lowest index on ties);
//   * TOPK: the K best items per user by tensor-core score -- forward.py:47-61 ranks a user's scores and keeps 50.  A
//     row's candidates live UNSORTED in its [K] slice of cand_val / cand_idx (global memory, L2-resident); the row's
//     current K-th best score is the threshold a column has to reach to take the slow path (an insert under a per-row
//     shared-memory lock: replace the minimum, rescan it).  After the first tiles almost no column does.  The caller
//     rescores the candidates exactly and certifies the result (allpairs_rescore_kernel);
//   * OBS: the squared error on the OBSERVED pairs, als3.py:110-120,139-143 (predict = M[user_ids, work_ids], then
//     compute_rmse): the pairs come as CSR by user with ascending item ids; every row's thread walks its list as the
//     tiles go by and accumulates (score - rating)^2 in float64.
//   * EXCL (with TOPK, without OBS): items the user must not be recommended (the ones already rated), CSR by user with
//     ascending item ids, duplicates allowed; the row's lane walks its list like the OBS walk and a column equal to the
//     next excluded id is never appended to the candidate buffer.  Everything else of TOPK is unchanged.
constexpr int AP_THREADS = 320, AP_EPI_WARPS = 8;
enum { BAR_A = 0, BAR_FULL_B = 1, BAR_EMPTY_B = 3, BAR_TMEM_FULL = 5, BAR_TMEM_EMPTY = 7, AP_NBARS = 9 };
constexpr int AP_MAX_CAND = 128;

struct ApConsumers {
  float* scores;             // [n_users, n_items] or null
  float* best_score;         // [n_users] or null
  int32_t* best_item;        // [n_users] or null
  float* cand_val;           // TOPK: [n_users, 2, 4K]: one buffer per row and column half
  int32_t* cand_idx;         // TOPK: [n_users, 2, 4K]
  int32_t* cand_cnt;         // TOPK: [n_users, 2] entries in the buffer at the end of the sweep
  float* cand_thr;           // TOPK: [n_users, 2] the buffer's threshold: no dropped column scored above it
  int K;
  const int64_t* obs_indptr; // OBS: [n_users + 1]
  const int32_t* obs_item;   // OBS: [nnz] ascending inside a user's range
  const float* obs_rate;     // OBS: [nnz]
  double* row_se;            // OBS: [n_users] sum over the user's observed pairs of (score - rating)^2
  const int64_t* excl_indptr; // EXCL: [n_users + 1]
  const int32_t* excl_item;   // EXCL: [nnz] ascending inside a user's range
};

// order of the ranking: higher score first, lower item index on ties
__device__ __forceinline__ bool ap_better(float s, int i, float s2, int i2) { return s > s2 || (s == s2 && i < i2); }

// TOPK consumer.  Each epilogue warp keeps its OWN candidate buffer per row (the two warps that share a row's TMEM lanes
// split the columns in halves: a row has two buffers, merged by the rescore), so nothing is shared between warps: a
// buffer's length and threshold live in the registers of the row's lane.
//   hot path:   a column whose score exceeds the row's threshold is APPENDED by the row's own lane (two stores, nothing
//               waits for them);
//   slow path:  when a buffer of C = 4K entries is full, the warp COMPACTS it together: a radix select over the scores'
//               order-preserving keys finds the K-th best, the K best entries (lowest item index on ties) are kept and the
//               K-th best score becomes the threshold.  A row-half sees ~K ln(N/K) appends in all, i.e. two or three
//               compactions per sweep -- against one latency-bound list scan PER INSERT in the first version
//               (profiles/r02_allpairs_ncu_full.md).
// Columns arrive in ascending index order, so an entry appended later never beats a kept one of equal score.
constexpr int AP_EPL = 4 * AP_MAX_CAND / 32;   // buffer entries per lane at the largest C
struct ApListState { int cnt; float thr; };
__device__ __forceinline__ uint32_t ap_key(float f) {   // unsigned order == float order
  const uint32_t u = __float_as_uint(f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ int warp_sum_i(int x) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
  return x;
}
// (not inlined: called from a 64-times unrolled column loop).  The buffer holds `cnt` (<= C) entries; afterwards its first
// min(cnt, K) slots hold the K best and the returned threshold is the K-th best score (-inf if cnt < K).
__device__ __noinline__ ApListState ap_compact_warp(float* __restrict__ cval, int32_t* __restrict__ cidx, int cnt, int K,
                                                    int lane) {
  ApListState out;
  if (cnt <= K) { out.cnt = cnt; out.thr = cnt == K ? INFINITY : -INFINITY; }
  float v[AP_EPL];
  int ix[AP_EPL];
  uint32_t key[AP_EPL];
  bool valid[AP_EPL];
#pragma unroll
  for (int j = 0; j < AP_EPL; ++j) {
    const int p = lane + 32 * j;
    valid[j] = p < cnt;
    v[j] = 0.0f; ix[j] = 0x7fffffff; key[j] = 0u;
    if (valid[j]) { v[j] = __ldcg(cval + p); ix[j] = __ldcg(cidx + p); key[j] = ap_key(v[j]); }
  }
  if (cnt < K) return out;   // (uniform) nothing to drop yet
  // K-th largest key
  uint32_t tk = 0u;
#pragma unroll 1
  for (int bit = 31; bit >= 0; --bit) {
    const uint32_t cand = tk | (1u << bit);
    int c = 0;
#pragma unroll
    for (int j = 0; j < AP_EPL; ++j) c += (valid[j] && key[j] >= cand) ? 1 : 0;
    if (warp_sum_i(c) >= K) tk = cand;
  }
  int n_gt = 0, n_eq = 0;
#pragma unroll
  for (int j = 0; j < AP_EPL; ++j) {
    n_gt += (valid[j] && key[j] > tk) ? 1 : 0;
    n_eq += (valid[j] && key[j] == tk) ? 1 : 0;
  }
  n_gt = warp_sum_i(n_gt);
  n_eq = warp_sum_i(n_eq);
  const int need_eq = K - n_gt;   // >= 1: how many of the entries that tie with the K-th best are kept
  int it = 0x7fffffff;            // they are the ones with the lowest item index: the need_eq-th smallest index among them
  if (n_eq > need_eq) {
    uint32_t ip = 0u;             // largest x with #{ties: idx < x} < need_eq  ==  the need_eq-th smallest tie index
#pragma unroll 1
    for (int bit = 30; bit >= 0; --bit) {
      const uint32_t cand = ip | (1u << bit);
      int c = 0;
#pragma unroll
      for (int j = 0; j < AP_EPL; ++j) c += (valid[j] && key[j] == tk && (uint32_t)ix[j] < cand) ? 1 : 0;
      if (warp_sum_i(c) < need_eq) ip = cand;
    }
    it = (int)ip;
  }
  __syncwarp();   // every lane holds its entries in registers: the buffer may be overwritten
  int base = 0;
#pragma unroll
  for (int j = 0; j < AP_EPL; ++j) {
    const bool keep = valid[j] && (key[j] > tk || (key[j] == tk && ix[j] <= it));
    const unsigned m = __ballot_sync(0xffffffffu, keep);
    if (keep) {
      const int pos = base + __popc(m & ((1u << lane) - 1u));
      __stcg(cval + pos, v[j]);
      __stcg(cidx + pos, ix[j]);
    }
    base += __popc(m);
  }
  __syncwarp();
  // the K-th best score back from its key (the inverse of ap_key)
  const float t0 = __uint_as_float((tk & 0x80000000u) ? (tk & 0x7fffffffu) : ~tk);
  out.cnt = base;
  out.thr = t0;
  return out;
}

template <int KCHUNKS, bool TOPK, bool OBS, bool EXCL>
__global__ void __launch_bounds__(AP_THREADS, 1)
    allpairs_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                       const float* __restrict__ ub, const float* __restrict__ ib, const float* __restrict__ mu,
                       int n_users, int n_items, const ApConsumers cs) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* base = reinterpret_cast<uint8_t*>(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);  // swizzle atoms: 1024 B
  uint8_t* sA = base;
  uint8_t* sB[2] = {base + KCHUNKS * AP_CHUNK_BYTES, base + 2 * KCHUNKS * AP_CHUNK_BYTES};
  uint64_t* bars = reinterpret_cast<uint64_t*>(base + 3 * KCHUNKS * AP_CHUNK_BYTES);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + AP_NBARS);
  // barriers + TMEM slot live in the first 128 bytes after the tiles; the arrays behind them stay 16-byte aligned
  // (s_bias is read with LDS.128, s_se holds doubles)
  static_assert(AP_NBARS * 8 + 16 <= 128, "barrier block");
  float* s_best = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(bars) + 128);   // [2][128] halves' best score per row
  int32_t* s_besti = reinterpret_cast<int32_t*>(s_best + 256);   // [2][128]
  float* s_bias = reinterpret_cast<float*>(s_besti + 256);       // [8][64] item bias + mu of each epilogue warp's columns
  double* s_se = reinterpret_cast<double*>(s_bias + 512);        // [2][128] OBS: halves' squared-error sums
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int m0 = blockIdx.x * AP_BM;
  const int n_tiles = (n_items + AP_BN - 1) / AP_BN;
  constexpr uint32_t kTileBytes = KCHUNKS * AP_CHUNK_BYTES;
  constexpr uint32_t kIdesc = ap_idesc(AP_BM, AP_BN);

  if (tid == 0) {
    mbar_init(&bars[BAR_A], 1);
    for (int i = 0; i < 2; ++i) {
      mbar_init(&bars[BAR_FULL_B + i], 1);
      mbar_init(&bars[BAR_EMPTY_B + i], 1);
      mbar_init(&bars[BAR_TMEM_FULL + i], 1);
      mbar_init(&bars[BAR_TMEM_EMPTY + i], AP_EPI_WARPS);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {  // 256 TMEM columns = two 128x128 fp32 accumulators
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 256;" ::"r"(smem_u32(tmem_slot)) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem = *tmem_slot;

  if (warp == 0) {
    // ===== TMA producer =====
    if (lane == 0) {
      mbar_expect_tx(&bars[BAR_A], kTileBytes);
#pragma unroll
      for (int c = 0; c < KCHUNKS; ++c) tma_load_2d(sA + c * AP_CHUNK_BYTES, &tmA, c * AP_KC, m0, &bars[BAR_A]);
      for (int t = 0; t < n_tiles; ++t) {
        const int buf = t & 1;
        if (t >= 2) mbar_wait_polite(&bars[BAR_EMPTY_B + buf], ((t >> 1) - 1) & 1);  // MMAs of tile t-2 have read the buffer
        mbar_expect_tx(&bars[BAR_FULL_B + buf], kTileBytes);
#pragma unroll
        for (int c = 0; c < KCHUNKS; ++c)
          tma_load_2d(sB[buf] + c * AP_CHUNK_BYTES, &tmB, c * AP_KC, t * AP_BN, &bars[BAR_FULL_B + buf]);
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer: one thread on behalf of the CTA =====
    if (lane == 0) {
      mbar_wait(&bars[BAR_A], 0);
      const uint32_t a0 = smem_u32(sA);
      for (int t = 0; t < n_tiles; ++t) {
        const int buf = t & 1, acc = t & 1;
        mbar_wait_polite(&bars[BAR_FULL_B + buf], (t >> 1) & 1);
        if (t >= 2) mbar_wait_polite(&bars[BAR_TMEM_EMPTY + acc], ((t >> 1) - 1) & 1);  // epilogue drained accumulator acc
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const uint32_t b0 = smem_u32(sB[buf]);
#pragma unroll
        for (int c = 0; c < KCHUNKS; ++c) {
#pragma unroll
          for (int k = 0; k < AP_KC / 8; ++k) {  // UMMA_K = 8 tf32 = 32 B inside the 128 B swizzle atom
            const uint64_t da = umma_desc_sw128(a0 + c * AP_CHUNK_BYTES + k * 32);
            const uint64_t db = umma_desc_sw128(b0 + c * AP_CHUNK_BYTES + k * 32);
            umma_tf32(tmem + (uint32_t)(acc * AP_BN), da, db, kIdesc, (c | k) ? 1u : 0u);
          }
        }
        umma_commit(&bars[BAR_EMPTY_B + buf]);     // shared-memory tile free once these MMAs have read it
        umma_commit(&bars[BAR_TMEM_FULL + acc]);   // accumulator ready for the epilogue
      }
    }
  } else {
    // ===== epilogue: TMEM -> registers -> biases -> consume =====
    const int ew = warp - 2;              // 0..7
    const int quarter = warp & 3;         // TMEM lane quarter this warp may access
    const int half = ew >> 2;             // which 64 of the tile's 128 columns
    const int r_in_tile = quarter * 32 + lane;
    const int row = m0 + r_in_tile;
    const bool row_ok = row < n_users;
    const float bu = row_ok ? ub[row] : 0.0f;
    const float mu_ = *mu;
    float best[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};  // 4 independent chains (column % 4)
    int32_t besti[4] = {-1, -1, -1, -1};
    int lcnt = 0;               // TOPK: length and threshold of this lane's row's buffer (this warp's half of the columns)
    float thr = -INFINITY;
    const int K = cs.K, C = 4 * cs.K;     // kept entries / buffer capacity
    float* const cand_val = cs.cand_val;
    int32_t* const cand_idx = cs.cand_idx;
    float* const scores = cs.scores;
    float* const my_val = TOPK ? cs.cand_val + ((size_t)(row_ok ? row : 0) * 2 + half) * (size_t)C : nullptr;
    int32_t* const my_idx = TOPK ? cs.cand_idx + ((size_t)(row_ok ? row : 0) * 2 + half) * (size_t)C : nullptr;
    // OBS: this row's observed pairs [op, oend), next one's item id / rating
    int64_t op = 0, oend = 0;
    int onext = 0x7fffffff, onext2 = 0x7fffffff;   // the next pair's item id, and the one after it (fetched ahead: a
    float orate = 0.0f, orate2 = 0.0f;             // hit then never waits for a load it has just issued)
    double se = 0.0;
    // EXCL: this row's excluded items [xp, xend), the next one's id and the one after it (fetched ahead, as for OBS)
    int64_t xp = 0, xend = 0;
    int xnext = 0x7fffffff, xnext2 = 0x7fffffff;
    if (EXCL && row_ok) {
      xp = cs.excl_indptr[row];
      xend = cs.excl_indptr[row + 1];
      if (xp < xend) xnext = cs.excl_item[xp];
      if (xp + 1 < xend) xnext2 = cs.excl_item[xp + 1];
    }
    auto excl_advance = [&]() {
      ++xp;
      xnext = xnext2;
      xnext2 = xp + 1 < xend ? cs.excl_item[xp + 1] : 0x7fffffff;
    };
    if (OBS && row_ok) {
      op = cs.obs_indptr[row];
      oend = cs.obs_indptr[row + 1];
      if (op < oend) { onext = cs.obs_item[op]; orate = cs.obs_rate[op]; }
      if (op + 1 < oend) { onext2 = cs.obs_item[op + 1]; orate2 = cs.obs_rate[op + 1]; }
    }
    auto obs_advance = [&]() {   // on to the next pair of this row
      ++op;
      onext = onext2; orate = orate2;
      if (op + 1 < oend) { onext2 = cs.obs_item[op + 1]; orate2 = cs.obs_rate[op + 1]; } else onext2 = 0x7fffffff;
    };
    for (int t = 0; t < n_tiles; ++t) {
      const int acc = t & 1;
      const int n0 = t * AP_BN + half * 64;
      // the tile's item biases (+ mu: (dot + b_u) + (b_i + mu), the tensor-core path is tf32-approximate anyway) go
      // to shared memory once per tile; a column's bias is then one broadcast LDS.128 per four columns
      // (per WARP: its own 64 columns, two per lane -- no barrier between the epilogue warps)
      {
        float* const wb = s_bias + (size_t)ew * 64;
#pragma unroll
        for (int x = 0; x < 2; ++x) {
          const int cc = n0 + lane + 32 * x;
          wb[lane + 32 * x] = cc < n_items ? add_rn(__ldg(ib + cc), mu_) : 0.0f;
        }
        __syncwarp();
      }
      if (OBS) {
        while (onext < n0) obs_advance();  // pairs of the columns the other half owns, or of earlier tiles
      }
      if (EXCL) {
        while (xnext < n0) excl_advance();
      }
      mbar_wait(&bars[BAR_TMEM_FULL + acc], (t >> 1) & 1);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        float v[32];
        tmem_ld_32x32(tmem + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(acc * AP_BN + half * 64 + j * 32), v);
        const float4* sb4 = reinterpret_cast<const float4*>(s_bias + (size_t)ew * 64 + j * 32);
#pragma unroll
        for (int c4 = 0; c4 < 8; ++c4) {
          const float4 b4 = sb4[c4];
          const float bb[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const int c = c4 * 4 + q;
            const int col = n0 + j * 32 + c;
            const float s = add_rn(add_rn(v[c], bu), bb[q]);   // als3.py:112: U.V^T + W_user + W_work + bias
            const bool ok = row_ok && col < n_items;
            if (scores && ok) scores[(size_t)row * n_items + col] = s;
            if (ok && s > best[q]) { best[q] = s; besti[q] = col; }
            bool excluded = false;
            if (EXCL) {
              if (col == xnext) {
                excluded = true;
                do excl_advance(); while (xnext == col);   // duplicates of an id
              }
            }
            if (TOPK) {
              // hot path: the row's own lane appends (two stores); compaction is checked once per 32-column chunk
              if (ok && s > thr && !excluded) {
                __stcg(my_val + lcnt, s);
                __stcg(my_idx + lcnt, col);
                ++lcnt;
              }
            }
            if (OBS) {
              if (col == onext) {
                // duplicates of a pair (the same item twice in a user's list) all count, like fancy indexing does
                do {
                  const double d = (double)s - (double)orate;
                  se += d * d;
                  obs_advance();
                } while (onext == col);
              }
            }
          }
        }
        if (TOPK) {
          // a chunk appends at most 32 entries per row: a buffer with less than that left is compacted now, by the whole
          // warp, one row after the other
          unsigned full = __ballot_sync(0xffffffffu, lcnt > C - 32);
          while (full) {
            const int src = __ffs(full) - 1;
            full &= full - 1;
            const int bcnt = __shfl_sync(0xffffffffu, lcnt, src);
            const size_t list = ((size_t)(m0 + quarter * 32 + src) * 2 + half) * (size_t)C;
            const ApListState ns = ap_compact_warp(cand_val + list, cand_idx + list, bcnt, K, lane);
            if (lane == src) { lcnt = ns.cnt; thr = ns.thr; }
          }
        }
      }
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      __syncwarp();
      if (lane == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(&bars[BAR_TMEM_EMPTY + acc])) : "memory");
    }
    // merge the 4 chains (lower item index wins ties), then the two column halves through shared memory
    float bs = best[0];
    int32_t bi_ = besti[0];
#pragma unroll
    for (int q = 1; q < 4; ++q)
      if (best[q] > bs || (best[q] == bs && besti[q] >= 0 && (bi_ < 0 || besti[q] < bi_))) { bs = best[q]; bi_ = besti[q]; }
    s_best[half * 128 + r_in_tile] = bs;
    s_besti[half * 128 + r_in_tile] = bi_;
    if (OBS) s_se[half * 128 + r_in_tile] = se;
    if (TOPK && row_ok) {   // the buffer's final length and threshold, for the rescore
      cs.cand_cnt[(size_t)row * 2 + half] = lcnt;
      cs.cand_thr[(size_t)row * 2 + half] = thr;
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (tid < 128) {
    const int row = m0 + tid;
    if (row < n_users) {
      float bs = s_best[tid];
      int32_t bi_ = s_besti[tid];
      const float b1 = s_best[128 + tid];
      const int32_t i1 = s_besti[128 + tid];
      if (b1 > bs || (b1 == bs && i1 >= 0 && (bi_ < 0 || i1 < bi_))) { bs = b1; bi_ = i1; }
      if (cs.best_score) cs.best_score[row] = bs;
      if (cs.best_item) cs.best_item[row] = bi_;
      if (OBS) cs.row_se[row] = s_se[tid] + s_se[128 + tid];
    }
  }
  if (warp == 1) {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 256;" ::"r"(tmem) : "memory");
  }
}

// ---- exact rescore of the tensor-core candidates, with a certificate --------------------------------------------------
// The sweep ranks s = fl(fl(D + b_u) + fl(b_i + mu)) (fp32, round to nearest), D the tensor cores' fp32 dot product of
// tf32 operands.  Its distance from the exact score u.v + b_u + b_i + mu is at most
//   E_u = (2^-9 + dim * 2^-22) * ||u|| * V  +  2^-22 * (||u|| * V + |b_u| + B),   V = max_i ||v_i||, B = max_i |fl(b_i + mu)|:
//   * tf32: the MMA reads 10 of an operand's 23 mantissa bits, |x' - x| < 2^-10 |x| whether it truncates or rounds, so
//     |u'v' - uv| < (2^-9 + 2^-20) |uv|;
//   * accumulation: dim/8 k-steps each add 8 exact products to the fp32 accumulator.  Even a step that aligns its 9
//     addends to the largest and truncates each of them and its result to 24 bits loses < 10 ulps (2^-23 relative) of
//     values <= sum |u'v'|: over the sweep < dim/8 * 20 * 2^-24 = 0.625 * dim * 2^-22 of sum |u'v'|.  With the 2^-20 of
//     the products (dim >= 32) the dot product is within (2^-9 + dim * 2^-22) * sum_k |u_k v_k|, and sum_k |u_k v_k| <=
//     ||u|| * V;
//   * the three additions round to nearest, each by <= 2^-24 of its result: fl(b_i + mu) is <= B, fl(D + b_u) and s are
//     <= |D| + |b_u| (+ B), so together <= 2^-23 (1 + 2^-23) (|D| + |b_u| + B): 2^-22 leaves a factor of 2.  This term is
//     what is left when ||u|| * V vanishes (a zero user row, an all-zero item table) and the biases do not.
// V and B come from allpairs_vmax2_kernel (V^2 rounded up).  Measured on a B200 (1000 W power limit) with
// tests/test_topk_certificate.py's inputs: |s - exact| <= 0.47 E_u, and on random operands the dot product's error is
// <= 0.27 * 2^-9 * sum_k |u_k v_k|; kind::tf32 truncates (its scores equal a truncating model's bit for bit).
// Every item that is NOT in a row's two buffers scored at most T = max of the buffers' thresholds on the tensor cores,
// hence at most T + E_u exactly (a buffer that never had to drop anything has threshold -inf).  The candidates are
// rescored in float64 -- the reference's own precision: als3.py:112 is numpy float64 -- and the k best picked (score
// descending, lowest item index on ties); they are the exact top-k of the WHOLE row if the k-th exact score is > T + E_u.
// Rows for which that cannot be shown (near-ties deeper than the spare candidates) are appended to `uncert` and redone
// exactly over all items by allpairs_exact_rows_kernel.  One warp per row.
// With an exclusion list (EXCL sweep) the argument is the same over the row's RANKABLE items: an excluded item is never a
// candidate, and every other item that is not one scored at most T.  The row ranks min(k, rankable_u) items, rankable_u =
// n_items - (distinct excluded ids of u); the ranks past that are (-inf, -1), and a row whose items are all excluded is
// all (-inf, -1) and certified.
constexpr int RS_WARPS = 2;
__global__ void __launch_bounds__(32 * RS_WARPS) allpairs_rescore_kernel(
    const float* __restrict__ U, const float* __restrict__ V, const float* __restrict__ ub, const float* __restrict__ ib,
    const float* __restrict__ mu, int n_users, int n_items, int dim, int64_t us, int64_t is,
    const float* __restrict__ cand_val, const int32_t* __restrict__ cand_idx, const int32_t* __restrict__ cand_cnt,
    const float* __restrict__ cand_thr, int K, int k, const float* __restrict__ vmax2 /* [V^2, B] */,
    double* __restrict__ out_val, int32_t* __restrict__ out_idx, int32_t* __restrict__ uncert, int32_t* __restrict__ n_uncert,
    const int64_t* __restrict__ excl_indptr, const int32_t* __restrict__ excl_item) {
  __shared__ double s_sc[RS_WARPS][8 * AP_MAX_CAND];
  __shared__ int s_ix[RS_WARPS][8 * AP_MAX_CAND];
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int row = blockIdx.x * RS_WARPS + w;
  if (row >= n_users) return;
  const int C = 4 * K;
  __shared__ float s_u[RS_WARPS][512];
  const float* urow = U + (size_t)row * us;
  double un2 = 0.0;
  for (int d = lane; d < dim; d += 32) {
    const float x = urow[d];
    s_u[w][d] = x;
    un2 += (double)x * (double)x;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) un2 += __shfl_xor_sync(0xffffffffu, un2, o);
  __syncwarp();
  const int cnt0 = min(cand_cnt[(size_t)row * 2], C), cnt1 = min(cand_cnt[(size_t)row * 2 + 1], C);
  const float T = fmaxf(cand_thr[(size_t)row * 2], cand_thr[(size_t)row * 2 + 1]);
  const int n = cnt0 + cnt1;
  // a candidate per lane at a time: the lanes' row gathers are independent and in flight together (one warp walking
  // the candidates one by one paid two dependent global latencies per candidate)
  const bool vec = (dim % 4 == 0) && (is % 4 == 0) && (((uintptr_t)V & 15u) == 0);
  for (int c = lane; c < n; c += 32) {
    const size_t at = c < cnt0 ? (size_t)row * 2 * C + c : ((size_t)row * 2 + 1) * C + (c - cnt0);
    const int it = cand_idx[at];
    const float* vrow = V + (size_t)it * is;
    double acc = 0.0;
    if (vec) {
      for (int d = 0; d < dim; d += 4) {
        const float4 q = ld_gather_f4(reinterpret_cast<const float4*>(vrow + d));
        acc += (double)s_u[w][d] * (double)q.x;
        acc += (double)s_u[w][d + 1] * (double)q.y;
        acc += (double)s_u[w][d + 2] * (double)q.z;
        acc += (double)s_u[w][d + 3] * (double)q.w;
      }
    } else {
      for (int d = 0; d < dim; ++d) acc += (double)s_u[w][d] * (double)vrow[d];
    }
    s_sc[w][c] = ((acc + (double)ub[row]) + (double)ib[it]) + (double)mu[0];   // als3.py:112, in float64 like numpy
    s_ix[w][c] = it;
  }
  __syncwarp();
  // k rounds of a warp-wide arg-max over the candidates that come AFTER the previous pick in the total order
  double last_v = INFINITY, kth = -INFINITY;
  int last_i = -1, got = 0;
  for (int r = 0; r < k; ++r) {
    double bv = -INFINITY;
    int bi = -1;
    for (int c = lane; c < n; c += 32) {
      const double v = s_sc[w][c];
      const int i = s_ix[w][c];
      const bool after = v < last_v || (v == last_v && i > last_i);
      if (after && (bi < 0 || v > bv || (v == bv && i < bi))) { bv = v; bi = i; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const double ov = __shfl_xor_sync(0xffffffffu, bv, o);
      const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
      if (oi >= 0 && (bi < 0 || ov > bv || (ov == bv && oi < bi))) { bv = ov; bi = oi; }
    }
    if (lane == 0) {
      out_val[(size_t)row * k + r] = bi >= 0 ? bv : -INFINITY;
      out_idx[(size_t)row * k + r] = bi;
    }
    if (bi < 0) {
      if (lane == 0)
        for (int rr = r + 1; rr < k; ++rr) { out_val[(size_t)row * k + rr] = -INFINITY; out_idx[(size_t)row * k + rr] = -1; }
      break;
    }
    last_v = bv; last_i = bi; kth = bv; ++got;
  }
  int rankable = n_items;
  if (excl_indptr && got < k) {   // (warp-uniform) only a short row needs its number of rankable items
    const int64_t x0 = excl_indptr[row], x1 = excl_indptr[row + 1];
    int distinct = 0;
    for (int64_t p = x0 + lane; p < x1; p += 32) distinct += (p == x0 || excl_item[p] != excl_item[p - 1]) ? 1 : 0;
    rankable -= warp_sum_i(distinct);
  }
  if (lane == 0) {
    const int kk = k < rankable ? k : rankable;
    bool certified = T == -INFINITY;   // nothing was ever dropped: every rankable item is a candidate
    if (!certified && got >= kk) {
      const double uv = sqrt(un2) * sqrt((double)vmax2[0]);
      const double E = (0x1p-9 + dim * 0x1p-22) * uv + 0x1p-22 * (uv + fabs((double)ub[row]) + (double)vmax2[1]);
      certified = kth > (double)T + E;
    }
    if (!certified) uncert[atomicAdd(n_uncert, 1)] = row;
  }
}

// out[0] = max over the item rows of ||v||^2, out[1] = max |fl(b_i + mu)| (the sweep's add_rn), both by atomicMax on the
// bit pattern of a non-negative float; out zeroed by the caller
__global__ void allpairs_vmax2_kernel(const float* __restrict__ V, const float* __restrict__ ib, const float* __restrict__ mu,
                                      int n_items, int dim, int64_t is, float* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const int it = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (it >= n_items) return;
  const float* vrow = V + (size_t)it * is;
  float n2 = 0.0f;
  for (int d = lane; d < dim; d += 32) n2 = fmaf(vrow[d], vrow[d], n2);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) n2 += __shfl_xor_sync(0xffffffffu, n2, o);
  n2 = n2 * 1.0001f;  // the float sum may round down
  if (lane == 0) {
    atomicMax(reinterpret_cast<int*>(out), __float_as_int(n2));
    atomicMax(reinterpret_cast<int*>(out) + 1, __float_as_int(fabsf(add_rn(ib[it], *mu))));
  }
}

// The uncertified rows, redone exactly over ALL items: a persistent CTA per row computes the row's float64 scores into
// its scratch line, then picks the k best by k rounds of a block-wide arg-max (the total order of ap_better).
// Excluded items (excl_indptr != null) are marked NaN in the line, which the arg-max never picks: they are skipped, and
// the ranks past the row's rankable items are (-inf, -1).
__global__ void __launch_bounds__(1024) allpairs_exact_rows_kernel(const float* __restrict__ U, const float* __restrict__ V,
                                                                  const float* __restrict__ ub, const float* __restrict__ ib,
                                                                  const float* __restrict__ mu, int n_items, int dim,
                                                                  int64_t us, int64_t is, const int32_t* __restrict__ uncert,
                                                                  const int32_t* __restrict__ n_uncert, int k,
                                                                  double* __restrict__ scratch, double* __restrict__ out_val,
                                                                  int32_t* __restrict__ out_idx,
                                                                  const int64_t* __restrict__ excl_indptr,
                                                                  const int32_t* __restrict__ excl_item) {
  __shared__ float s_u[512];
  __shared__ double s_v[32];
  __shared__ int s_i[32];
  __shared__ double s_last_v;
  __shared__ int s_last_i;
  double* line = scratch + (size_t)blockIdx.x * n_items;
  const int n = *n_uncert;
  for (int e = blockIdx.x; e < n; e += gridDim.x) {
    const int row = uncert[e];
    __syncthreads();
    for (int d = threadIdx.x; d < dim; d += blockDim.x) s_u[d] = U[(size_t)row * us + d];
    __syncthreads();
    const double bu = (double)ub[row], m = (double)mu[0];
    for (int it = threadIdx.x; it < n_items; it += blockDim.x) {
      const float* vrow = V + (size_t)it * is;
      double acc = 0.0;
      for (int d = 0; d < dim; ++d) acc += (double)s_u[d] * (double)vrow[d];
      line[it] = ((acc + bu) + (double)ib[it]) + m;
    }
    __syncthreads();
    if (excl_indptr) {
      for (int64_t p = excl_indptr[row] + threadIdx.x; p < excl_indptr[row + 1]; p += blockDim.x) line[excl_item[p]] = nan("");
      __syncthreads();
    }
    double last_v = INFINITY;
    int last_i = -1;
    for (int r = 0; r < k; ++r) {
      double bv = -INFINITY;
      int bi = -1;
      for (int c = threadIdx.x; c < n_items; c += blockDim.x) {
        const double v = line[c];
        const bool after = v < last_v || (v == last_v && c > last_i);
        if (after && (bi < 0 || v > bv || (v == bv && c < bi))) { bv = v; bi = c; }
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const double ov = __shfl_xor_sync(0xffffffffu, bv, o);
        const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
        if (oi >= 0 && (bi < 0 || ov > bv || (ov == bv && oi < bi))) { bv = ov; bi = oi; }
      }
      if ((threadIdx.x & 31) == 0) { s_v[threadIdx.x >> 5] = bv; s_i[threadIdx.x >> 5] = bi; }
      __syncthreads();
      if (threadIdx.x < 32) {
        bv = s_v[threadIdx.x];
        bi = s_i[threadIdx.x];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
          const double ov = __shfl_xor_sync(0xffffffffu, bv, o);
          const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
          if (oi >= 0 && (bi < 0 || ov > bv || (ov == bv && oi < bi))) { bv = ov; bi = oi; }
        }
        if (threadIdx.x == 0) {
          s_last_v = bv;
          s_last_i = bi;
          out_val[(size_t)row * k + r] = bi >= 0 ? bv : -INFINITY;
          out_idx[(size_t)row * k + r] = bi;
        }
      }
      __syncthreads();
      last_v = s_last_v;
      last_i = s_last_i;
      if (last_i < 0) {
        for (int rr = r + 1 + threadIdx.x; rr < k; rr += blockDim.x) {
          out_val[(size_t)row * k + rr] = -INFINITY;
          out_idx[(size_t)row * k + rr] = -1;
        }
        break;
      }
    }
  }
}

// every row to the exact path (dims the tcgen05 sweep cannot take): uncert = 0 .. n_users - 1, *n_uncert = n_users
__global__ void allpairs_all_rows_kernel(int n_users, int32_t* __restrict__ uncert, int32_t* __restrict__ n_uncert) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n_users; i += gridDim.x * blockDim.x) uncert[i] = i;
  if (blockIdx.x == 0 && threadIdx.x == 0) *n_uncert = n_users;
}

// ---- CUDA-core path: exact fp32, any dim --------------------------------------------------------------------
// 64 users x 64 items per CTA, both tiles staged in shared memory (transposed, padded), 4x4 register blocking.
__global__ void __launch_bounds__(256) allpairs_simt_kernel(const float* __restrict__ U, const float* __restrict__ V,
                                                            const float* __restrict__ ub, const float* __restrict__ ib,
                                                            const float* __restrict__ mu, int n_users, int n_items, int dim,
                                                            int64_t us, int64_t is,  // floats between rows of U / V
                                                            float* __restrict__ scores, float* __restrict__ tile_best,
                                                            int32_t* __restrict__ tile_best_item, int n_item_tiles) {
  __shared__ float sU[32][65], sV[32][65];
  const int m0 = blockIdx.y * 64, n0 = blockIdx.x * 64;
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  float acc[4][4] = {};
  for (int k0 = 0; k0 < dim; k0 += 32) {
    for (int e = threadIdx.x; e < 64 * 32; e += 256) {
      const int r = e / 32, k = e % 32;
      sU[k][r] = (m0 + r < n_users && k0 + k < dim) ? U[(size_t)(m0 + r) * us + k0 + k] : 0.0f;
      sV[k][r] = (n0 + r < n_items && k0 + k < dim) ? V[(size_t)(n0 + r) * is + k0 + k] : 0.0f;
    }
    __syncthreads();
#pragma unroll 8
    for (int k = 0; k < 32; ++k) {
      float a[4], b[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) { a[i] = sU[k][ty * 4 + i]; b[i] = sV[k][tx * 4 + i]; }
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
  }
  const float mu_ = *mu;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int row = m0 + ty * 4 + i;
    float best = -INFINITY;
    int32_t best_i = -1;
    if (row < n_users) {
      const float bu = ub[row];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int col = n0 + tx * 4 + j;
        if (col < n_items) {
          float s = add_rn(add_rn(add_rn(acc[i][j], bu), ib[col]), mu_);
          if (scores) scores[(size_t)row * n_items + col] = s;
          if (s > best) { best = s; best_i = col; }
        }
      }
    }
    // best over the 16 threads that share this row (tx = 0..15): lower item index wins ties
#pragma unroll
    for (int o = 8; o > 0; o >>= 1) {
      const float ob = __shfl_xor_sync(0xffffffffu, best, o, 16);
      const int32_t oi = __shfl_xor_sync(0xffffffffu, best_i, o, 16);
      if (ob > best || (ob == best && oi >= 0 && (best_i < 0 || oi < best_i))) { best = ob; best_i = oi; }
    }
    if (tile_best && tx == 0 && row < n_users) {
      tile_best[(size_t)row * n_item_tiles + blockIdx.x] = best;
      tile_best_item[(size_t)row * n_item_tiles + blockIdx.x] = best_i;
    }
  }
}

__global__ void allpairs_best_reduce_kernel(const float* __restrict__ tile_best, const int32_t* __restrict__ tile_item,
                                            int n_users, int n_item_tiles, float* __restrict__ best_score,
                                            int32_t* __restrict__ best_item) {
  const int row = blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= n_users) return;
  float best = -INFINITY;
  int32_t bi = -1;
  for (int t = 0; t < n_item_tiles; ++t) {  // tiles in item order: strict > keeps the lowest item on ties
    const float s = tile_best[(size_t)row * n_item_tiles + t];
    if (s > best) { best = s; bi = tile_item[(size_t)row * n_item_tiles + t]; }
  }
  if (best_score) best_score[row] = best;
  if (best_item) best_item[row] = bi;
}

// ---- ranking consumer: the k best entries of every row of a score matrix ------------------------------------------
// forward.py:47-61 `get_ranking`: sort one user's scores over all items, keep the first 50.  One CTA per row; k rounds of
// a block-wide arg-max over the entries that come AFTER the previous pick in the total order (score descending, index
// ascending) -- no exclusion list, ties go to the lowest index (as in the fused top-1), NaN scores are never picked.
__global__ void __launch_bounds__(1024) topk_rows_kernel(const float* __restrict__ scores, int64_t n_cols, int64_t row_stride,
                                                         int k, float* __restrict__ out_val, int32_t* __restrict__ out_idx) {
  const float* row = scores + (size_t)blockIdx.x * row_stride;
  __shared__ float s_v[32];
  __shared__ int s_i[32];
  __shared__ float s_last_v;
  __shared__ int s_last_i;
  float last_v = INFINITY;
  int last_i = -1;
  for (int r = 0; r < k; ++r) {
    float bv = -INFINITY;
    int bi = -1;
    for (int64_t c = threadIdx.x; c < n_cols; c += blockDim.x) {
      const float v = row[c];
      const bool after = v < last_v || (v == last_v && (int)c > last_i);   // false for NaN
      if (after && (v > bv || (v == bv && (bi < 0 || (int)c < bi)) || bi < 0)) { bv = v; bi = (int)c; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
      const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
      if (oi >= 0 && (bi < 0 || ov > bv || (ov == bv && oi < bi))) { bv = ov; bi = oi; }
    }
    if ((threadIdx.x & 31) == 0) { s_v[threadIdx.x >> 5] = bv; s_i[threadIdx.x >> 5] = bi; }
    __syncthreads();
    if (threadIdx.x < 32) {
      const int nw = (blockDim.x + 31) >> 5;
      bv = threadIdx.x < nw ? s_v[threadIdx.x] : -INFINITY;
      bi = threadIdx.x < nw ? s_i[threadIdx.x] : -1;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
        const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
        if (oi >= 0 && (bi < 0 || ov > bv || (ov == bv && oi < bi))) { bv = ov; bi = oi; }
      }
      if (threadIdx.x == 0) {
        s_last_v = bv;
        s_last_i = bi;
        out_val[(size_t)blockIdx.x * k + r] = bi >= 0 ? bv : -INFINITY;
        out_idx[(size_t)blockIdx.x * k + r] = bi;   // -1: fewer than k rankable entries
      }
    }
    __syncthreads();
    last_v = s_last_v;
    last_i = s_last_i;
    if (last_i < 0) {  // nothing left: fill the rest
      for (int rr = r + 1 + threadIdx.x; rr < k; rr += blockDim.x) {
        out_val[(size_t)blockIdx.x * k + rr] = -INFINITY;
        out_idx[(size_t)blockIdx.x * k + rr] = -1;
      }
      break;
    }
    __syncthreads();
  }
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static int make_map(CUtensorMap* map, const float* table, int64_t rows, int dim, int64_t stride) {
  static EncodeTiledFn encode = nullptr;
  if (!encode) {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult q;
    TFR_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q));
    if (!fn || q != cudaDriverEntryPointSuccess) {
      set_error("cuTensorMapEncodeTiled is not available from the driver");
      return TFR_ERR_CUDA;
    }
    encode = (EncodeTiledFn)fn;
  }
  const cuuint64_t gdim[2] = {(cuuint64_t)dim, (cuuint64_t)rows};
  const cuuint64_t gstride[1] = {(cuuint64_t)stride * 4};  // row pitch: dim, or 3*dim for interleaved tables
  const cuuint32_t box[2] = {AP_KC, 128};
  const cuuint32_t estr[2] = {1, 1};
  const CUresult r = encode(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(table), gdim, gstride, box, estr,
                            CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed with CUresult %d (rows %lld dim %d)", (int)r, (long long)rows, dim);
    return TFR_ERR_CUDA;
  }
  return TFR_OK;
}

}  // namespace tfr

using namespace tfr;

extern "C" int tfr_topk_rows(const float* scores, int64_t n_rows, int64_t n_cols, int64_t row_stride, int32_t k,
                             float* out_val, int32_t* out_idx, void* stream) {
  TFR_CHECK_ARG(n_rows >= 0 && n_cols >= 0 && k > 0 && n_cols < ((int64_t)1 << 31) && n_rows < ((int64_t)1 << 31));
  if (n_rows == 0) return TFR_OK;
  TFR_CHECK_ARG(scores && out_val && out_idx && (row_stride == 0 || row_stride >= n_cols));
  topk_rows_kernel<<<(unsigned)n_rows, 1024, 0, (cudaStream_t)stream>>>(scores, n_cols, row_stride ? row_stride : n_cols, k,
                                                                      out_val, out_idx);
  TFR_LAUNCH_CHECK();
  return TFR_OK;
}

extern "C" int64_t tfr_allpairs_workspace_bytes(int64_t n_users, int64_t n_items, int32_t dim, int32_t use_tensor_cores) {
  if (n_users < 0 || n_items < 0 || dim <= 0) return TFR_ERR_INVALID;
  if (use_tensor_cores && dim % 32 == 0 && dim <= 128) return 256;
  const int64_t tiles = (n_items + 63) / 64;
  return 2 * align_up(n_users * tiles * 4, 256) + 256;
}

static int launch_allpairs_tc(const float* user_feat, const float* item_feat, const float* user_bias,
                              const float* item_bias, const float* mu, int64_t n_users, int64_t n_items, int32_t dim,
                              int64_t user_stride, int64_t item_stride, const ApConsumers& cs, cudaStream_t st) {
  if (dim % 32 != 0 || dim > 128) {
    set_error("tcgen05 all-pairs path needs dim %% 32 == 0 and dim <= 128 (got %d): pass use_tensor_cores = 0", dim);
    return TFR_ERR_INVALID;
  }
  TFR_CHECK_ARG(((uintptr_t)user_feat % 16 == 0) && ((uintptr_t)item_feat % 16 == 0));
  CUtensorMap ma, mb;
  int rc;
  if ((rc = make_map(&ma, user_feat, n_users, dim, user_stride))) return rc;
  if ((rc = make_map(&mb, item_feat, n_items, dim, item_stride))) return rc;
  const int kch = dim / 32;
  const size_t smem = (size_t)3 * kch * AP_CHUNK_BYTES + 1024 + 128 + (2 * 256 + 512) * 4 + 256 * 8 + 64;
  const unsigned grid = (unsigned)((n_users + AP_BM - 1) / AP_BM);
  const bool topk = cs.cand_val != nullptr, obs = cs.obs_indptr != nullptr, excl = cs.excl_indptr != nullptr;
  TFR_CHECK_ARG(!excl || (topk && !obs));   // the exclusion walk exists only in the top-k sweep
#define TFR_AP_LAUNCH(KC_, TK_, OB_, EX_)                                                                              \
  {                                                                                                                    \
    TFR_CUDA(cudaFuncSetAttribute(allpairs_tc_kernel<KC_, TK_, OB_, EX_>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
    allpairs_tc_kernel<KC_, TK_, OB_, EX_><<<grid, AP_THREADS, smem, st>>>(ma, mb, user_bias, item_bias, mu, (int)n_users, \
                                                                           (int)n_items, cs);                         \
  }
#define TFR_AP_CASE(KC_)                                          \
  if (kch == KC_) {                                               \
    if (excl) TFR_AP_LAUNCH(KC_, true, false, true)               \
    else if (topk && obs) TFR_AP_LAUNCH(KC_, true, true, false)   \
    else if (topk) TFR_AP_LAUNCH(KC_, true, false, false)         \
    else if (obs) TFR_AP_LAUNCH(KC_, false, true, false)          \
    else TFR_AP_LAUNCH(KC_, false, false, false)                  \
  }
  TFR_AP_CASE(1) TFR_AP_CASE(2) TFR_AP_CASE(3) TFR_AP_CASE(4)
#undef TFR_AP_CASE
#undef TFR_AP_LAUNCH
  TFR_LAUNCH_CHECK();
  return TFR_OK;
}

static int ap_exact_ctas() { return 2 * sm_count(); }

// Candidates the sweep keeps per row-half.  A buffer of C = 4K entries must take the K kept after a compaction plus the up
// to 32 appends of the next column chunk (the sweep compacts a buffer with more than C - 32 entries after each chunk):
// 4K >= K + 32, so a smaller n_cand keeps 11.  More candidates than asked only make the certificate easier to meet.
static int ap_buffer_k(int n_cand) { return n_cand > 11 ? n_cand : 11; }

extern "C" int64_t tfr_allpairs_topk_workspace_bytes(int64_t n_users, int64_t n_items, int32_t k, int32_t n_cand) {
  if (n_users < 0 || n_items < 0 || k <= 0 || n_cand < k || n_cand > AP_MAX_CAND) return TFR_ERR_INVALID;
  n_cand = ap_buffer_k(n_cand);
  return 256 + 2 * align_up(8 * n_users * (int64_t)n_cand * 4, 256) + 3 * align_up(2 * n_users * 4, 256) +
         align_up((int64_t)ap_exact_ctas() * n_items * 8, 256) + 256;
}

// Per-user top-k ranking over ALL items (forward.py:47-61 for every user at once) and / or the squared error on the
// observed pairs (als3.py:110-120,139-143), consumed in the epilogue of the tcgen05 GEMM.  One launcher for both entry
// points: tfr_allpairs_consume (no exclusion, tcgen05 dims only) and tfr_allpairs_rank_excluding (top-k only, optional
// exclusion list, any dim <= 512).  any_dim: a dim the tcgen05 sweep cannot take (dim % 32 != 0 or dim > 128) sends EVERY
// row through allpairs_exact_rows_kernel, O(n_users * n_items * (dim + k)) on CUDA cores -- fine at the ML-1M shape, not
// meant for ML-25M.
static int allpairs_consume_impl(const float* user_feat, const float* item_feat, const float* user_bias,
                                 const float* item_bias, const float* mu, int64_t n_users, int64_t n_items, int32_t dim,
                                 int64_t user_stride, int64_t item_stride, int32_t k, int32_t n_cand, double* topk_val,
                                 int32_t* topk_idx, int32_t* n_uncertified, const int64_t* obs_indptr,
                                 const int32_t* obs_item, const float* obs_rate, double* row_se,
                                 const int64_t* excl_indptr, const int32_t* excl_item, bool any_dim, void* workspace,
                                 int64_t workspace_bytes, void* stream) {
  if (user_stride == 0) user_stride = dim;
  if (item_stride == 0) item_stride = dim;
  TFR_CHECK_ARG(user_stride >= dim && item_stride >= dim);
  TFR_CHECK_ARG(n_users >= 0 && n_items >= 0 && dim > 0 && n_users < ((int64_t)1 << 31) && n_items < ((int64_t)1 << 31));
  const bool topk = k > 0;
  const bool obs = obs_indptr != nullptr;
  TFR_CHECK_ARG(topk || obs);
  TFR_CHECK_ARG(!topk || (topk_val && topk_idx && n_uncertified && n_cand >= k && n_cand <= AP_MAX_CAND && dim <= 512));
  TFR_CHECK_ARG(!obs || (obs_item && obs_rate && row_se));
  TFR_CHECK_ARG(!excl_indptr || (topk && !obs && excl_item));
  if (n_users == 0 || n_items == 0) return TFR_OK;
  TFR_CHECK_ARG(user_feat && item_feat && user_bias && item_bias && mu);
  cudaStream_t st = (cudaStream_t)stream;
  ApConsumers cs;
  memset(&cs, 0, sizeof(cs));
  float* vmax2 = nullptr;
  int32_t* uncert = nullptr;
  double* scratch = nullptr;
  if (topk) {
    if (!workspace || workspace_bytes < tfr_allpairs_topk_workspace_bytes(n_users, n_items, k, n_cand)) {
      set_error("all-pairs top-k workspace too small");
      return TFR_ERR_WORKSPACE;
    }
    n_cand = ap_buffer_k(n_cand);
    char* w = reinterpret_cast<char*>(align_up((int64_t)(uintptr_t)workspace, 256));
    vmax2 = reinterpret_cast<float*>(w); w += 256;
    cs.cand_val = reinterpret_cast<float*>(w); w += align_up(8 * n_users * (int64_t)n_cand * 4, 256);
    cs.cand_idx = reinterpret_cast<int32_t*>(w); w += align_up(8 * n_users * (int64_t)n_cand * 4, 256);
    cs.cand_cnt = reinterpret_cast<int32_t*>(w); w += align_up(2 * n_users * 4, 256);
    cs.cand_thr = reinterpret_cast<float*>(w); w += align_up(2 * n_users * 4, 256);
    uncert = reinterpret_cast<int32_t*>(w); w += align_up(2 * n_users * 4, 256);   // >= n_users rows: all of them fit
    scratch = reinterpret_cast<double*>(w);
    cs.K = n_cand;
    TFR_CUDA(cudaMemsetAsync(vmax2, 0, 256, st));
    TFR_CUDA(cudaMemsetAsync(n_uncertified, 0, sizeof(int32_t), st));
  }
  if (obs) { cs.obs_indptr = obs_indptr; cs.obs_item = obs_item; cs.obs_rate = obs_rate; cs.row_se = row_se; }
  cs.excl_indptr = excl_indptr; cs.excl_item = excl_item;
  if (any_dim && (dim % 32 != 0 || dim > 128)) {   // (top-k only: checked above) every row through the exact path
    allpairs_all_rows_kernel<<<(unsigned)((n_users + 255) / 256 < 1024 ? (n_users + 255) / 256 : 1024), 256, 0, st>>>(
        (int)n_users, uncert, n_uncertified);
    TFR_LAUNCH_CHECK();
    allpairs_exact_rows_kernel<<<(unsigned)ap_exact_ctas(), 1024, 0, st>>>(user_feat, item_feat, user_bias, item_bias, mu,
                                                                         (int)n_items, dim, user_stride, item_stride, uncert,
                                                                         n_uncertified, k, scratch, topk_val, topk_idx,
                                                                         excl_indptr, excl_item);
    TFR_LAUNCH_CHECK();
    return TFR_OK;
  }
  const int stages = tune(TUNE_AP_STAGES);
  int rc = TFR_OK;
  if (!topk || (stages & 1))
    rc = launch_allpairs_tc(user_feat, item_feat, user_bias, item_bias, mu, n_users, n_items, dim, user_stride, item_stride,
                            cs, st);
  if (rc) return rc;
  if (topk && (stages & 2)) {
    allpairs_vmax2_kernel<<<(unsigned)((n_items * 32 + 255) / 256), 256, 0, st>>>(item_feat, item_bias, mu, (int)n_items, dim,
                                                                               item_stride, vmax2);
    TFR_LAUNCH_CHECK();
    allpairs_rescore_kernel<<<(unsigned)((n_users + RS_WARPS - 1) / RS_WARPS), 32 * RS_WARPS, 0, st>>>(
        user_feat, item_feat, user_bias, item_bias, mu, (int)n_users, (int)n_items, dim, user_stride, item_stride,
        cs.cand_val, cs.cand_idx, cs.cand_cnt, cs.cand_thr, n_cand, k, vmax2, topk_val, topk_idx, uncert, n_uncertified,
        excl_indptr, excl_item);
    TFR_LAUNCH_CHECK();
    if (stages & 4)
    allpairs_exact_rows_kernel<<<(unsigned)ap_exact_ctas(), 1024, 0, st>>>(user_feat, item_feat, user_bias, item_bias, mu,
                                                                         (int)n_items, dim, user_stride, item_stride, uncert,
                                                                         n_uncertified, k, scratch, topk_val, topk_idx,
                                                                         excl_indptr, excl_item);
    TFR_LAUNCH_CHECK();
  }
  return TFR_OK;
}

extern "C" int tfr_allpairs_consume(const float* user_feat, const float* item_feat, const float* user_bias,
                                    const float* item_bias, const float* mu, int64_t n_users, int64_t n_items, int32_t dim,
                                    int64_t user_stride, int64_t item_stride, int32_t k, int32_t n_cand, double* topk_val,
                                    int32_t* topk_idx, int32_t* n_uncertified, const int64_t* obs_indptr,
                                    const int32_t* obs_item, const float* obs_rate, double* row_se, void* workspace,
                                    int64_t workspace_bytes, void* stream) {
  return allpairs_consume_impl(user_feat, item_feat, user_bias, item_bias, mu, n_users, n_items, dim, user_stride,
                               item_stride, k, n_cand, topk_val, topk_idx, n_uncertified, obs_indptr, obs_item, obs_rate,
                               row_se, nullptr, nullptr, false, workspace, workspace_bytes, stream);
}

extern "C" int tfr_allpairs_rank_excluding(const float* user_feat, const float* item_feat, const float* user_bias,
                                           const float* item_bias, const float* mu, int64_t n_users, int64_t n_items,
                                           int32_t dim, int64_t user_stride, int64_t item_stride, int32_t k, int32_t n_cand,
                                           const int64_t* excl_indptr, const int32_t* excl_item, double* topk_val,
                                           int32_t* topk_idx, int32_t* n_uncertified, void* workspace,
                                           int64_t workspace_bytes, void* stream) {
  TFR_CHECK_ARG(k > 0);
  return allpairs_consume_impl(user_feat, item_feat, user_bias, item_bias, mu, n_users, n_items, dim, user_stride,
                               item_stride, k, n_cand, topk_val, topk_idx, n_uncertified, nullptr, nullptr, nullptr, nullptr,
                               excl_indptr, excl_item, true, workspace, workspace_bytes, stream);
}

extern "C" int tfr_allpairs(const float* user_feat, const float* item_feat, const float* user_bias,
                            const float* item_bias, const float* mu, int64_t n_users, int64_t n_items, int32_t dim,
                            int64_t user_stride, int64_t item_stride, int32_t use_tensor_cores, float* scores,
                            float* best_score, int32_t* best_item, void* workspace, int64_t workspace_bytes,
                            void* stream) {
  if (user_stride == 0) user_stride = dim;
  if (item_stride == 0) item_stride = dim;
  TFR_CHECK_ARG(user_stride >= dim && item_stride >= dim);
  TFR_CHECK_ARG(n_users >= 0 && n_items >= 0 && dim > 0 && n_users < ((int64_t)1 << 31) && n_items < ((int64_t)1 << 31));
  if (n_users == 0 || n_items == 0) return TFR_OK;
  TFR_CHECK_ARG(user_feat && item_feat && user_bias && item_bias && mu && (scores || best_score || best_item));
  cudaStream_t st = (cudaStream_t)stream;
  if (use_tensor_cores) {
    ApConsumers cs;
    memset(&cs, 0, sizeof(cs));
    cs.scores = scores; cs.best_score = best_score; cs.best_item = best_item;
    return launch_allpairs_tc(user_feat, item_feat, user_bias, item_bias, mu, n_users, n_items, dim, user_stride,
                              item_stride, cs, st);
  }
  const int tiles = (int)((n_items + 63) / 64);
  float* tile_best = nullptr;
  int32_t* tile_item = nullptr;
  if (best_score || best_item) {
    if (!workspace || workspace_bytes < tfr_allpairs_workspace_bytes(n_users, n_items, dim, 0)) {
      set_error("all-pairs workspace too small");
      return TFR_ERR_WORKSPACE;
    }
    char* w = reinterpret_cast<char*>(align_up((int64_t)(uintptr_t)workspace, 256));
    tile_best = reinterpret_cast<float*>(w);
    tile_item = reinterpret_cast<int32_t*>(w + align_up(n_users * tiles * 4, 256));
  }
  dim3 grid((unsigned)tiles, (unsigned)((n_users + 63) / 64));
  allpairs_simt_kernel<<<grid, 256, 0, st>>>(user_feat, item_feat, user_bias, item_bias, mu, (int)n_users, (int)n_items,
                                             dim, user_stride, item_stride, scores, tile_best, tile_item, tiles);
  TFR_LAUNCH_CHECK();
  if (tile_best) {
    allpairs_best_reduce_kernel<<<(unsigned)((n_users + 255) / 256), 256, 0, st>>>(tile_best, tile_item, (int)n_users,
                                                                                   tiles, best_score, best_item);
    TFR_LAUNCH_CHECK();
  }
  return TFR_OK;
}
