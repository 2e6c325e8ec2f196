// Deterministic exclusive prefix sum of int32 counts into int64 offsets: three phases (block sums, scan of the sums,
// apply).  The count -> scan -> fill builders of CSR arrays on the device share it (metrics.cu, shard_rank.cu).
#pragma once
#include "common.cuh"

namespace tfr {

constexpr int SCAN_THREADS = 256, SCAN_ITEMS = 8, SCAN_TILE = SCAN_THREADS * SCAN_ITEMS;

// block-wide exclusive scan of one value per thread; returns the thread's exclusive prefix, *total = block total
__device__ __forceinline__ int64_t block_exclusive_scan(int64_t x, int64_t* s_warp, int64_t* total) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int64_t incl = x;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int64_t y = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += y;
  }
  if (lane == 31) s_warp[warp] = incl;
  __syncthreads();
  int64_t off = 0, tot = 0;
  for (int w = 0; w < SCAN_THREADS / 32; ++w) {
    if (w < warp) off += s_warp[w];
    tot += s_warp[w];
  }
  __syncthreads();
  if (total) *total = tot;
  return off + incl - x;
}

// phase 1: per-tile sums of in[] (int32 counts)
static __global__ void __launch_bounds__(SCAN_THREADS) scan_tile_sums_kernel(const int32_t* __restrict__ in, int64_t n,
                                                                     int64_t* __restrict__ tile_sums) {
  __shared__ int64_t s_warp[SCAN_THREADS / 32];
  const int64_t base = (int64_t)blockIdx.x * SCAN_TILE;
  int64_t x = 0;
#pragma unroll
  for (int j = 0; j < SCAN_ITEMS; ++j) {
    const int64_t i = base + (int64_t)threadIdx.x * SCAN_ITEMS + j;
    if (i < n) x += in[i];
  }
  int64_t tot;
  block_exclusive_scan(x, s_warp, &tot);
  if (threadIdx.x == 0) tile_sums[blockIdx.x] = tot;
}
// phase 2: exclusive scan of the tile sums in place (one CTA), total -> tile_sums[n_tiles]
static __global__ void __launch_bounds__(SCAN_THREADS) scan_of_sums_kernel(int64_t* __restrict__ tile_sums, int64_t n_tiles) {
  __shared__ int64_t s_warp[SCAN_THREADS / 32];
  __shared__ int64_t s_carry;
  if (threadIdx.x == 0) s_carry = 0;
  __syncthreads();
  for (int64_t b0 = 0; b0 < n_tiles; b0 += SCAN_THREADS) {
    const int64_t i = b0 + threadIdx.x;
    const int64_t x = i < n_tiles ? tile_sums[i] : 0;
    int64_t tot;
    const int64_t ex = block_exclusive_scan(x, s_warp, &tot);
    const int64_t carry = s_carry;
    if (i < n_tiles) tile_sums[i] = carry + ex;
    __syncthreads();
    if (threadIdx.x == 0) s_carry = carry + tot;
    __syncthreads();
  }
  if (threadIdx.x == 0) tile_sums[n_tiles] = s_carry;
}
// phase 3: out[i] = exclusive prefix of in[0..i), out[n] = total
static __global__ void __launch_bounds__(SCAN_THREADS) scan_apply_kernel(const int32_t* __restrict__ in, int64_t n,
                                                                 const int64_t* __restrict__ tile_sums,
                                                                 int64_t* __restrict__ out) {
  __shared__ int64_t s_warp[SCAN_THREADS / 32];
  const int64_t base = (int64_t)blockIdx.x * SCAN_TILE;
  int32_t v[SCAN_ITEMS];
  int64_t x = 0;
#pragma unroll
  for (int j = 0; j < SCAN_ITEMS; ++j) {
    const int64_t i = base + (int64_t)threadIdx.x * SCAN_ITEMS + j;
    v[j] = i < n ? in[i] : 0;
    x += v[j];
  }
  int64_t run = tile_sums[blockIdx.x] + block_exclusive_scan(x, s_warp, nullptr);
#pragma unroll
  for (int j = 0; j < SCAN_ITEMS; ++j) {
    const int64_t i = base + (int64_t)threadIdx.x * SCAN_ITEMS + j;
    if (i < n) out[i] = run;
    run += v[j];
  }
  if (blockIdx.x == gridDim.x - 1 && threadIdx.x == 0) out[n] = tile_sums[gridDim.x];
}

// out [n + 1] int64 = exclusive scan of in [n] int32; tile_sums: ceil(n / SCAN_TILE) + 1 int64 of scratch
static int exclusive_scan(const int32_t* in, int64_t n, int64_t* out, int64_t* tile_sums, cudaStream_t st) {
  const int64_t n_tiles = (n + SCAN_TILE - 1) / SCAN_TILE;
  scan_tile_sums_kernel<<<(unsigned)n_tiles, SCAN_THREADS, 0, st>>>(in, n, tile_sums);
  TFR_LAUNCH_CHECK();
  scan_of_sums_kernel<<<1, SCAN_THREADS, 0, st>>>(tile_sums, n_tiles);
  TFR_LAUNCH_CHECK();
  scan_apply_kernel<<<(unsigned)n_tiles, SCAN_THREADS, 0, st>>>(in, n, tile_sums, out);
  TFR_LAUNCH_CHECK();
  return TFR_OK;
}
static int64_t scan_tiles(int64_t n) { return (n + SCAN_TILE - 1) / SCAN_TILE + 1; }

}  // namespace tfr
