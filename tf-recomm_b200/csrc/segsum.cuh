// The ordered segment sums' shared definitions: segsum.cu (every geometry and model variant) and chain.cu (the lean
// tiles kernel of the default path) write the same partial rows, tile kinds and work lists for the same fix-up.
#pragma once
#include "common.cuh"

namespace tfr {

struct SegSide {
  const int32_t* sid;      // sorted ids of this table
  const int32_t* spos;     // batch positions
  const int32_t* partner;  // the OTHER id column of the batch (items for the user table)
  const float* own_feat;   // this table's rows
  const float* partner_feat;
  int64_t own_stride, partner_stride;  // floats between consecutive rows (dim, or 3*dim for interleaved tables)
  const float* own_bias;
  const float* partner_bias;  // fused forward only
  float *gsum, *gsum_b, *cont, *cont_b, *tail, *tail_b;
  uint8_t* kind;  // per tile: TILE_MID | TILE_START (see segsum_fixup_kernel)
  int32_t* fix_list;     // work list of the fix-up: the TILE_START tiles, in no particular order
  uint32_t* fix_count;   // its length (zeroed by the id sort and by the fix-up's last CTA)
  int64_t* slot;  // [rows] row -> (step stamp << 32 | head index of its run, where its gsum lives)
  int32_t n_rows; // ids >= n_rows mark occurrences owned by another rank (row-sharded mode): skipped
  // factorization-machine mode (xval != null): the sorted ids are FEATURE ids of the batch's non-zeros, position =
  // index p of the non-zero; partner row = sums[rowof[p]] (the CSR row's sum_i V_i x_i), and
  //   g_V = e_r * (x_p * (sums_r - V_f * x_p)) + reg * V_f        (Rendle 2010 eq. 4; forward.py:21-22's model)
  //   g_W = e_r * x_p (+ reg * W_f if TFR_REG_BIAS)
  const float* xval;      // [nnz] feature values
  const int32_t* rowof;   // [nnz] CSR row of every non-zero
  int is_item;
};

// The forward fused into the segment sums (FUSED = true): a tile holds, for every occurrence, the own row and the
// partner row, i.e. everything ops.py:44-47 needs -- each side recomputes logits = ((sum_k u*v' + mu) + b_u) + b_i
// and d cost/d logits itself (same operands, same order on both sides: bit-identical e), the user side writes
// logits / infer and the fixed-order partial sums of e and of the float64 squared error.  No forward kernel, no
// err array, one launch less in front of the table pass.
struct FwdArgs {
  const float* mu;
  const float* rates;
  float *logits, *infer;       // by batch position; optional
  float* partials;             // [gridDim.x] per-CTA sums of e (user side)
  double* se_partials;
};

// tile classification written by the tiles kernel, read by the fix-up:
//   TILE_MID   the whole tile is ONE run that began in an earlier tile and goes on into the next
//   TILE_START the tile's last run begins here and goes on into the next tile (tail[t] is valid)
constexpr uint8_t TILE_MID = 1, TILE_START = 2;

constexpr int SEG_THREADS = 128;  // CTA of the tiles kernels

__device__ __forceinline__ int64_t pack_slot(uint32_t stamp, int64_t k) {
  return (int64_t)(((uint64_t)stamp << 32) | (uint32_t)k);
}

// opts a tiles kernel in to `smem` bytes of dynamic shared memory and gives it the step's carve-out (once per kernel)
int prep_tiles(const void* fn, size_t smem);

// chain.cu: the tiles kernel of the default path -- fused forward, README model (no |v|, no SGD), rows of four units
// of float4 per lane over L = 8, 16 or 32 lanes.  Same results, bit for bit, as segsum_tiles_kernel<4, L, 4, true,
// false> at the same tile; the fix-up that follows is segsum.cu's.
bool chain_tiles_supported(int lanes, int tile);
int launch_chain_tiles(const SegSide& su, const SegSide& si, const FwdArgs& fw, const tfr_opt_scalars* opt, int64_t B,
                       int dim, int n_tiles, int tile, int lanes, dim3 grid, bool pdl, cudaStream_t st);

}  // namespace tfr
