// Shared device/host helpers for libtfrecomm (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/tfrecomm.h"

namespace tfr {

void set_error(const char* fmt, ...);
int sm_count();

// Tuning knobs: the ONE piece of process-wide state of the library (include/tfrecomm.h: tfr_tune_set / tfr_tune_get).
// A knob's value is, in this order: what tfr_tune_set gave it, the environment variable TFR_<NAME> read at first use,
// its default.  Every launch reads its knobs through tune(): nothing is cached at the call sites.
enum TuneKey {
  TUNE_SMEM_CARVEOUT,     // preferred shared-memory carve-out (%) given to every kernel of the step (see prep_kernel)
  TUNE_TILES_CARVEOUT,    // < 0: same as SMEM_CARVEOUT
  TUNE_SEG_MAX_UNITS,     // segment sums: force 1 / 2 / 4 units per lane (0 = heuristic)
  TUNE_SEG_TILE,          // segment sums: force tiles of 8 / 16 / 32 entries (0 = heuristic)
  TUNE_STREAM_COPY_ONLY,  // LDG pass without arithmetic (memory ceiling experiment)
  TUNE_STREAM_LD, TUNE_STREAM_ST,  // cache hints of the LDG pass (0 = .cs, 1 = default, 2 = .cg, 3 = .lu / .wt)
  TUNE_STREAM_CTAS_PER_SM, TUNE_STREAM_UNROLL, TUNE_STREAM_THREADS, TUNE_STREAM_DYNAMIC,
  TUNE_PASS_RING,         // 1: interleaved tables take the TMA-bulk ring pass (adam_ring.cu), 0: the LDG pass
  TUNE_RING_STAGES, TUNE_RING_STAGE_KB, TUNE_RING_THREADS, TUNE_RING_L2_HINT, TUNE_RING_CTAS_PER_SM,
  TUNE_RING_SLOT_MODE,
  TUNE_AP_STAGES,         // debug: which stages of tfr_allpairs_consume's ranking run (1 sweep | 2 rescore | 4 exact rows)
  TUNE_TL_EVERY_CTA,      // debug timeline: the pass's exit stamp from every CTA instead of a sample
  TUNE_PDL,               // 1: programmatic dependent launch along the step's critical path (see pdl_wait)
  TUNE_SORT_SPLIT,        // 1: every id sort in its one-launch-per-phase form (default: only inside the feed graph)
  TUNE_RANK_CHUNK,        // tfr_rank_users: items per selection chunk (a multiple of 1024, 1024 .. 16384)
  TUNE_RANK_STAGES,       // debug: which kernels of tfr_rank_users run (1 score | 2 select | 4 merge)
  TUNE_COUNT
};
int tune(TuneKey k);
// Gives every kernel of the step the SAME shared-memory carve-out.  An SM cannot host CTAs of two kernels
// whose carve-outs differ, so without this the persistent streaming pass (no shared memory -> "max L1")
// keeps the forward / sort / segment-sum kernels (which use shared memory) off every SM until it drains.
void prep_kernel(const void* fn);
// same, for a kernel whose resident CTAs need `smem_per_sm` bytes of shared memory per SM: the common carve-out if
// that is enough, else the smallest percentage that is (a preferred carve-out is a ceiling for occupancy: the driver
// only guarantees that ONE CTA fits)
void prep_kernel_carveout(const void* fn, size_t smem_per_sm);
// tfr_dedup_sort_pairs_tl with the launch form chosen by the caller: split = one launch per phase, no grid barrier
int dedup_sort_pairs_impl(const int32_t* ids_a, int64_t max_id_a, int32_t* sorted_ids_a, int32_t* sorted_pos_a,
                          const int32_t* ids_b, int64_t max_id_b, int32_t* sorted_ids_b, int32_t* sorted_pos_b, int64_t n,
                          void* workspace, int64_t workspace_bytes, const tfr_opt_scalars* opt, void* stream, bool split);
#define TFR_PREP(kernel) tfr::prep_kernel(reinterpret_cast<const void*>(kernel))

#define TFR_CHECK_ARG(cond)                                                        \
  do {                                                                             \
    if (!(cond)) {                                                                 \
      tfr::set_error("%s:%d: invalid argument: %s", __FILE__, __LINE__, #cond);    \
      return TFR_ERR_INVALID;                                                      \
    }                                                                              \
  } while (0)

#define TFR_CUDA(expr)                                                             \
  do {                                                                             \
    cudaError_t e__ = (expr);                                                      \
    if (e__ != cudaSuccess) {                                                      \
      tfr::set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(e__)); \
      return TFR_ERR_CUDA;                                                         \
    }                                                                              \
  } while (0)

#define TFR_LAUNCH_CHECK() TFR_CUDA(cudaGetLastError())

// ---- programmatic dependent launch (PDL) ----------------------------------------------------------------------
// The kernels of the step's critical path (segment sums -> fix-up -> table pass -> next step's segment sums) are
// launched with programmaticStreamSerializationAllowed: a kernel's CTAs become resident while its predecessor drains
// and block at pdl_wait() until the predecessor grid has completed and flushed -- the launch latency between two
// kernels disappears from the critical path.  Every kernel calls pdl_wait() BEFORE pdl_launch_dependents(), so a
// kernel can only start once its predecessor's predecessor is complete (dependencies stay transitive).  Both are
// no-ops in a kernel that was launched the plain way.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

#ifdef __CUDACC__
template <typename... KArgs, typename... Args>
inline cudaError_t launch_kernel(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, bool pdl,
                                 Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  if (pdl) {
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
  }
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}
#endif

// ---- explicit-rounding fp32 arithmetic: every TensorFlow op is its own rounding, never an FMA ----
__device__ __forceinline__ float mul_rn(float a, float b) { return __fmul_rn(a, b); }
__device__ __forceinline__ float add_rn(float a, float b) { return __fadd_rn(a, b); }
__device__ __forceinline__ float sub_rn(float a, float b) { return __fsub_rn(a, b); }
__device__ __forceinline__ float div_rn(float a, float b) { return __fdiv_rn(a, b); }
__device__ __forceinline__ float sqrt_rn(float a) { return __fsqrt_rn(a); }

// ---- cache-hinted 128-bit / 32-bit accesses ---------------------------------------------------
// Streaming table data (the Adam pass reads and writes every byte exactly once per step): .cs =
// cache-streaming (evict-first), so the pass does not push the batch's gathered rows out of L2.
__device__ __forceinline__ float4 ld_stream_f4(const float4* p) {
  float4 r;
  asm volatile("ld.global.cs.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
               : "l"(p));
  return r;
}
__device__ __forceinline__ void st_stream_f4(float4* p, const float4& v) {
  asm volatile("st.global.cs.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(v.x),
               "f"(v.y), "f"(v.z), "f"(v.w)
               : "memory");
}
__device__ __forceinline__ float ld_stream_f1(const float* p) {
  float r;
  asm volatile("ld.global.cs.f32 %0, [%1];" : "=f"(r) : "l"(p));
  return r;
}
__device__ __forceinline__ void st_stream_f1(float* p, float v) {
  asm volatile("st.global.cs.f32 [%0], %1;" ::"l"(p), "f"(v) : "memory");
}
// Gathered rows: read-only path.  Safe because no kernel that gathers also writes the tables (they are
// only written by the Adam kernels of the previous step), and the rows are re-read from L2 by the
// segment-sum and the slice-row update.
__device__ __forceinline__ float4 ld_gather_f4(const float4* p) {
  float4 r;
  asm("ld.global.nc.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
               : "l"(p));
  return r;
}
__device__ __forceinline__ float ld_gather_f1(const float* p) {
  float r;
  asm("ld.global.nc.f32 %0, [%1];" : "=f"(r) : "l"(p));
  return r;
}

// ---- debug timeline (no nsys on the box): earliest block entry / latest warp exit per kernel --------------
__device__ __forceinline__ unsigned long long gtimer() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
struct TlScope {
  unsigned long long* tl;
  int slot;
  __device__ __forceinline__ TlScope(const tfr_opt_scalars* opt, int slot_, bool every_cta = false)
      : tl(nullptr), slot(slot_) {
    if (opt) tl = reinterpret_cast<unsigned long long*>(opt->timeline);
    // sampled so that the stamps do not serialise on one address: entry = first CTAs, exit = every 64th CTA
    // and the grid's last 8 (which are scheduled last), one warp each; every_cta: kernels whose CTAs finish at very
    // different times (the fix-up: the CTA with the hottest row ends last, whatever its index)
    if (tl) {
      const unsigned bid = blockIdx.x + blockIdx.y * gridDim.x, nb = gridDim.x * gridDim.y;
      sampled = every_cta || bid + 8 >= nb || (bid & 63u) == 0;
      if (bid < 4 && threadIdx.x == 0) atomicMin(tl + slot, gtimer());
    }
  }
  __device__ __forceinline__ ~TlScope() {
    if (tl && sampled && (threadIdx.x & 31) == 0) atomicMax(tl + TFR_TL_SLOTS + slot, gtimer());
  }
  bool sampled = false;
};

// lane-group (L = 1..32, power of two) butterfly sum; every lane of the group gets the total.
template <int L>
__device__ __forceinline__ float group_sum(float x) {
#pragma unroll
  for (int o = L / 2; o > 0; o >>= 1) x = add_rn(x, __shfl_xor_sync(0xffffffffu, x, o, L));
  return x;
}

// TF: tf.sigmoid (Eigen scalar_logistic_op) = 1/(1+exp(-x)); tf.round = round-half-to-even.
__device__ __forceinline__ float sigmoid_tf(float x) { return div_rn(1.0f, add_rn(1.0f, expf(-x))); }

// d cost / d logits (SURVEY 8a rows a9/a10).  README: l2_loss(infer-rate) -> x - z (ops.py:124).
// fork: sigmoid_cross_entropy_with_logits (ops.py:125), autodiff of TF's relu(x)-x*z+log1p(exp(-|x|)).
__device__ __forceinline__ float dloss(int flags, float x, float z) {
  if (!(flags & TFR_LOSS_SIGMOID_CE)) return sub_rn(x, z);
  const bool cond = x >= 0.0f;
  const float n = cond ? -x : x;
  const float t = expf(n);
  const float sgm = mul_rn(div_rn(1.0f, add_rn(1.0f, t)), t);
  const float g = sub_rn(cond ? 1.0f : 0.0f, z);
  return add_rn(g, cond ? -sgm : sgm);
}

inline int64_t align_up(int64_t x, int64_t a) { return (x + a - 1) / a * a; }

// lane-group geometry for a row of `dim` floats: VEC = 4 when rows are 16-byte aligned (dim % 4 == 0),
// else scalar; L = lanes cooperating on one row (power of two <= 32).
struct RowGeom {
  int vec, lanes;
};
inline RowGeom row_geom(int dim) {
  RowGeom g;
  g.vec = (dim % 4 == 0) ? 4 : 1;
  int units = dim / g.vec;
  int l = 1;
  while (l < units && l < 32) l <<= 1;
  g.lanes = l;
  return g;
}

}  // namespace tfr
