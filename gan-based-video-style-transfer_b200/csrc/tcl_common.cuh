// Shared device helpers: vector I/O, fixed-order reductions, the in-launch pair/batch finalisation.
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/tcl_b200.h"
#include "tcl_math.cuh"

namespace tcl {

constexpr int kV = V_ATEN_CUDA;  // arithmetic flavour of the product kernels (see tcl_math.cuh)
#ifndef TCL_WARPS
#define TCL_WARPS 8
#endif
constexpr int kWarps = TCL_WARPS;  // warps per CTA
constexpr int kThreads = 32 * kWarps;
constexpr float kNearBand = 1e-6f;  // north_star's near-threshold exemption band

enum : int { MASK_NONE = 0, MASK_GIVEN = 1, MASK_COMPUTED = 2 };

__host__ __device__ constexpr size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// ---------------------------------------------------------------------------------------------
// scalar frame I/O (fp32 / bf16 <-> fp32 registers)
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ float ld_stream(const float* p) { return __ldcs(p); }
__device__ __forceinline__ float ld_stream(const __nv_bfloat16* p) {
  return __bfloat162float(__ushort_as_bfloat16(__ldcs(reinterpret_cast<const unsigned short*>(p))));
}
// read-only gather through the non-coherent cache (bilinear taps that neighbouring lanes re-read)
__device__ __forceinline__ float ld_gather(const float* p) { return __ldg(p); }
__device__ __forceinline__ float ld_gather(const __nv_bfloat16* p) { return __bfloat162float(__ldg(p)); }
__device__ __forceinline__ void st_stream(float* p, float v) { __stcs(p, v); }
__device__ __forceinline__ void st_stream(__nv_bfloat16* p, float v) {
  __stcs(reinterpret_cast<unsigned short*>(p), __bfloat16_as_ushort(__float2bfloat16_rn(v)));
}

// ---------------------------------------------------------------------------------------------
// reductions
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// fixed-order CTA sum of per-thread doubles; result valid in thread 0
__device__ __forceinline__ double block_sum(double v, double* smem /*[kWarps]*/) {
  v = warp_sum(v);
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  __syncthreads();
  if (lane == 0) smem[w] = v;
  __syncthreads();
  double s = 0.0;
  if (threadIdx.x == 0) {
#pragma unroll
    for (int i = 0; i < kWarps; ++i) s += smem[i];
  }
  return s;
}

struct Scratch {
  double* partials;        // [B * tiles_per_pair]; all zero between launches
  unsigned* pair_ticket;   // [B]; all zero between launches
  unsigned* batch_ticket;  // [1]
  unsigned* tile_ctr;      // [2] tile counter / finished-CTA counter of the dynamic tile schedule (nullptr: static); zero between launches
};

struct FwdParams {
  const float* ff;
  const float* bf;
  const float* mask_in;
  const void* prev;
  const void* cur;
  size_t ff_plane, ff_batch, bf_plane, bf_batch;   // element strides between the two flow components / between pairs (rows are dense)
  const int* prev_index;   // clip mode: frame of `prev` / `cur` each pair reads (nullptr: its own)
  const int* cur_index;
  const int* bf_index;     // flow field each pair reads as `bf` / `ff` (nullptr: its own)
  const int* ff_index;
  int pair_group;          // > 1: tiles of this many consecutive pairs are interleaved (window evaluations)
  int cw_packed;           // host side only: launch the 8-consumer-warp variant (the tensor maps' boxes are sized for it)
  int row_begin, row_end;  // rows of every pair this launch covers ([0, H) unless the frame is split into bands over several GPUs)
  void* warp_out;
  float* mask_out;
  void* blend_out;
  double* pair_sums;
  double* total_sums;
  float* pair_vals;
  float* total_val;
  unsigned long long* near_threshold;
  Scratch scratch;
  Geo geo;
  int B, C;
  int tiles_x, tiles_per_pair;
  int flags, loss, finalize;
  double inv_count;  // 1/(C*H*W)
};

__device__ __forceinline__ float finalise_value(double mean, int finalize) {
  return (float)(finalize == TCLB200_FIN_RMSE ? sqrt(mean) : mean);
}

// CTA partial -> pair sum -> batch sum inside the launch.  Every CTA stores its partial and takes a ticket;
// the last CTA of a pair folds that pair's partials in index order, the last pair folds the batch in index
// order: results do not depend on CTA scheduling (deterministic).  Consumed slots are re-zeroed, so the
// scratch is all-zero again when the launch retires, whatever (B,H,W) the next call uses.
__device__ __forceinline__ void reduce_and_finalise(float err, const FwdParams& p, int pair, int tile) {
  __shared__ double red[kWarps];
  __shared__ int s_last;
  const double bsum = block_sum((double)err, red);
  const unsigned tpp = p.tiles_per_pair;
  if (threadIdx.x == 0) {
    __stcg(&p.scratch.partials[(size_t)pair * tpp + tile], bsum);
    __threadfence();
    const unsigned tk = atomicAdd(&p.scratch.pair_ticket[pair], 1u);
    s_last = (tk == tpp - 1);
  }
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  double s = 0.0;
  double* pp = p.scratch.partials + (size_t)pair * tpp;
  for (unsigned i = threadIdx.x; i < tpp; i += kThreads) {
    s += __ldcg(pp + i);
    __stcg(pp + i, 0.0);
  }
  const double S = block_sum(s, red);
  if (threadIdx.x == 0) {
    if (p.pair_sums) p.pair_sums[pair] = S;
    if (p.pair_vals) p.pair_vals[pair] = finalise_value(S * p.inv_count, p.finalize);
    __stcg(pp, S);  // this pair's record for the batch fold
    p.scratch.pair_ticket[pair] = 0;
    __threadfence();
    const unsigned tk = atomicAdd(p.scratch.batch_ticket, 1u);
    s_last = (tk == (unsigned)p.B - 1) ? 2 : 1;
  }
  __syncthreads();
  if (s_last != 2) return;
  __threadfence();
  double a = 0.0, b = 0.0;
  for (int i = threadIdx.x; i < p.B; i += kThreads) {
    double* rec = p.scratch.partials + (size_t)i * tpp;
    const double Si = __ldcg(rec);
    __stcg(rec, 0.0);
    a += Si;
    b += (double)finalise_value(Si * p.inv_count, p.finalize);
  }
  const double A = block_sum(a, red);
  const double Bv = block_sum(b, red);
  if (threadIdx.x == 0) {
    if (p.total_sums) { p.total_sums[0] = A; p.total_sums[1] = Bv; }
    if (p.total_val) *p.total_val = finalise_value(A * p.inv_count / (double)p.B, p.finalize);
    *p.scratch.batch_ticket = 0;
  }
}

__device__ __forceinline__ void count_near(unsigned near, unsigned long long* counter) {
  if (counter == nullptr) return;
  near = __reduce_add_sync(0xffffffffu, near);
  if ((threadIdx.x & 31) == 0 && near) atomicAdd(counter, (unsigned long long)near);
}

// ---------------------------------------------------------------------------------------------
// mbarrier + TMA (cp.async.bulk.tensor) PTX
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, unsigned count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
#ifndef TCL_IDLE_SLEEP_NS
#define TCL_IDLE_SLEEP_NS 40   // back-off of the helper warps' waits (producer, scanners)
#endif
#ifndef TCL_WAIT_HINT_NS
#define TCL_WAIT_HINT_NS 0   // > 0: let the hardware park a waiting warp for up to this many ns per poll
#endif
__device__ __forceinline__ void mbar_wait(uint64_t* bar, unsigned parity) {
#if TCL_WAIT_HINT_NS > 0
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n"
      "@p bra DONE_%=;\n"
      "bra WAIT_%=;\n"
      "DONE_%=:\n"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(parity), "r"((unsigned)TCL_WAIT_HINT_NS)
      : "memory");
#else
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONE_%=;\n"
      "bra WAIT_%=;\n"
      "DONE_%=:\n"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
#endif
}
// same, for a warp that has nothing else to do while it waits: sleeps between polls so that its polling does not
// take issue slots from the warps that share its scheduler
__device__ __forceinline__ void mbar_wait_idle(uint64_t* bar, unsigned parity) {
  for (;;) {
    unsigned done;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(done)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    if (done) return;
    __nanosleep(TCL_IDLE_SLEEP_NS);
  }
}
// TMA prefetch of a 4-D tile into L2 (no shared-memory destination, nothing to wait for)
__device__ __forceinline__ void tma_prefetch_l2_4d(const void* tmap, int c0, int c1, int c2, int c3) {
  asm volatile("cp.async.bulk.prefetch.tensor.4d.L2.global.tile [%0, {%1, %2, %3, %4}];"
               ::"l"(tmap), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
               : "memory");
}
// 4-D tiled TMA load global -> shared, completion on an mbarrier; out-of-range elements are zero-filled
__device__ __forceinline__ void tma_load_4d(void* dst, const void* tmap, uint64_t* bar, int c0, int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(smem_u32(dst)), "l"(tmap), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void prefetch_tmap(const void* tmap) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(tmap) : "memory");
}

}  // namespace tcl
