// Hand-written sm_100a kernels + C ABI for the flow-based temporal-consistency path
// (backward warp, forward-backward occlusion / motion-boundary mask, masked temporal error).
//
// Boundary: include/tcl_b200.h.  Reference semantics: utils/flowtools.py:12-58,
// methods/learning-based/fs_lib.py:5-39, utils/sintel_eval.py:104-110, utils/metrics/eval.py:137-138,
// methods/GAN-based/StarGANv2AdvCon/core/solver.py:427-446 of the upstream repository.
//
// Data layout in HBM: planar NCHW, fp32 flows/masks, fp32 or bf16 frames.
//
// fused_forward_ws_kernel (the hot kernel, details at its definition): persistent, warp-specialised, one CTA per SM.
//   producer warp    TMA pipeline: flow tiles of `bf` (+1 px halo, zero-filled outside the image = the zero padding of
//                    flowtools.gradient) NB tiles ahead; source boxes of `ff` (2 planes) and `prev` (3 planes) NS tiles
//                    ahead, placed where the flow points (fixed 80 x BH size, zero-filled outside the image =
//                    grid_sample's padding_mode='zeros'); L2 prefetch of `cur`; one fp64 partial sum per tile.
//   16 consumer warps one pass per pixel, 4 pixels per lane: motion-boundary test, sampling position (the reference's
//                    exact rounding sequence), 4*(2+3) taps from shared memory (16 x 2 lane footprint, pitch 80:
//                    conflict-free), occlusion test, masked error against `cur`.  They also fold the extent of x+u, y+v
//                    of the flow tile two tiles ahead, from which the producer places that tile's boxes.
//   mixed tiles      (a motion boundary runs through the tile): pixels whose taps leave the boxes gather from global
//                    memory inside the same loop; non-finite / absurd flow: whole tile through the exact guarded path.
//   tile schedule    static round robin for short launches, a global atomic counter for long ones (keeps the CTAs
//                    within a few tiles of each other so that the overlapping box halos hit in L2).
//   reduction        lane -> warp butterfly -> fp64 per tile (plain store) -> fold_partials_kernel (programmatic
//                    dependent launch) sums tiles per pair, pairs per batch in index order: deterministic.
// fused_forward_generic_kernel covers shapes TMA cannot describe (W % 4 != 0, unaligned views, C != 3).
// warp_backward_kernel: autograd of warp / fused backward of the training loss.  gradient_kernel.  hwc_split_kernel
// (dataset ingest) and upsample_flow_kernel (RAFT's convex upsampling) are the steps either side of the path.
// HBM-bound fp32 streaming + gather: no tensor cores, nothing here is a contraction.
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <limits.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <type_traits>

#include "../../include/tcl_b200.h"
#include "tcl_common.cuh"
#include "tcl_math.cuh"

// tile geometry of the TMA kernel (overridable at build time for tuning sweeps, see tools/sweep_build.py)
#ifndef TCL_TH
#define TCL_TH 32     // tile height (the width is 64)
#endif
#ifndef TCL_BH
#define TCL_BH 42     // source-box height with 16 consumer warps (32 rows + 1 + 9 rows of slack for the flow's local spread) ...
#endif
#ifndef TCL_BH8
#define TCL_BH8 44    // ... and with 8 (their control block is smaller): as tall as 227 KB of shared memory allow -- measured on the
#endif                // Sintel shape, sustained: 40 / 42 / 44 rows = 115.7 / 118.2 / 120.2 Gpix/s (fewer tiles straddle a motion boundary)
#ifndef TCL_BH16
#define TCL_BH16 TCL_BH   // ... with bf16 frames (their boxes are smaller: room for more rows)
#endif
#ifndef TCL_BW
#define TCL_BW 80     // source-box width for fp32 frames: 16 (mod 32), see WsCfg
#endif
#ifndef TCL_BW16
#define TCL_BW16 80   // ... for bf16 frames (TMA: rows are multiples of 16 bytes)
#endif
#ifndef TCL_NS
#define TCL_NS 2      // source-box stages in flight
#endif
#ifndef TCL_NB
#define TCL_NB (TCL_NS + 2)   // flow-tile stages in flight
#endif
// Configurations without a computed mask (dataset mask: the training loss; no mask: warp on its own, blend) stage no `ff`
// planes: their source stage is 3/5 of the size and a THIRD one fits, which takes the wait for the source boxes off their
// (shorter) per-tile critical path.
#ifndef TCL_NS_NOFF
#define TCL_NS_NOFF 3
#endif
#ifndef TCL_BH_NOFF
#define TCL_BH_NOFF 40
#endif
#ifndef TCL_SCANNERS
#define TCL_SCANNERS 2   // scanner warps (one warp needs about a tile period per tile and would pace the pipeline)
#endif
#ifndef TCL_PACKED
#define TCL_PACKED 1  // interior staged tiles of the reducing hot configurations use packed fp32 arithmetic (lean_tile_packed)
#endif
#ifndef TCL_NS_MASK
#define TCL_NS_MASK 3   // source-box stages of fbcCheckTorch on its own (two `ff` planes per stage)
#endif
#ifndef TCL_PACKED_MASK
#define TCL_PACKED_MASK 1    // ... and for fbcCheckTorch on its own (mask_out only)
#endif
#ifndef TCL_PACKED_GIVEN
#define TCL_PACKED_GIVEN 1   // ... also with a dataset mask (the training loss)
#endif
#ifndef TCL_DIAG
#define TCL_DIAG 0    // tuning aids (tools/sweep_build.py): 1 = no source-box traffic, 3 = boxes at the tile's own position (no scan)
#endif

namespace tcl {

// ---------------------------------------------------------------------------------------------
// per-pixel pieces shared by both forward kernels
// ---------------------------------------------------------------------------------------------
struct PixTaps {   // four bilinear taps of one target pixel
  int x0, y0;
  float nw, ne, sw, se;
};

__device__ __forceinline__ PixTaps pix_taps(float u, float v, int x, int y, const Geo& g) {
  const float ix = source_coord(x, u, g.Wf, g.dxf, g.inv_dx, kV);
  const float iy = source_coord(y, v, g.Hf, g.dyf, g.inv_dy, kV);
  PixTaps t;
  t.x0 = __float2int_rd(ix);  // = static_cast<int>(::floor(ix)): saturating, NaN -> 0
  t.y0 = __float2int_rd(iy);
  const float fx1 = __fsub_rn((float)(int)((unsigned)t.x0 + 1u), ix), fx0 = __fsub_rn(ix, (float)t.x0);
  const float fy1 = __fsub_rn((float)(int)((unsigned)t.y0 + 1u), iy), fy0 = __fsub_rn(iy, (float)t.y0);
  t.nw = __fmul_rn(fx1, fy1); t.ne = __fmul_rn(fx0, fy1);
  t.sw = __fmul_rn(fx1, fy0); t.se = __fmul_rn(fx0, fy0);
  return t;
}

__device__ __forceinline__ Taps full_taps(const PixTaps& s, const Geo& g) {
  Taps t;
  const int x1 = (int)((unsigned)s.x0 + 1u), y1 = (int)((unsigned)s.y0 + 1u);
  const bool xin0 = (unsigned)s.x0 < (unsigned)g.W, xin1 = (unsigned)x1 < (unsigned)g.W;
  const bool yin0 = (unsigned)s.y0 < (unsigned)g.H, yin1 = (unsigned)y1 < (unsigned)g.H;
  t.p00 = xin0 && yin0; t.p10 = xin1 && yin0; t.p01 = xin0 && yin1; t.p11 = xin1 && yin1;
  t.o00 = (int)((unsigned)s.y0 * (unsigned)g.W + (unsigned)s.x0);
  t.nw = s.nw; t.ne = s.ne; t.sw = s.sw; t.se = s.se;
  return t;
}

// source planes in global memory: exact predicated gather (grid_sampler_2d skips out-of-image taps)
template <typename T>
struct GlobalSrc {
  const T* base;   // plane 0 of this pair
  size_t plane;
  Geo g;
  __device__ __forceinline__ float sample(int c, const PixTaps& s) const {
    return sample_global(base + (size_t)c * plane, full_taps(s, g), g.W, kV);
  }
};

// source box in shared memory, origin (ox,oy), zero-filled outside the image: all four taps are plain reads.
// fma(0, w, acc) == acc for the finite weights of an in-box pixel, so this equals the predicated form.
template <typename T, int PITCH, int CH_STRIDE>
struct SmemSrc {
  const T* base;
  int ox, oy;
  __device__ __forceinline__ float sample(int c, const PixTaps& s) const {
    const T* q = base + c * CH_STRIDE + (s.y0 - oy) * PITCH + (s.x0 - ox);
    float acc = __fmul_rn(to_f32(q[0]), s.nw);
    acc = __fmaf_rn(to_f32(q[1]), s.ne, acc);
    acc = __fmaf_rn(to_f32(q[PITCH]), s.sw, acc);
    acc = __fmaf_rn(to_f32(q[PITCH + 1]), s.se, acc);
    return acc;
  }
};

template <typename FrameT>
struct PairPtrs {
  const FrameT* cur;
  FrameT* wout;
  FrameT* bout;
};

// everything that happens to one pixel once its taps and motion-boundary verdict are known.
// LEAN fixes the hot configuration at compile time (both mask tests, L2 error, no optional outputs, no
// near-threshold count) so the per-pixel code carries no runtime feature checks.
// `cv` = this pixel's prefetched `cur` values (CT of them) or nullptr to load them here.
template <typename FrameT, int MASK, bool REDUCE, int CT, int LEAN, typename FlowSrc, typename FrameSrc>
__device__ __forceinline__ void finish_pixel(const FwdParams& p, const PixTaps& s, float u, float v, float nb, float keep,
                                             size_t o, size_t plane, int pair, const FlowSrc& fsrc, const FrameSrc& psrc,
                                             const PairPtrs<FrameT>& io, const float* cv, float& err, unsigned& near) {
  if (MASK == MASK_COMPUTED && (LEAN || (p.flags & TCLB200_OCC))) {
    const float wu = fsrc.sample(0, s), wv = fsrc.sample(1, s);
    float margin;
    if (occluded(wu, wv, u, v, nb, kV, &margin)) keep = 0.0f;
    if (!LEAN) near += fabsf(margin) < kNearBand;
  }
  if ((!LEAN || CT == 0) && p.mask_out) __stcs(p.mask_out + (size_t)pair * plane + o, keep);
  if (p.prev == nullptr) return;
  const bool validity = (!LEAN || MASK == MASK_NONE) && (p.flags & TCLB200_VALIDITY);
  float valid = 1.0f;
  if (validity) valid = binarise_validity(ones_sample(full_taps(s, p.geo), kV));
  const int C = CT > 0 ? CT : p.C;
#pragma unroll
  for (int c = 0; c < C; ++c) {
    float w = psrc.sample(c, s);
    if (validity) w = __fmul_rn(w, valid);
    if ((!LEAN || MASK == MASK_NONE) && io.wout) st_stream(io.wout + (size_t)c * plane + o, w);   // (LEAN + MASK_NONE = warp only)
    if ((LEAN && MASK != MASK_NONE) || (!LEAN && io.cur)) {
      const float x = cv ? cv[c] : ld_stream(io.cur + (size_t)c * plane + o);
      if (REDUCE) {
        if (LEAN == 1 || (!LEAN && p.loss == TCLB200_L2)) {   // LEAN: 1 = L2, 2 = L1 fixed at compile time
          const float md = __fmul_rn(keep, __fsub_rn(x, w));     // mask*(cur - warp)   sintel_eval.py:110
          err = __fmaf_rn(md, md, err);
        } else {
          err += __fmul_rn(keep, fabsf(__fsub_rn(w, x)));        // mask*|warp - cur|   MoGAN cycle_gan_model.py:281
        }
      }
      if (!LEAN && io.bout)                                      // m*warp + (1-m)*img   obst_eval.py:500
        st_stream(io.bout + (size_t)c * plane + o, __fadd_rn(__fmul_rn(keep, w), __fmul_rn(__fsub_rn(1.0f, keep), x)));
    }
  }
}

// frame of `prev` / `cur` pair b reads: its own, or -- clip mode -- the one an index array names, so that a video frame
// stored once can be the `cur` of pair t and the `prev` of pair t+1 (the second read then comes out of L2)
__device__ __forceinline__ int prev_frame(const FwdParams& p, int pair) { return p.prev_index ? __ldg(p.prev_index + pair) : pair; }
__device__ __forceinline__ int cur_frame(const FwdParams& p, int pair) { return p.cur_index ? __ldg(p.cur_index + pair) : pair; }
// ... and the same for the flow fields: a window evaluation uses each field twice, as the `bf` of (s -> t) and the `ff` of (t -> s)
__device__ __forceinline__ int bf_field(const FwdParams& p, int pair) { return p.bf_index ? __ldg(p.bf_index + pair) : pair; }
__device__ __forceinline__ int ff_field(const FwdParams& p, int pair) { return p.ff_index ? __ldg(p.ff_index + pair) : pair; }

template <typename FrameT>
__device__ __forceinline__ PairPtrs<FrameT> pair_ptrs(const FwdParams& p, int pair, int cf, int C, size_t plane) {
  PairPtrs<FrameT> io;
  const size_t off = (size_t)pair * C * plane;
  io.cur = p.cur ? reinterpret_cast<const FrameT*>(p.cur) + (size_t)cf * C * plane : nullptr;
  io.wout = p.warp_out ? reinterpret_cast<FrameT*>(p.warp_out) + off : nullptr;
  io.bout = p.blend_out ? reinterpret_cast<FrameT*>(p.blend_out) + off : nullptr;
  return io;
}

// ---------------------------------------------------------------------------------------------
// generic forward kernel: one pixel per lane, everything straight from global memory
// ---------------------------------------------------------------------------------------------
template <typename FrameT, int MASK, bool REDUCE, int CT>
__global__ void __launch_bounds__(kThreads) fused_forward_generic_kernel(const FwdParams p) {
  const Geo& g = p.geo;
  const int W = g.W, H = g.H;
  const size_t plane = (size_t)H * W;
  const int lane = threadIdx.x & 31, wrp = threadIdx.x >> 5;
  const int pair = blockIdx.x / p.tiles_per_pair;
  const int tile = blockIdx.x - pair * p.tiles_per_pair;
  const int ty = tile / p.tiles_x, tx = tile - ty * p.tiles_x;
  const int x = tx * 32 + lane, y = p.row_begin + ty * kWarps + wrp;   // (band mode: rows [row_begin, row_end) only)
  const int C = CT > 0 ? CT : p.C;
  float err = 0.0f;
  unsigned near = 0;
  if (x < W && y < p.row_end) {
    const size_t o = (size_t)y * W + x;
    const float* bu = p.bf + (size_t)bf_field(p, pair) * p.bf_batch;
    const float* bv = bu + p.bf_plane;
    const float u = __ldg(bu + o), v = __ldg(bv + o);
    float nb = sqnorm2(u, v, kV);
    float keep = 1.0f;
    if (MASK == MASK_GIVEN) keep = __ldcs(p.mask_in + (size_t)pair * plane + o);
    if (MASK == MASK_COMPUTED && (p.flags & TCLB200_MOB)) {
      const float ul = x > 0 ? __ldg(bu + o - 1) : 0.0f, ur = x + 1 < W ? __ldg(bu + o + 1) : 0.0f;
      const float uu = y > 0 ? __ldg(bu + o - W) : 0.0f, ud = y + 1 < H ? __ldg(bu + o + W) : 0.0f;
      const float vl = x > 0 ? __ldg(bv + o - 1) : 0.0f, vr = x + 1 < W ? __ldg(bv + o + 1) : 0.0f;
      const float vu = y > 0 ? __ldg(bv + o - W) : 0.0f, vd = y + 1 < H ? __ldg(bv + o + W) : 0.0f;
      float margin;
      if (motion_boundary(u, v, ul, ur, uu, ud, vl, vr, vu, vd, kV, &nb, &margin)) keep = 0.0f;
      near += fabsf(margin) < kNearBand;
    }
    const PixTaps s = pix_taps(u, v, x, y, g);
    GlobalSrc<float> fsrc{p.ff ? p.ff + (size_t)ff_field(p, pair) * p.ff_batch : nullptr, p.ff_plane, g};
    GlobalSrc<FrameT> psrc{p.prev ? reinterpret_cast<const FrameT*>(p.prev) + (size_t)prev_frame(p, pair) * C * plane : nullptr, plane, g};
    finish_pixel<FrameT, MASK, REDUCE, CT, false>(p, s, u, v, nb, keep, o, plane, pair, fsrc, psrc,
                                                  pair_ptrs<FrameT>(p, pair, cur_frame(p, pair), C, plane), nullptr, err, near);
  }
  count_near(near, p.near_threshold);
  if (REDUCE) reduce_and_finalise(err, p, pair, tile);
}

// ---------------------------------------------------------------------------------------------
// direct forward kernel: short launches of the training loss (dataset mask, C == 3, reduction only)
// ---------------------------------------------------------------------------------------------
// The persistent TMA pipeline below needs ~7 us to fill and drain and works a tile at a time; a training batch
// (16 x 256 x 256, solver.py:427-446) is only 3.5 tile rounds long.  This kernel puts the launch in flight at once instead:
// one CTA of 256 threads per 512 consecutive pixels of a pair (two pixels per thread, one step), 12 KB of shared memory,
// four or more CTAs resident per SM.  Thread 0 requests the chunk's flow, mask and `cur` values with six bulk copies
// (cp.async.bulk: no registers tied up while they fly) and prefetches the chunk's own stretch of `prev` into L2; the taps
// of `prev` are exact predicated gathers from global memory (grid_sample's zero padding), consecutive lanes on
// consecutive pixels.  One fp64 partial per chunk, then the fold kernel behind it (programmatic dependent launch) exactly
// as for the TMA kernel.  Measured (tools/small_launch.py, CUDA-graph replay over L2-rotating buffers): 4 / 16 / 32 pairs of
// 256 x 256: 7.2 / 17.9 / 29.6 us against 10.2 / 21.7 / 34 us on the pipeline; from 64 pairs on the pipeline wins.
// Variants measured and dropped: 128 threads x 8 pixels (19.4 us at 16 pairs), 512 threads x 2 pixels (18.1), 256 x 4 (18.5),
// six resident CTAs at 42 registers (18.0), no L2 prefetch (+0.4 us, +1.9 us at 4 pairs).
constexpr int kDirectThreads = 256, kDirectChunk = 512, kDirectResident = 4;

__device__ __forceinline__ void bulk_load_1d(void* dst, const void* src, unsigned bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

template <typename FrameT, int LOSS>
__global__ void __launch_bounds__(kDirectThreads, kDirectResident) fused_forward_direct_kernel(const FwdParams p) {
  constexpr int CH = kDirectChunk, PPT = CH / kDirectThreads;
  __shared__ __align__(128) float s_f[3][CH];      // u, v, mask of the chunk
  __shared__ __align__(128) FrameT s_c[3][CH];     // cur
  __shared__ __align__(8) uint64_t s_bar[2];       // [0] flow landed, [1] mask and cur landed
  __shared__ double s_red[kDirectThreads / 32];
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");   // let the fold kernel get resident early
  const Geo& g = p.geo;
  const int W = g.W;
  const size_t plane = (size_t)g.H * W;
  const int pair = blockIdx.x / p.tiles_per_pair, chunk = blockIdx.x - pair * p.tiles_per_pair;
  const int i0 = p.row_begin * W + chunk * CH;               // (band mode: rows [row_begin, row_end) only)
  const int n = min(CH, p.row_end * W - i0);                 // a multiple of 4 (8 with bf16 frames): the host checks W
  const FrameT* prev = reinterpret_cast<const FrameT*>(p.prev) + (size_t)prev_frame(p, pair) * 3 * plane;
  if (threadIdx.x == 0) {
    const float* bu = p.bf + (size_t)bf_field(p, pair) * p.bf_batch + i0;
    const FrameT* cur = reinterpret_cast<const FrameT*>(p.cur) + (size_t)cur_frame(p, pair) * 3 * plane + i0;
    const unsigned fb = (unsigned)n * 4u, cb = (unsigned)n * (unsigned)sizeof(FrameT);
    mbar_init(&s_bar[0], 1);
    mbar_init(&s_bar[1], 1);
    fence_barrier_init();
    mbar_expect_tx(&s_bar[0], 2u * fb);
    bulk_load_1d(s_f[0], bu, fb, &s_bar[0]);
    bulk_load_1d(s_f[1], bu + p.bf_plane, fb, &s_bar[0]);
    // this chunk's own stretch of the three `prev` planes into L2: the taps of a chunk land elsewhere (where the flow
    // points), but all chunks together cover the frames, so the whole launch's DRAM reads are requested in its first
    // microsecond and the gathers below mostly hit L2
#pragma unroll
    for (int c = 0; c < 3; ++c)
      asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(prev + (size_t)c * plane + i0), "r"(cb) : "memory");
    mbar_expect_tx(&s_bar[1], fb + 3u * cb);
    bulk_load_1d(s_f[2], p.mask_in + (size_t)pair * plane + i0, fb, &s_bar[1]);
    bulk_load_1d(s_c[0], cur, cb, &s_bar[1]);
    bulk_load_1d(s_c[1], cur + plane, cb, &s_bar[1]);
    bulk_load_1d(s_c[2], cur + 2 * plane, cb, &s_bar[1]);
  }
  int i = threadIdx.x;
  int y = (int)((unsigned)(i0 + i) / (unsigned)W), x = i0 + i - y * W;
  const int step_y = kDirectThreads / W, step_x = kDirectThreads - step_y * W;   // pixel i + 256 is that far from pixel i
  __syncthreads();               // the barriers are initialised
  mbar_wait(&s_bar[0], 0);
  float err = 0.0f;
  // two pixels per step, branch-free (a lane beyond the chunk's end recomputes pixel 0 and drops it): the 24 gathers of
  // a step are independent and in flight together
#pragma unroll 1
  for (int j = 0; j < PPT; j += 2) {
    Taps t[2];
    float keep[2];
    int ii[2];
    bool ok[2];
#pragma unroll
    for (int q = 0; q < 2; ++q) {
      ok[q] = i < n;
      ii[q] = ok[q] ? i : 0;
      t[q] = full_taps(pix_taps(s_f[0][ii[q]], s_f[1][ii[q]], x, y, g), g);
      i += kDirectThreads;
      x += step_x; y += step_y;
      if (x >= W) { x -= W; ++y; }
    }
    float w[2][3];
#pragma unroll
    for (int q = 0; q < 2; ++q)
#pragma unroll
      for (int c = 0; c < 3; ++c) w[q][c] = sample_global(prev + (size_t)c * plane, t[q], W, kV);
    // (a warp-uniform interior fast path -- plain loads off one address per pixel when every tap of every lane is inside the
    // image -- was measured: 18.2 vs 17.4 us at 16 x 256^2, 84 vs 69 us at 128: the vote and the branch cost the overlap of the
    // two pixels' loads)
    if (j == 0) mbar_wait(&s_bar[1], 0);   // (the first gathers are under way before mask and cur are needed)
    keep[0] = s_f[2][ii[0]]; keep[1] = s_f[2][ii[1]];
#pragma unroll
    for (int q = 0; q < 2; ++q) {
      float e = err;
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        const float xc = to_f32(s_c[c][ii[q]]);
        if (LOSS == TCLB200_L2) {
          const float md = __fmul_rn(keep[q], __fsub_rn(xc, w[q][c]));   // mask*(cur - warp)   solver.py:444
          e = __fmaf_rn(md, md, e);
        } else {
          e = __fadd_rn(e, __fmul_rn(keep[q], fabsf(__fsub_rn(w[q][c], xc))));   // mask*|warp - cur|   MoGAN cycle_gan_model.py:281
        }
      }
      err = ok[q] ? e : err;
    }
  }
  double s = warp_sum((double)err);
  if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    s = 0.0;
#pragma unroll
    for (int k = 0; k < kDirectThreads / 32; ++k) s += s_red[k];
    __stcg(&p.scratch.partials[(size_t)pair * p.tiles_per_pair + chunk], s);
  }
}

// ---------------------------------------------------------------------------------------------
// pieces of the TMA-staged, persistent, warp-specialised forward kernel (the hot kernel, described at its definition)
// ---------------------------------------------------------------------------------------------
__device__ unsigned long long g_tile_stats[2];   // debug statistics: tiles taken from global memory entirely / mixed tiles
#ifdef TCL_TRACE
// tuning aid (tools/trace_pipeline.py): per CTA and local tile, globaltimer stamps of the pipeline events
constexpr int kTraceTiles = 64;
__device__ unsigned long long g_trace[160][kTraceTiles][4];   // src requested, src observed ready (before / after the wait), tile done
__device__ __forceinline__ unsigned long long gtime() { unsigned long long t; asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t)); return t; }
#define TCL_STAMP(k, slot) do { if ((k) < kTraceTiles && blockIdx.x < 160) g_trace[blockIdx.x][(k)][(slot)] = gtime(); } while (0)
#else
#define TCL_STAMP(k, slot) do { } while (0)
#endif
// consumer warps per CTA: 8 (eight pixels per lane and tile) for the packed-arithmetic configuration, 16 (four pixels
// per lane) for everything else -- measured per configuration (DESIGN.md); TCL_CWARPS forces one value (tuning builds)
#ifdef TCL_CWARPS
constexpr int kCWarpsPacked = TCL_CWARPS, kCWarpsOther = TCL_CWARPS;
#else
constexpr int kCWarpsPacked = 8, kCWarpsOther = 16;
#endif

// Lane -> pixel mapping of the consumer warps.  A warp owns a 16-column x kRows-row block of the 64 x TH tile (4 column
// blocks x CW/4 row blocks); lane = 16 * h + c works on column c and on rows h, h + 2, h + 4, ... of the block.  One
// warp instruction therefore covers 16 columns x 2 ADJACENT rows, and all shared-memory pitches are 80 words = 16 (mod 32):
// the two rows fall into disjoint halves of the 32 banks, also when the flow shifts some lanes to the next source row, so
// the reads of the flow tile are conflict-free and the taps nearly so (measured: rows four apart -- vertical strips of
// adjacent pixels per lane -- lose more to the shear of real flows, 1.5 wavefronts per tap read, than their register
// reuse saves).  A lane's rows interleave with its partner's, so the column's flow values are still shared between a
// lane's pixels: 2 * P + 1 + 2 * P shared-memory reads per flow component and P pixels instead of 5 * P.
template <typename FrameT, int CT, int TW_, int TH_, int BW_, int BH_, int NB_, int NS_, int CW_, bool FF_ = true>
struct WsCfg {
  static constexpr int TW = TW_, TH = TH_, BW = BW_, BH = BH_, NB = NB_, NS = NS_;
  static constexpr int CW = CW_;                 // consumer warps; then the producer warp (TMA requests, box placement, per-tile
  static constexpr int kProducerWarp = CW;       // fold of the partial sums) and the scanner warp (extent of the sampling
  static constexpr int kScannerWarp = CW + 1;    // positions of every flow tile; kScanners of them take the tiles in turn)
  static constexpr int kScanners = TCL_SCANNERS;
  static constexpr int kThreads = 32 * (CW + 1 + kScanners);
  static constexpr int kHaloL = 4;               // TMA needs the box's innermost start on a 16-byte boundary
  static constexpr int kBfW = TW + 16, kBfH = TH + 2;   // 4 + 64 + 12 columns (the right halo needs 1; 80 = 16 mod 32)
  static constexpr int kXAlign = 16 / (int)sizeof(FrameT);   // source-box origin is rounded down to this many pixels
  static constexpr int kRowBlocks = CW / 4;
  static constexpr int kRows = TH / kRowBlocks;  // rows of a warp's block
  static constexpr int kPPL = kRows / 2;         // pixels per lane per tile
  static constexpr int kC = CT > 0 ? CT : 1;
  static constexpr unsigned kBfLoad = 2u * kBfH * kBfW * 4u;
  static constexpr unsigned kFfLoad = 2u * BH * BW * 4u;
  static constexpr unsigned kPrevLoad = (unsigned)(CT > 0 ? CT : 0) * BH * BW * (unsigned)sizeof(FrameT);
  static constexpr size_t kBfStage = align_up(kBfLoad, 128);
  static constexpr size_t kFfStage = FF_ ? align_up(kFfLoad, 128) : 0;   // (configurations without a computed mask stage no `ff` planes)
  static constexpr size_t kSrcStage = kFfStage + align_up(kPrevLoad, 128);
  static constexpr size_t kBfOff = 0;
  static constexpr size_t kSrcOff = kBfOff + NB * kBfStage;
  static constexpr size_t kCtlOff = kSrcOff + NS * kSrcStage;
  static constexpr size_t kCtlBytes = 1024 + (size_t)NS * CW * 32 * 4;
  static constexpr size_t kSmemBytes = kCtlOff + kCtlBytes + 128;  // + slack for manual 128-byte alignment
  static_assert(TW == 64 && CW % 4 == 0 && TH % kRowBlocks == 0 && kRows % 2 == 0, "lane mapping: 16-column blocks, row pairs");
  static_assert(kBfW % 32 == 16, "flow-tile pitch must be 16 (mod 32) words: adjacent rows fall into disjoint bank halves");
  static_assert((BW * (int)sizeof(FrameT)) % 16 == 0 && BW % 4 == 0, "TMA: box rows are multiples of 16 bytes");
#if TCL_DIAG != 3
  static_assert(NB >= NS + 1, "the flow tile of a tile is scanned NS tiles ahead of its use");
  static_assert(kSmemBytes <= 232448, "a CTA has at most 227 KB of shared memory");
#endif
};
// row of pixel k of a lane, relative to the lane's first row
__host__ __device__ constexpr int pix_dy(int k) { return 2 * k; }
template <typename Cfg>
__device__ __forceinline__ void lane_origin(int warp, int lane, int& lx0, int& ly0) {
  lx0 = 16 * (warp & 3) + (lane & 15);
  ly0 = Cfg::kRows * (warp >> 2) + (lane >> 4);
}

struct TileId { int pair, tile, x0, y0, pf, cf, bfi, ffi; };   // pf / cf: frame of `prev` / `cur` this pair reads; bfi / ffi: its flow fields

template <int NB, int NS, int CW>
struct WsCtl {              // control block in shared memory
  uint64_t bf_full[NB], scanned[NB], src_full[NS], done[NS];
  TileId tinfo[NB];         // written by the producer with the flow-tile request
  int meta[NS][4];          // per source stage: ox, oy, staged?
  int box[NB][4];           // per flow stage: extent of x+u, y+v over the tile (ordered-int encoding): xmin, ymin, xmax, ymax
  float red[NS][CW * 32];   // per source stage: every consumer lane's error sum of the tile
};

// order-preserving float <-> int (total order of IEEE bit patterns; NaNs land beyond +-Inf): lets redux.sync work on
// float extents
__device__ __forceinline__ int f2ord(float f) { const int i = __float_as_int(f); return i ^ ((i >> 31) & 0x7fffffff); }
__device__ __forceinline__ float ord2f(int i) { return __int_as_float(i ^ ((i >> 31) & 0x7fffffff)); }
__device__ __forceinline__ float fmin_nan(float a, float b) { float r; asm("min.NaN.f32 %0, %1, %2;" : "=f"(r) : "f"(a), "f"(b)); return r; }
__device__ __forceinline__ float fmax_nan(float a, float b) { float r; asm("max.NaN.f32 %0, %1, %2;" : "=f"(r) : "f"(a), "f"(b)); return r; }

// scanner warp: extent of x+u, y+v (the sums the sampling positions start from) over the pixels of flow tile `t` that lie
// inside the image -> box[4].  Non-finite flow propagates (min/max.NaN; a NaN wins the min or the max of the ordered
// encoding, depending on its sign) and is rejected by the placement.  One LDS.128 per component and four pixels.
template <typename Cfg>
__device__ __forceinline__ void scan_flow_tile(const float* s_bu, const TileId& t, const Geo& g, int row_end, int* box, int lane) {
  const float* s_bv = s_bu + Cfg::kBfH * Cfg::kBfW;
  const int c4 = 4 * (lane & 15), rh = lane >> 4;
  // W % 4 == 0: a lane's four columns are all inside the image or all outside
  const bool colok = t.x0 + c4 < g.W;
  const float xf = (float)(t.x0 + c4);
  const float inf = __int_as_float(0x7f800000);
  float xmin = inf, ymin = inf, xmax = -inf, ymax = -inf;
  const int rows = min(Cfg::TH, row_end - t.y0);
  if (colok) {
#pragma unroll 4
    for (int r = rh; r < rows; r += 2) {
      const float4 u4 = *reinterpret_cast<const float4*>(s_bu + (r + 1) * Cfg::kBfW + Cfg::kHaloL + c4);
      const float4 v4 = *reinterpret_cast<const float4*>(s_bv + (r + 1) * Cfg::kBfW + Cfg::kHaloL + c4);
      const float yf = (float)(t.y0 + r);
      const float a0 = __fadd_rn(xf, u4.x), a1 = __fadd_rn(xf + 1.0f, u4.y), a2 = __fadd_rn(xf + 2.0f, u4.z), a3 = __fadd_rn(xf + 3.0f, u4.w);
      xmin = fmin_nan(xmin, fmin_nan(fmin_nan(a0, a1), fmin_nan(a2, a3)));
      xmax = fmax_nan(xmax, fmax_nan(fmax_nan(a0, a1), fmax_nan(a2, a3)));
      ymin = fmin_nan(ymin, __fadd_rn(yf, fmin_nan(fmin_nan(v4.x, v4.y), fmin_nan(v4.z, v4.w))));
      ymax = fmax_nan(ymax, __fadd_rn(yf, fmax_nan(fmax_nan(v4.x, v4.y), fmax_nan(v4.z, v4.w))));
    }
  }
  const int ixmin = __reduce_min_sync(0xffffffffu, f2ord(xmin)), iymin = __reduce_min_sync(0xffffffffu, f2ord(ymin));
  const int ixmax = __reduce_max_sync(0xffffffffu, f2ord(xmax)), iymax = __reduce_max_sync(0xffffffffu, f2ord(ymax));
  if (lane == 0) { box[0] = ixmin; box[1] = iymin; box[2] = ixmax; box[3] = iymax; }
}

__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// the same on precomputed shared-memory addresses (the consumers' per-tile waits: no address arithmetic in the loop)
__device__ __forceinline__ void mbar_arrive_s(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
#ifndef TCL_CONS_HINT_NS
#define TCL_CONS_HINT_NS 0   // > 0: the consumers' waits let the hardware park the warp for up to this many ns per poll
#endif
__device__ __forceinline__ void mbar_wait_s(uint32_t bar, unsigned parity) {
#if TCL_CONS_HINT_NS > 0
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n"
      "@p bra DONE_%=;\n"
      "bra WAIT_%=;\n"
      "DONE_%=:\n"
      "}\n" ::"r"(bar),
      "r"(parity), "r"((unsigned)TCL_CONS_HINT_NS)
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
      "}\n" ::"r"(bar),
      "r"(parity)
      : "memory");
#endif
}

// Fold kernel of the warp-specialised path: the hot kernel only stores one fp64 partial per tile (no fences, no
// atomics on its critical path); this kernel, launched behind it with programmatic dependent launch so that its
// launch latency overlaps the hot kernel, sums each pair's partials in index order and the pairs in index order
// (deterministic), finalises (mean / RMSE) and leaves the scratch zeroed as the protocol of tcl_common.cuh wants.
__global__ void __launch_bounds__(kThreads) fold_partials_kernel(const FwdParams p) {
  __shared__ double red[kWarps];
  __shared__ int s_last;
  asm volatile("griddepcontrol.wait;" ::: "memory");   // all of the hot kernel's stores are visible after this
  const int pair = blockIdx.x;
  const unsigned tpp = p.tiles_per_pair;
  double* pp = p.scratch.partials + (size_t)pair * tpp;
  double s = 0.0;
  for (unsigned i = threadIdx.x; i < tpp; i += kThreads) {
    s += __ldcg(pp + i);
    __stcg(pp + i, 0.0);
  }
  const double S = block_sum(s, red);
  if (threadIdx.x == 0) {
    if (p.pair_sums) p.pair_sums[pair] = S;
    if (p.pair_vals) p.pair_vals[pair] = finalise_value(S * p.inv_count, p.finalize);
    __stcg(pp, S);  // this pair's record for the batch fold
    __threadfence();
    s_last = atomicAdd(p.scratch.batch_ticket, 1u) == (unsigned)p.B - 1;
  }
  __syncthreads();
  if (!s_last) return;
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

// The same for short launches (<= kFoldSmallPairs pairs, a few thousand partials): ONE CTA, 256 threads per pair and four
// pairs at a time, no tickets and no second trip through L2 -- about half the latency of the two-level fold above, which
// matters when the whole launch is 10-20 us.  Same summation order as fold_partials_kernel, so a pair's value does not
// depend on which of the two folded it.
constexpr int kFoldSmallPairs = 64, kFoldSmallPartials = 16384, kFoldSmallGroups = 1024 / kThreads;
__global__ void __launch_bounds__(1024) fold_partials_small_kernel(const FwdParams p) {
  __shared__ double s_S[kFoldSmallPairs];
  __shared__ double s_red[kFoldSmallGroups][kWarps];
  asm volatile("griddepcontrol.wait;" ::: "memory");
  const int grp = threadIdx.x / kThreads, t = threadIdx.x - grp * kThreads, lane = t & 31, w = t >> 5;
  const unsigned tpp = p.tiles_per_pair;
  for (int base = 0; base < p.B; base += kFoldSmallGroups) {
    const int pair = base + grp;
    double s = 0.0;
    if (pair < p.B) {
      double* pp = p.scratch.partials + (size_t)pair * tpp;
      for (unsigned i = t; i < tpp; i += kThreads) {
        s += __ldcg(pp + i);
        __stcg(pp + i, 0.0);
      }
    }
    s = warp_sum(s);
    if (lane == 0) s_red[grp][w] = s;
    __syncthreads();
    if (t == 0 && pair < p.B) {
      double S = 0.0;
#pragma unroll
      for (int i = 0; i < kWarps; ++i) S += s_red[grp][i];
      if (p.pair_sums) p.pair_sums[pair] = S;
      if (p.pair_vals) p.pair_vals[pair] = finalise_value(S * p.inv_count, p.finalize);
      s_S[pair] = S;
    }
    __syncthreads();
  }
  if (grp != 0) return;
  double a = 0.0, b = 0.0;
  for (int i = t; i < p.B; i += kThreads) {
    a += s_S[i];
    b += (double)finalise_value(s_S[i] * p.inv_count, p.finalize);
  }
  a = warp_sum(a); b = warp_sum(b);
  if (lane == 0) { s_red[0][w] = a; s_red[1][w] = b; }
  asm volatile("bar.sync 1, 256;" ::: "memory");   // (the first group's 256 threads only)
  if (t == 0) {
    double A = 0.0, Bv = 0.0;
#pragma unroll
    for (int i = 0; i < kWarps; ++i) { A += s_red[0][i]; Bv += s_red[1][i]; }
    if (p.total_sums) { p.total_sums[0] = A; p.total_sums[1] = Bv; }
    if (p.total_val) *p.total_val = finalise_value(A * p.inv_count / (double)p.B, p.finalize);
  }
}

// Global tile number -> pair and tile.  pair_group G > 1 interleaves the tiles of G consecutive pairs (tile 0 of pairs
// g*G .. g*G+G-1, then their tiles 1, ...): the evaluations of one target frame's window read the same `cur` tile, the same
// flow tiles and neighbouring boxes within microseconds of each other, so every re-read is an L2 hit.
__device__ __forceinline__ TileId tile_id(const FwdParams& p, int tg, int TW, int TH) {
  TileId t;
  if (p.pair_group > 1) {
    const int span = p.tiles_per_pair * p.pair_group;
    const int grp = tg / span, r = tg - grp * span;
    const int gsize = min(p.pair_group, p.B - grp * p.pair_group);
    t.tile = r / gsize;
    t.pair = grp * p.pair_group + (r - t.tile * gsize);
  } else {
    t.pair = tg / p.tiles_per_pair;
    t.tile = tg - t.pair * p.tiles_per_pair;
  }
  const int ty = t.tile / p.tiles_x, tx = t.tile - ty * p.tiles_x;
  t.x0 = tx * TW; t.y0 = p.row_begin + ty * TH;
  t.pf = prev_frame(p, t.pair); t.cf = cur_frame(p, t.pair);
  t.bfi = bf_field(p, t.pair); t.ffi = ff_field(p, t.pair);
  return t;
}
template <typename Cfg>
__device__ __forceinline__ bool tile_edge(const TileId& t, const Geo& g, int row_end) { return (t.x0 + Cfg::TW > g.W) || (t.y0 + Cfg::TH > row_end); }

// ---- consumer: exact per-pixel path (all features; staged boxes, global gathers, or both in a mixed tile) -------
template <typename FrameT, int MASK, bool REDUCE, int CT, int LEAN, typename Cfg, bool EDGE>
__device__ __forceinline__ float full_tile(const FwdParams& p, const float* s_bu, const float* s_ff, const FrameT* s_prev,
                                           const int* meta, const TileId& t, int lx0, int ly0,
                                           const float (&cur)[Cfg::kPPL][Cfg::kC], const float (&mk)[Cfg::kPPL], bool have_cur,
                                           unsigned& near) {
  const Geo& g = p.geo;
  const int W = g.W, H = g.H;
  const size_t plane = (size_t)H * W;
  const bool want_mob = MASK == MASK_COMPUTED && (LEAN || (p.flags & TCLB200_MOB));
  const float* s_bv = s_bu + Cfg::kBfH * Cfg::kBfW;
  const PairPtrs<FrameT> io = pair_ptrs<FrameT>(p, t.pair, t.cf, CT > 0 ? CT : p.C, plane);
  const int ox = meta[0], oy = meta[1], mode = meta[2];   // mode 0: nothing staged, 1: every tap in the boxes, 2: mixed
  const SmemSrc<float, Cfg::BW, Cfg::BH * Cfg::BW> fs{s_ff, ox, oy};
  const SmemSrc<FrameT, Cfg::BW, Cfg::BH * Cfg::BW> ps{s_prev, ox, oy};
  const GlobalSrc<float> fg{p.ff ? p.ff + (size_t)t.ffi * p.ff_batch : nullptr, p.ff_plane, g};
  const GlobalSrc<FrameT> pg{p.prev ? reinterpret_cast<const FrameT*>(p.prev) + (size_t)t.pf * (CT > 0 ? CT : p.C) * plane : nullptr, plane, g};
  float err = 0.0f;
#pragma unroll
  for (int k = 0; k < Cfg::kPPL; ++k) {   // fully unrolled: cur[k] / mk[k] must stay in registers
    const int lx = lx0, ly = ly0 + pix_dy(k);
    const int x = t.x0 + lx, y = t.y0 + ly;
    if (EDGE && (x >= W || y >= p.row_end)) continue;
    const int c = (ly + 1) * Cfg::kBfW + lx + Cfg::kHaloL;
    const float u = s_bu[c], v = s_bv[c];
    float nb, keep = 1.0f;
    if (want_mob) {
      float margin;
      if (motion_boundary(u, v, s_bu[c - 1], s_bu[c + 1], s_bu[c - Cfg::kBfW], s_bu[c + Cfg::kBfW], s_bv[c - 1], s_bv[c + 1],
                          s_bv[c - Cfg::kBfW], s_bv[c + Cfg::kBfW], kV, &nb, &margin))
        keep = 0.0f;
      if (!LEAN) near += fabsf(margin) < kNearBand;
    } else {
      nb = sqnorm2(u, v, kV);
    }
    const PixTaps taps = pix_taps(u, v, x, y, g);
    const size_t o = (size_t)y * W + x;
    if (MASK == MASK_GIVEN) keep = mk[k];
    const float* cv = have_cur ? cur[k] : nullptr;
    // taps [x0, x0+1] x [y0, y0+1] inside the staged boxes?  (unsigned compare: also catches negatives / saturation)
    const bool inbox = mode == 1 || (mode == 2 && (unsigned)(taps.x0 - ox) < (unsigned)(Cfg::BW - 1) &&
                                     (unsigned)(taps.y0 - oy) < (unsigned)(Cfg::BH - 1));
    if (inbox) finish_pixel<FrameT, MASK, REDUCE, CT, LEAN>(p, taps, u, v, nb, keep, o, plane, t.pair, fs, ps, io, cv, err, near);
    else finish_pixel<FrameT, MASK, REDUCE, CT, LEAN>(p, taps, u, v, nb, keep, o, plane, t.pair, fg, pg, io, cv, err, near);   // exact predicated gathers
  }
  return err;
}

// ---- consumer: the hot configuration (LEAN: C == 3, L2 error, no optional outputs), staged tiles only ----------
// The mask tests compare  lhs > rhs  where both sides are sums of torch.norm(.)**2 terms, i.e. sqrt-then-square
// of a sum of squares (flowtools.py:41-53).  Each such term differs from the plain sum of squares by at most a few
// ulp (< 12 * 2^-24 relative per side), so the plain (sqrt-free) evaluation decides the test whenever lhs lies outside
// [rhs * (1 - kFilterEps), rhs * (1 + kFilterEps)]; only the remaining pixels (a few per million) replay the exact
// sequence after the branch-free pixel loop.  Results are identical to the exact path.
constexpr float kFilterEps = 4e-6f;

struct LeanGeo {   // per-thread constants of lean_tile
  float i2x, i2y, Wf, Hf;
};

// sampling position of one pixel of a staged tile: floor parts (as floats: exact integers) + the four weights
struct LeanTaps {
  float fxf, fyf;   // floor(ix), floor(iy)
  float nw, ne, sw, se;
};
__device__ __forceinline__ LeanTaps lean_taps(float xf, float yf, float u, float v, const LeanGeo& lg) {
  // the reference's [-1,1] round trip (flowtools.py:28-29 + grid_sampler's unnormalise).  Inside a staged tile every
  // coordinate is finite and far inside the int range: no safe_downgrade guard needed.
  const float ax = __fadd_rn(xf, u), ay = __fadd_rn(yf, v);
  const float tx = __fadd_rn(__fsub_rn(__fmul_rn(ax, lg.i2x), 1.0f), 1.0f), ty = __fadd_rn(__fsub_rn(__fmul_rn(ay, lg.i2y), 1.0f), 1.0f);
  const float ix = __fmul_rn(__fmaf_rn(tx, lg.Wf, -1.0f), 0.5f), iy = __fmul_rn(__fmaf_rn(ty, lg.Hf, -1.0f), 0.5f);
  LeanTaps t;
  t.fxf = floorf(ix); t.fyf = floorf(iy);
  const float fx1 = __fsub_rn(__fadd_rn(t.fxf, 1.0f), ix), fx0 = __fsub_rn(ix, t.fxf);
  const float fy1 = __fsub_rn(__fadd_rn(t.fyf, 1.0f), iy), fy0 = __fsub_rn(iy, t.fyf);
  t.nw = __fmul_rn(fx1, fy1); t.ne = __fmul_rn(fx0, fy1); t.sw = __fmul_rn(fx1, fy0); t.se = __fmul_rn(fx0, fy0);
  return t;
}

// exact mask verdict of one pixel of a staged tile (the rare replay of lean_tile)
template <typename Cfg, bool OCC>
__device__ __noinline__ bool exact_keep(const float* s_bu, const float* s_ff, int c, float xf, float yf, LeanGeo lg, float box_xf, float box_yf) {
  constexpr int BW = Cfg::BW, BFW = Cfg::kBfW, PL = Cfg::BH * Cfg::BW;
  const float* s_bv = s_bu + Cfg::kBfH * BFW;
  const float u = s_bu[c], v = s_bv[c];
  float nb, m1, m2;
  const bool mob = motion_boundary(u, v, s_bu[c - 1], s_bu[c + 1], s_bu[c - BFW], s_bu[c + BFW], s_bv[c - 1], s_bv[c + 1],
                                   s_bv[c - BFW], s_bv[c + BFW], kV, &nb, &m1);
  if (!OCC) return !mob;   // the optimisation-based variant: motion-boundary test only
  const LeanTaps t = lean_taps(xf, yf, u, v, lg);
  const float* f0 = s_ff + (int)__fmaf_rn(__fsub_rn(t.fyf, box_yf), (float)BW, __fsub_rn(t.fxf, box_xf));
  float a = __fmul_rn(f0[0], t.nw);
  a = __fmaf_rn(f0[1], t.ne, a); a = __fmaf_rn(f0[BW], t.sw, a); a = __fmaf_rn(f0[BW + 1], t.se, a);
  float b = __fmul_rn(f0[PL], t.nw);
  b = __fmaf_rn(f0[PL + 1], t.ne, b); b = __fmaf_rn(f0[PL + BW], t.sw, b); b = __fmaf_rn(f0[PL + BW + 1], t.se, b);
  const bool occ = occluded(a, b, u, v, nb, kV, &m2);
  return !mob && !occ;
}

// one pixel of the hot configuration entirely from global memory with the exact sequences: the pixels of a "mixed" tile
// (a motion boundary runs through it) whose taps lie outside the staged source boxes.  Returns the masked squared error.
template <typename FrameT, int MASK, bool KEEP_ONLY, int LOSS>
__device__ __noinline__ float pixel_global(const float* bf_pair, size_t bf_plane, const float* ff_pair, size_t ff_plane, const FrameT* prev_pair,
                                           Geo g, int x, int y, float c0, float c1, float c2, float mkv) {
  const int W = g.W, H = g.H;
  const size_t plane = (size_t)H * W;
  const size_t o = (size_t)y * W + x;
  const float* bu = bf_pair;
  const float* bv = bf_pair + bf_plane;
  const float u = __ldg(bu + o), v = __ldg(bv + o);
  bool keep = true;
  float nb = 0.0f;
  if (MASK == MASK_COMPUTED) {
    const float ul = x > 0 ? __ldg(bu + o - 1) : 0.0f, ur = x + 1 < W ? __ldg(bu + o + 1) : 0.0f;
    const float uu = y > 0 ? __ldg(bu + o - W) : 0.0f, ud = y + 1 < H ? __ldg(bu + o + W) : 0.0f;
    const float vl = x > 0 ? __ldg(bv + o - 1) : 0.0f, vr = x + 1 < W ? __ldg(bv + o + 1) : 0.0f;
    const float vu = y > 0 ? __ldg(bv + o - W) : 0.0f, vd = y + 1 < H ? __ldg(bv + o + W) : 0.0f;
    float margin;
    keep = !motion_boundary(u, v, ul, ur, uu, ud, vl, vr, vu, vd, kV, &nb, &margin);
  }
  const PixTaps s = pix_taps(u, v, x, y, g);
  if (MASK == MASK_COMPUTED) {
    const GlobalSrc<float> fsrc{ff_pair, ff_plane, g};
    const float wu = fsrc.sample(0, s), wv = fsrc.sample(1, s);
    float margin;
    if (occluded(wu, wv, u, v, nb, kV, &margin)) keep = false;
  }
  if (KEEP_ONLY) return keep ? 1.0f : 0.0f;
  const GlobalSrc<FrameT> psrc{prev_pair, plane, g};
  const float d0 = __fsub_rn(c0, psrc.sample(0, s)), d1 = __fsub_rn(c1, psrc.sample(1, s)), d2 = __fsub_rn(c2, psrc.sample(2, s));
  const float acc = LOSS == TCLB200_L1 ? __fadd_rn(__fadd_rn(fabsf(d0), fabsf(d1)), fabsf(d2)) : __fmaf_rn(d2, d2, __fmaf_rn(d1, d1, __fmul_rn(d0, d0)));
  if (MASK == MASK_GIVEN) return __fmul_rn(LOSS == TCLB200_L1 ? mkv : __fmul_rn(mkv, mkv), acc);
  return keep ? acc : 0.0f;
}

// shared-memory reads at a 32-bit shared address + compile-time offset (the tap reads of the staged tiles: the box
// address of a pixel is computed in floating point straight from floor(ix), floor(iy) and serves all planes)
template <int OFF>
__device__ __forceinline__ float lds_tap(uint32_t a, float) {
  float v;
  asm volatile("ld.shared.f32 %0, [%1+%2];" : "=f"(v) : "r"(a), "n"(OFF));
  return v;
}
template <int OFF>
__device__ __forceinline__ float lds_tap(uint32_t a, __nv_bfloat16) {
  unsigned h;   // (ld may write a register wider than its type: zero-extended)
  asm volatile("ld.shared.u16 %0, [%1+%2];" : "=r"(h) : "r"(a), "n"(OFF));
  return __uint_as_float(h << 16);
}
// one plane of a staged box, grid_sampler_2d's accumulation order (zero-filled outside the image: all four taps are plain reads)
template <typename T, int OFF, int PITCH>
__device__ __forceinline__ float staged_tap4(uint32_t a, const LeanTaps& tp) {
  constexpr int E = (int)sizeof(T);
  float w = __fmul_rn(lds_tap<OFF>(a, T()), tp.nw);
  w = __fmaf_rn(lds_tap<OFF + E>(a, T()), tp.ne, w);
  w = __fmaf_rn(lds_tap<OFF + PITCH * E>(a, T()), tp.sw, w);
  w = __fmaf_rn(lds_tap<OFF + PITCH * E + E>(a, T()), tp.se, w);
  return w;
}

// CT == 3: masked squared error against `cur` (returned); CT == 0: mask-only (fbcCheckTorch), the verdicts go to mask_out
// OCC == false (mask-only): the optimisation-based variant of fbcCheckTorch, motion-boundary test alone -- no source
// boxes are staged and no sampling position is needed (methods/optimization-based/flowtools.py:34-58)
// OUTS (staged, non-mixed tiles of the reducing configurations): the optional per-pixel outputs -- warp_out, mask_out,
// blend_out, whichever pointers are set -- are stored from the same pass (the warped values wait in registers until the
// mask verdicts are final)
template <typename FrameT, int MASK, int CT, int LOSS, typename Cfg, bool EDGE, bool MIXED, bool OCC = true, bool OUTS = false>
__device__ __forceinline__ float lean_tile(const FwdParams& p, const float* s_bu, const float* s_ff, const int* meta, const TileId& t,
                                           int lx0, int ly0, const float (&cur)[Cfg::kPPL][Cfg::kC], const float (&mk)[Cfg::kPPL]) {
  constexpr int P = Cfg::kPPL, BW = Cfg::BW, BFW = Cfg::kBfW, PL = Cfg::BH * Cfg::BW;
  constexpr float kHi = 1.0f + kFilterEps, kLo = 1.0f - kFilterEps;
  constexpr int FE = (int)sizeof(FrameT);
  const Geo& g = p.geo;
  const float* s_bv = s_bu + Cfg::kBfH * BFW;
  // the prev boxes follow the ff boxes in the stage
  const FrameT* s_prev = reinterpret_cast<const FrameT*>(reinterpret_cast<const unsigned char*>(s_ff) + Cfg::kFfStage);
  const int box_x = meta[0], box_y = meta[1];
  const float box_xf = (float)box_x, box_yf = (float)box_y;
  const ptrdiff_t gplane = (ptrdiff_t)g.H * g.W;
  const float* gff = (MIXED && MASK == MASK_COMPUTED) ? p.ff + (size_t)t.ffi * p.ff_batch : nullptr;
  const FrameT* gprev = (MIXED && CT == 3) ? reinterpret_cast<const FrameT*>(p.prev) + (size_t)t.pf * 3 * gplane : nullptr;
  LeanGeo lg;
  lg.i2x = __fmul_rn(2.0f, g.inv_dx); lg.i2y = __fmul_rn(2.0f, g.inv_dy);   // exact doubling: (2a)*r == a*(2r)
  lg.Wf = g.Wf; lg.Hf = g.Hf;
  const float xf = (float)(t.x0 + lx0), yf0 = (float)(t.y0 + ly0);
  const int c0 = (ly0 + 1) * BFW + lx0 + Cfg::kHaloL;
  const bool xin = !EDGE || t.x0 + lx0 < g.W;
  const bool validity = MASK == MASK_NONE && (p.flags & TCLB200_VALIDITY);
  // staged tiles: byte address of a pixel's top-left tap = base + 4 * ((fyf - box_y) * BW + (fxf - box_x)), evaluated with two
  // fmas on exact small integers (the placement keeps |box| < 2^15, so every intermediate is an integer below 2^24)
  const uint32_t ff_base = smem_u32(s_ff), prev_base = smem_u32(s_prev);
  const float ff_k = __fsub_rn((float)ff_base, 4.0f * __fmaf_rn(box_yf, (float)BW, box_xf));
  const float prev_k = __fsub_rn((float)prev_base, (float)FE * __fmaf_rn(box_yf, (float)BW, box_xf));
  float e[P];
  float wv[OUTS ? P : 1][3];
  unsigned keepbits = 0, ambbits = 0, outbits = 0;
  {
    // this lane's column of the flow tile: rows -1 .. 2 * P - 1 relative to the lane's first row (its own pixels are the
    // odd entries, the even ones belong to the partner lane)
    float uc[2 * P + 1], vc[2 * P + 1], ul[P], ur[P], vl[P], vr[P];
#pragma unroll
    for (int r = 0; r < 2 * P + 1; ++r) {
      if (MASK == MASK_COMPUTED || (r & 1)) { uc[r] = s_bu[c0 + (r - 1) * BFW]; vc[r] = s_bv[c0 + (r - 1) * BFW]; }
      else { uc[r] = 0.0f; vc[r] = 0.0f; }
    }
#pragma unroll
    for (int j = 0; j < P; ++j) {
      if (MASK == MASK_COMPUTED) {
        ul[j] = s_bu[c0 + 2 * j * BFW - 1]; ur[j] = s_bu[c0 + 2 * j * BFW + 1];
        vl[j] = s_bv[c0 + 2 * j * BFW - 1]; vr[j] = s_bv[c0 + 2 * j * BFW + 1];
      } else { ul[j] = ur[j] = vl[j] = vr[j] = 0.0f; }
    }
#pragma unroll
    for (int j = 0; j < P; ++j) {
      const int k = j, dyk = 2 * j;
      const bool inside = !EDGE || (xin && t.y0 + ly0 + dyk < p.row_end);
      const float u = uc[2 * j + 1], v = vc[2 * j + 1];
      const float s0 = __fmaf_rn(u, u, __fmul_rn(v, v));
      bool keep = inside, amb = false;
      if (MASK == MASK_COMPUTED) {
        // motion boundary: 4*(|grad u|^2 + |grad v|^2)  vs  4*(0.01*|bf|^2 + 0.002)
        const float dux = __fsub_rn(ur[j], ul[j]), duy = __fsub_rn(uc[2 * j + 2], uc[2 * j]);
        const float dvx = __fsub_rn(vr[j], vl[j]), dvy = __fsub_rn(vc[2 * j + 2], vc[2 * j]);
        const float G = __fmaf_rn(dux, dux, __fmaf_rn(duy, duy, __fmaf_rn(dvx, dvx, __fmul_rn(dvy, dvy))));
        const float Rhi = __fmaf_rn(4.0f * 0.01f * kHi, s0, 4.0f * 0.002f * kHi), Rlo = __fmaf_rn(4.0f * 0.01f * kLo, s0, 4.0f * 0.002f * kLo);
        const bool mob = G > Rhi;
        keep = keep && !mob;
        amb = !(mob || G < Rlo);
      }
      const float yf = yf0 + (float)dyk;
      const LeanTaps tp = lean_taps(xf, yf, u, v, lg);
      // pixels beyond the image edge read any in-box address, their result is discarded
      bool inbox = true;
      float rx = 0.0f, ry = 0.0f;
      if (MIXED) {
        rx = __fsub_rn(tp.fxf, box_xf); ry = __fsub_rn(tp.fyf, box_yf);
        inbox = !inside || (rx >= 0.0f && rx < (float)(BW - 1) && ry >= 0.0f && ry < (float)(Cfg::BH - 1));
      }
      float a = 0.0f, b = 0.0f, w3[3] = {0.0f, 0.0f, 0.0f};
      if (!MIXED) {
        // every tap of the tile lies inside the staged boxes (zero-filled outside the image)
        uint32_t fa = (uint32_t)__float2int_rn(__fmaf_rn(tp.fyf, 4.0f * (float)BW, __fmaf_rn(tp.fxf, 4.0f, ff_k)));
        if (EDGE && !inside) fa = ff_base;
#if TCL_DIAG == 3
        fa = ff_base + ((fa - ff_base) & 0xffcu);
#endif
        if (MASK == MASK_COMPUTED && OCC) {
          a = staged_tap4<float, 0, BW>(fa, tp);
          b = staged_tap4<float, PL * 4, BW>(fa, tp);
        }
        if (CT == 3) {
          if (FE == 4) {   // fp32 frames: the prev planes sit behind the ff planes, the same address register serves them
            w3[0] = staged_tap4<FrameT, (int)Cfg::kFfStage, BW>(fa, tp);
            w3[1] = staged_tap4<FrameT, (int)Cfg::kFfStage + PL * FE, BW>(fa, tp);
            w3[2] = staged_tap4<FrameT, (int)Cfg::kFfStage + 2 * PL * FE, BW>(fa, tp);
          } else {
            uint32_t pa = (uint32_t)__float2int_rn(__fmaf_rn(tp.fyf, (float)(FE * BW), __fmaf_rn(tp.fxf, (float)FE, prev_k)));
            if (EDGE && !inside) pa = prev_base;
            w3[0] = staged_tap4<FrameT, 0, BW>(pa, tp);
            w3[1] = staged_tap4<FrameT, PL * FE, BW>(pa, tp);
            w3[2] = staged_tap4<FrameT, 2 * PL * FE, BW>(pa, tp);
          }
        }
      } else {
        // mixed tile: the staged boxes, or -- pixels whose taps left the boxes -- global memory with grid_sample's zero
        // padding as per-tap predicates
        const int q = !(inside && inbox) ? 0 : (int)__fmaf_rn(ry, (float)BW, rx);
        const float* pf = s_ff + q;
        const FrameT* pp = s_prev + q;
        int rs = BW;
        ptrdiff_t ps = PL, psf = PL;   // plane pitch of the frame / flow planes behind pp / pf
        bool p00 = true, p10 = true, p01 = true, p11 = true;
        if (!inbox) {
          const int gx = (int)tp.fxf, gy = (int)tp.fyf;   // top-left tap in the image (sane: the placement checked)
          const ptrdiff_t off = (ptrdiff_t)gy * g.W + gx;
          if (MASK == MASK_COMPUTED) pf = gff + off;
          if (CT == 3) pp = gprev + off;
          rs = g.W; ps = gplane; psf = (ptrdiff_t)p.ff_plane;
          const bool xin0 = (unsigned)gx < (unsigned)g.W, xin1 = (unsigned)(gx + 1) < (unsigned)g.W;
          const bool yin0 = (unsigned)gy < (unsigned)g.H, yin1 = (unsigned)(gy + 1) < (unsigned)g.H;
          p00 = xin0 && yin0; p10 = xin1 && yin0; p01 = xin0 && yin1; p11 = xin1 && yin1;
        }
        auto tap4 = [&](auto* bp) {   // one plane, grid_sampler_2d's accumulation order
          float w = __fmul_rn(p00 ? to_f32(bp[0]) : 0.0f, tp.nw);
          w = __fmaf_rn(p10 ? to_f32(bp[1]) : 0.0f, tp.ne, w);
          w = __fmaf_rn(p01 ? to_f32(bp[rs]) : 0.0f, tp.sw, w);
          w = __fmaf_rn(p11 ? to_f32(bp[rs + 1]) : 0.0f, tp.se, w);
          return w;
        };
        if (MASK == MASK_COMPUTED && OCC) { a = tap4(pf); b = tap4(pf + psf); }
#pragma unroll
        for (int ch = 0; ch < CT; ++ch) w3[ch] = tap4(pp + ch * ps);
      }
      if (MASK == MASK_COMPUTED && OCC) {
        // occlusion: |wf+bf|^2  vs  0.01*(|wf|^2+|bf|^2) + 0.5
        const float su = __fadd_rn(a, u), sv = __fadd_rn(b, v);
        const float L = __fmaf_rn(su, su, __fmul_rn(sv, sv));
        const float nn = __fadd_rn(__fmaf_rn(a, a, __fmul_rn(b, b)), s0);
        const float Rhi = __fmaf_rn(0.01f * kHi, nn, 0.5f * kHi), Rlo = __fmaf_rn(0.01f * kLo, nn, 0.5f * kLo);
        const bool occ = L > Rhi;
        keep = keep && !occ;
        amb = amb || !(occ || L < Rlo);
      }
      float acc = 0.0f;
      float valid = 1.0f;
      if (MASK == MASK_NONE && validity) {   // fs_lib.warp: times the binarised warp of an all-ones image (fs_lib.py:29-37)
        const int gx = (int)tp.fxf, gy = (int)tp.fyf;
        Taps vt;
        const bool xin0 = (unsigned)gx < (unsigned)g.W, xin1 = (unsigned)(gx + 1) < (unsigned)g.W;
        const bool yin0 = (unsigned)gy < (unsigned)g.H, yin1 = (unsigned)(gy + 1) < (unsigned)g.H;
        vt.p00 = xin0 && yin0; vt.p10 = xin1 && yin0; vt.p01 = xin0 && yin1; vt.p11 = xin1 && yin1;
        vt.nw = tp.nw; vt.ne = tp.ne; vt.sw = tp.sw; vt.se = tp.se; vt.o00 = 0;
        valid = binarise_validity(ones_sample(vt, kV));
      }
#pragma unroll
      for (int ch = 0; ch < CT; ++ch) {
        const float w = w3[ch];
        if (MASK == MASK_NONE) {   // warp() on its own: store the warped frame (two coalesced row segments per warp instruction)
          if (inside)
            st_stream(reinterpret_cast<FrameT*>(p.warp_out) + ((size_t)t.pair * 3 + ch) * gplane + (size_t)(t.y0 + ly0 + dyk) * g.W + (t.x0 + lx0),
                      validity ? __fmul_rn(w, valid) : w);
          continue;
        }
        if (OUTS) wv[k][ch] = w;
        const float d = __fsub_rn(cur[k][ch], w);
        acc = LOSS == TCLB200_L1 ? __fadd_rn(acc, fabsf(d)) : __fmaf_rn(d, d, acc);   // mask*|warp - cur| (MoGAN :281) / (mask*(cur - warp))^2
      }
      // (m*d)^2 resp. m*|d| summed over channels (mk = 0 outside the image)
      e[k] = MASK == MASK_GIVEN ? __fmul_rn(LOSS == TCLB200_L1 ? mk[k] : __fmul_rn(mk[k], mk[k]), acc) : acc;
      keepbits |= (keep ? 1u : 0u) << k;
      ambbits |= (amb && inside && inbox ? 1u : 0u) << k;
      if (MIXED) outbits |= (amb && inside && !inbox ? 1u : 0u) << k;
    }
  }
  // rare, divergent: tests too close to call replay the exact sequences (a few pixels per million) ...
  if (MASK == MASK_COMPUTED && __builtin_expect(ambbits != 0, 0)) {
#pragma unroll
    for (int k = 0; k < P; ++k)
      if ((ambbits >> k) & 1u) {
        const bool kp = exact_keep<Cfg, OCC>(s_bu, s_ff, c0 + pix_dy(k) * BFW, xf, yf0 + (float)pix_dy(k), lg, box_xf, box_yf);
        keepbits = (keepbits & ~(1u << k)) | ((kp ? 1u : 0u) << k);
      }
  }
  // ... the same for pixels of a mixed tile whose taps left the boxes: redone from global memory
  if (MIXED && __builtin_expect(outbits != 0, 0)) {
    const size_t plane = (size_t)g.H * g.W;
#pragma unroll
    for (int k = 0; k < P; ++k)
      if ((outbits >> k) & 1u) {
        if (CT == 3) {
          e[k] = pixel_global<FrameT, MASK, false, LOSS>(p.bf + (size_t)t.bfi * p.bf_batch, p.bf_plane, p.ff + (size_t)t.ffi * p.ff_batch, p.ff_plane,
                                                   reinterpret_cast<const FrameT*>(p.prev) + (size_t)t.pf * 3 * plane, g, t.x0 + lx0,
                                                   t.y0 + ly0 + pix_dy(k), cur[k][0], cur[k][1], cur[k][2], mk[k]);
          keepbits |= 1u << k;   // the verdict is already applied
        } else {
          const float kp = pixel_global<FrameT, MASK, true, LOSS>(p.bf + (size_t)t.bfi * p.bf_batch, p.bf_plane, p.ff + (size_t)t.ffi * p.ff_batch, p.ff_plane, nullptr, g,
                                                            t.x0 + lx0, t.y0 + ly0 + pix_dy(k), 0.0f, 0.0f, 0.0f, 0.0f);
          keepbits = (keepbits & ~(1u << k)) | ((kp != 0.0f ? 1u : 0u) << k);
        }
      }
  }
  if (OUTS && CT == 3) {
    const size_t pix0 = (size_t)(t.y0 + ly0) * g.W + (t.x0 + lx0);
    FrameT* wo = p.warp_out ? reinterpret_cast<FrameT*>(p.warp_out) + (size_t)t.pair * 3 * gplane + pix0 : nullptr;
    FrameT* bo = p.blend_out ? reinterpret_cast<FrameT*>(p.blend_out) + (size_t)t.pair * 3 * gplane + pix0 : nullptr;
    float* mo = (MASK == MASK_COMPUTED && p.mask_out) ? p.mask_out + (size_t)t.pair * gplane + pix0 : nullptr;
#pragma unroll
    for (int k = 0; k < P; ++k) {
      const bool inside = !EDGE || (xin && t.y0 + ly0 + pix_dy(k) < p.row_end);
      if (!inside) continue;
      const ptrdiff_t off = (ptrdiff_t)pix_dy(k) * g.W;
      const float keepf = MASK == MASK_GIVEN ? mk[k] : (((keepbits >> k) & 1u) ? 1.0f : 0.0f);
      if (mo) __stcs(mo + off, keepf);
#pragma unroll
      for (int ch = 0; ch < 3; ++ch) {
        if (wo) st_stream(wo + ch * gplane + off, wv[k][ch]);
        if (bo)   // m*warp + (1-m)*img   obst_eval.py:500
          st_stream(bo + ch * gplane + off, __fadd_rn(__fmul_rn(keepf, wv[k][ch]), __fmul_rn(__fsub_rn(1.0f, keepf), cur[k][ch])));
      }
    }
  }
  if (CT == 0) {   // mask-only: store the verdicts (two coalesced 64-byte row segments per warp instruction)
    float* mo = p.mask_out + (size_t)t.pair * gplane + (size_t)(t.y0 + ly0) * g.W + (t.x0 + lx0);
#pragma unroll
    for (int k = 0; k < P; ++k) {
      const bool inside = !EDGE || (xin && t.y0 + ly0 + pix_dy(k) < p.row_end);
      if (inside) __stcs(mo + (ptrdiff_t)pix_dy(k) * g.W, ((keepbits >> k) & 1u) ? 1.0f : 0.0f);
    }
    return 0.0f;
  }
  float err = 0.0f;
#pragma unroll
  for (int k = 0; k < P; ++k) {
    if (MASK == MASK_GIVEN) err = __fadd_rn(err, e[k]);
    else err = ((keepbits >> k) & 1u) ? __fadd_rn(err, e[k]) : err;
  }
  return err;
}

// ---- consumer: the hot configurations on staged, interior tiles with packed fp32 arithmetic --------------------------
// Same operation sequence as lean_tile, two of the lane's pixels per instruction: sm_100's FFMA2 / FADD2 / FMUL2 round
// every component to nearest exactly like their scalar forms (results are bit-identical, the parity tests do not tell
// the two paths apart), but halve the issue slots and the instruction energy of the ~70 floating-point operations a
// pixel needs -- the kernel is bound by instruction issue and, sustained, by the board's power cap, not by the FMA pipe.
// Loads, floor, float -> int and the comparisons stay scalar.
__device__ __forceinline__ float2 f2(float a, float b) { return make_float2(a, b); }
__device__ __forceinline__ float2 f2(float a) { return make_float2(a, a); }
__device__ __forceinline__ float2 add2(float2 a, float2 b) { return __fadd2_rn(a, b); }
__device__ __forceinline__ float2 sub2(float2 a, float2 b) { return __fadd2_rn(a, make_float2(-b.x, -b.y)); }
__device__ __forceinline__ float2 mul2(float2 a, float2 b) { return __fmul2_rn(a, b); }
__device__ __forceinline__ float2 fma2(float2 a, float2 b, float2 c) { return __ffma2_rn(a, b, c); }

template <typename T, int OFF, int PITCH>
__device__ __forceinline__ float2 staged_tap4x2(uint32_t a0, uint32_t a1, float2 nw, float2 ne, float2 sw, float2 se) {
  constexpr int E = (int)sizeof(T);
  float2 w = mul2(f2(lds_tap<OFF>(a0, T()), lds_tap<OFF>(a1, T())), nw);
  w = fma2(f2(lds_tap<OFF + E>(a0, T()), lds_tap<OFF + E>(a1, T())), ne, w);
  w = fma2(f2(lds_tap<OFF + PITCH * E>(a0, T()), lds_tap<OFF + PITCH * E>(a1, T())), sw, w);
  w = fma2(f2(lds_tap<OFF + PITCH * E + E>(a0, T()), lds_tap<OFF + PITCH * E + E>(a1, T())), se, w);
  return w;
}

// EDGE: the tile overhangs the image (pixels outside are computed on a safe address and dropped); MIXED: a motion boundary
// runs through the tile and the taps of some pixels lie outside the staged boxes -- those pixels are redone one by one
// from global memory after the loop (pixel_global, exact), every other pixel of the tile keeps the fast path.
template <typename FrameT, int MASK, int LOSS, typename Cfg, bool EDGE = false, bool MIXED = false, int CT = 3>
__device__ __forceinline__ float lean_tile_packed(const FwdParams& p, const float* s_bu, const float* s_ff, const int* meta, const TileId& t,
                                                  int lx0, int ly0, const float (&cur)[Cfg::kPPL][Cfg::kC], const float (&mk)[Cfg::kPPL]) {
  constexpr int P = Cfg::kPPL, BW = Cfg::BW, BFW = Cfg::kBfW, PL = Cfg::BH * Cfg::BW;
  constexpr float kHi = 1.0f + kFilterEps, kLo = 1.0f - kFilterEps;
  constexpr int FE = (int)sizeof(FrameT);
  // CT == 3: the reducing configurations (computeTCL, training loss); CT == 0: fbcCheckTorch on its own (mask_out only, no frames)
  static_assert(P % 2 == 0 && MASK != MASK_NONE && ((CT == 3 && Cfg::kC == 3) || (CT == 0 && MASK == MASK_COMPUTED)), "pixel pairs; three channels or mask-only");
  // mixed tiles, pixels whose taps left the boxes: computed masks fetch those taps from global memory inside the loop (a
  // warp-uniform branch); with a dataset mask the pixel is so cheap that waiting for global loads inside the loop costs
  // more than redoing the few pixels after it (measured: 131 vs 149 Gpix/s on the Sintel shape)
  constexpr bool kFixInLoop = MASK == MASK_COMPUTED;
  const Geo& g = p.geo;
  const float* s_bv = s_bu + Cfg::kBfH * BFW;
  const FrameT* s_prev = reinterpret_cast<const FrameT*>(reinterpret_cast<const unsigned char*>(s_ff) + Cfg::kFfStage);
  const float box_xf = (float)meta[0], box_yf = (float)meta[1];
  LeanGeo lg;
  lg.i2x = __fmul_rn(2.0f, g.inv_dx); lg.i2y = __fmul_rn(2.0f, g.inv_dy);   // exact doubling: (2a)*r == a*(2r)
  lg.Wf = g.Wf; lg.Hf = g.Hf;
  const float xf = (float)(t.x0 + lx0), yf0 = (float)(t.y0 + ly0);
  const int c0 = (ly0 + 1) * BFW + lx0 + Cfg::kHaloL;
  const size_t gplane = (size_t)g.H * g.W;
  const GlobalSrc<float> fg{(MIXED && MASK == MASK_COMPUTED) ? p.ff + (size_t)t.ffi * p.ff_batch : nullptr, p.ff_plane, g};
  const GlobalSrc<FrameT> pg{(MIXED && CT == 3) ? reinterpret_cast<const FrameT*>(p.prev) + (size_t)t.pf * 3 * gplane : nullptr, gplane, g};
  const bool xin = !EDGE || t.x0 + lx0 < g.W;
  const int rows_in = EDGE ? p.row_end - (t.y0 + ly0) : INT_MAX;   // pixel k is inside the image iff 2 * k < rows_in (and xin)
  const float bx_hi = box_xf + (float)(BW - 2), by_hi = box_yf + (float)(Cfg::BH - 2);   // top-left taps inside the boxes: [box, box + size - 2]
  // byte address of a pixel's top-left tap, in floating point (see lean_tile)
  const uint32_t ff_base = smem_u32(s_ff), prev_base = smem_u32(s_prev);
  const float ff_k = __fsub_rn((float)ff_base, 4.0f * __fmaf_rn(box_yf, (float)BW, box_xf));
  const float prev_k = __fsub_rn((float)prev_base, (float)FE * __fmaf_rn(box_yf, (float)BW, box_xf));
  // this lane's column of the flow tile (see lean_tile)
  float uc[2 * P + 1], vc[2 * P + 1], ul[P], ur[P], vl[P], vr[P];
#pragma unroll
  for (int r = 0; r < 2 * P + 1; ++r) {
    if (MASK == MASK_COMPUTED || (r & 1)) { uc[r] = s_bu[c0 + (r - 1) * BFW]; vc[r] = s_bv[c0 + (r - 1) * BFW]; }
    else { uc[r] = 0.0f; vc[r] = 0.0f; }
  }
#pragma unroll
  for (int j = 0; j < P; ++j) {
    if (MASK == MASK_COMPUTED) {
      ul[j] = s_bu[c0 + 2 * j * BFW - 1]; ur[j] = s_bu[c0 + 2 * j * BFW + 1];
      vl[j] = s_bv[c0 + 2 * j * BFW - 1]; vr[j] = s_bv[c0 + 2 * j * BFW + 1];
    } else { ul[j] = ur[j] = vl[j] = vr[j] = 0.0f; }
  }
  float e[P];
  unsigned keepbits = 0, ambbits = 0, outbits = 0;
#pragma unroll
  for (int q = 0; q < P / 2; ++q) {
    const int j0 = 2 * q, j1 = 2 * q + 1;   // the pair's pixels: rows ly0 + 2 * j0, ly0 + 2 * j1
    const float2 u = f2(uc[2 * j0 + 1], uc[2 * j1 + 1]), v = f2(vc[2 * j0 + 1], vc[2 * j1 + 1]);
    const float2 s0 = fma2(u, u, mul2(v, v));
    const bool in0 = !EDGE || (xin && 2 * j0 < rows_in), in1 = !EDGE || (xin && 2 * j1 < rows_in);
    bool keep0 = in0, keep1 = in1, amb0 = false, amb1 = false;
    if (MASK == MASK_COMPUTED) {
      // motion boundary: 4*(|grad u|^2 + |grad v|^2)  vs  4*(0.01*|bf|^2 + 0.002)
      const float2 dux = sub2(f2(ur[j0], ur[j1]), f2(ul[j0], ul[j1])), duy = sub2(f2(uc[2 * j0 + 2], uc[2 * j1 + 2]), f2(uc[2 * j0], uc[2 * j1]));
      const float2 dvx = sub2(f2(vr[j0], vr[j1]), f2(vl[j0], vl[j1])), dvy = sub2(f2(vc[2 * j0 + 2], vc[2 * j1 + 2]), f2(vc[2 * j0], vc[2 * j1]));
      const float2 G = fma2(dux, dux, fma2(duy, duy, fma2(dvx, dvx, mul2(dvy, dvy))));
      const float2 Rhi = fma2(f2(4.0f * 0.01f * kHi), s0, f2(4.0f * 0.002f * kHi)), Rlo = fma2(f2(4.0f * 0.01f * kLo), s0, f2(4.0f * 0.002f * kLo));
      const bool mob0 = G.x > Rhi.x, mob1 = G.y > Rhi.y;
      keep0 = keep0 && !mob0; keep1 = keep1 && !mob1;
      amb0 = !(mob0 || G.x < Rlo.x); amb1 = !(mob1 || G.y < Rlo.y);
    }
    // sampling position: the reference's [-1,1] round trip (flowtools.py:28-29 + grid_sampler's unnormalise), see lean_taps
    const float2 ax = add2(f2(xf), u), ay = add2(f2(yf0 + (float)(2 * j0), yf0 + (float)(2 * j1)), v);
    // (the products are SCALAR multiplies on purpose: ptxas 12.9 contracts mul.rn.f32x2 + add.rn.f32x2 into one FFMA2 -- one
    // rounding instead of the reference's two -- although both carry .rn; it leaves scalar mul.rn / add.rn alone.  Seen as a
    // floor() one below the scanner's on a coordinate 5e-6 ulp from a rounding boundary: taps outside the staged box.)
    const float2 qx = f2(__fmul_rn(ax.x, lg.i2x), __fmul_rn(ax.y, lg.i2x)), qy = f2(__fmul_rn(ay.x, lg.i2y), __fmul_rn(ay.y, lg.i2y));
    const float2 tx = add2(add2(qx, f2(-1.0f)), f2(1.0f)), ty = add2(add2(qy, f2(-1.0f)), f2(1.0f));
    const float2 ix = mul2(fma2(tx, f2(lg.Wf), f2(-1.0f)), f2(0.5f)), iy = mul2(fma2(ty, f2(lg.Hf), f2(-1.0f)), f2(0.5f));
    const float2 fxf = f2(floorf(ix.x), floorf(ix.y)), fyf = f2(floorf(iy.x), floorf(iy.y));
    const float2 fx1 = sub2(add2(fxf, f2(1.0f)), ix), fx0 = sub2(ix, fxf);
    const float2 fy1 = sub2(add2(fyf, f2(1.0f)), iy), fy0 = sub2(iy, fyf);
    const float2 nw = mul2(fx1, fy1), ne = mul2(fx0, fy1), sw = mul2(fx1, fy0), se = mul2(fx0, fy0);
    const float2 faf = fma2(fyf, f2(4.0f * (float)BW), fma2(fxf, f2(4.0f), f2(ff_k)));
    uint32_t fa0 = (uint32_t)__float2int_rn(faf.x), fa1 = (uint32_t)__float2int_rn(faf.y);
    // pixels beyond the image edge, or -- mixed tiles -- with taps outside the boxes, read any in-box address; their
    // result is discarded (the latter are redone from global memory below)
    bool ok0 = in0, ok1 = in1;
    if (MIXED) {
      ok0 = ok0 && fxf.x >= box_xf && fxf.x <= bx_hi && fyf.x >= box_yf && fyf.x <= by_hi;
      ok1 = ok1 && fxf.y >= box_xf && fxf.y <= bx_hi && fyf.y >= box_yf && fyf.y <= by_hi;
    }
    if (EDGE || MIXED) { fa0 = ok0 ? fa0 : ff_base; fa1 = ok1 ? fa1 : ff_base; }
    float2 a = f2(0.0f), b = f2(0.0f), w3[3];
    if (MASK == MASK_COMPUTED) {
      a = staged_tap4x2<float, 0, BW>(fa0, fa1, nw, ne, sw, se);
      b = staged_tap4x2<float, PL * 4, BW>(fa0, fa1, nw, ne, sw, se);
    }
    if (CT == 0) {
      w3[0] = w3[1] = w3[2] = f2(0.0f);
    } else if (FE == 4) {   // fp32 frames: the prev planes sit behind the ff planes, the same address registers serve them
      w3[0] = staged_tap4x2<FrameT, (int)Cfg::kFfStage, BW>(fa0, fa1, nw, ne, sw, se);
      w3[1] = staged_tap4x2<FrameT, (int)Cfg::kFfStage + PL * FE, BW>(fa0, fa1, nw, ne, sw, se);
      w3[2] = staged_tap4x2<FrameT, (int)Cfg::kFfStage + 2 * PL * FE, BW>(fa0, fa1, nw, ne, sw, se);
    } else {
      const float2 paf = fma2(fyf, f2((float)(FE * BW)), fma2(fxf, f2((float)FE), f2(prev_k)));
      uint32_t pa0 = (uint32_t)__float2int_rn(paf.x), pa1 = (uint32_t)__float2int_rn(paf.y);
      if (EDGE || MIXED) { pa0 = ok0 ? pa0 : prev_base; pa1 = ok1 ? pa1 : prev_base; }
      w3[0] = staged_tap4x2<FrameT, 0, BW>(pa0, pa1, nw, ne, sw, se);
      w3[1] = staged_tap4x2<FrameT, PL * FE, BW>(pa0, pa1, nw, ne, sw, se);
      w3[2] = staged_tap4x2<FrameT, 2 * PL * FE, BW>(pa0, pa1, nw, ne, sw, se);
    }
    if (MIXED && kFixInLoop) {
      // pixels of the pair whose taps left the boxes: the same taps from global memory with grid_sample's zero padding as
      // per-tap predicates (exact); warp-uniform branch, most warps of a mixed tile never take it
      const bool o0 = in0 && !ok0, o1 = in1 && !ok1;
      if (__any_sync(0xffffffffu, o0 || o1)) {
        if (o0) {
          const PixTaps st{(int)fxf.x, (int)fyf.x, nw.x, ne.x, sw.x, se.x};
          if (MASK == MASK_COMPUTED) { a.x = fg.sample(0, st); b.x = fg.sample(1, st); }
          if (CT == 3) { w3[0].x = pg.sample(0, st); w3[1].x = pg.sample(1, st); w3[2].x = pg.sample(2, st); }
        }
        if (o1) {
          const PixTaps st{(int)fxf.y, (int)fyf.y, nw.y, ne.y, sw.y, se.y};
          if (MASK == MASK_COMPUTED) { a.y = fg.sample(0, st); b.y = fg.sample(1, st); }
          if (CT == 3) { w3[0].y = pg.sample(0, st); w3[1].y = pg.sample(1, st); w3[2].y = pg.sample(2, st); }
        }
      }
    }
    if (MASK == MASK_COMPUTED) {
      // occlusion: |wf+bf|^2  vs  0.01*(|wf|^2+|bf|^2) + 0.5
      const float2 su = add2(a, u), sv = add2(b, v);
      const float2 L = fma2(su, su, mul2(sv, sv));
      const float2 nn = add2(fma2(a, a, mul2(b, b)), s0);
      const float2 Rhi = fma2(f2(0.01f * kHi), nn, f2(0.5f * kHi)), Rlo = fma2(f2(0.01f * kLo), nn, f2(0.5f * kLo));
      const bool occ0 = L.x > Rhi.x, occ1 = L.y > Rhi.y;
      keep0 = keep0 && !occ0; keep1 = keep1 && !occ1;
      amb0 = amb0 || !(occ0 || L.x < Rlo.x); amb1 = amb1 || !(occ1 || L.y < Rlo.y);
    }
    float2 acc = f2(0.0f);
#pragma unroll
    for (int ch = 0; ch < (CT == 3 ? 3 : 0); ++ch) {
      const float2 d = sub2(f2(cur[j0][ch], cur[j1][ch]), w3[ch]);
      // mask*|warp - cur| (MoGAN :281) / (mask*(cur - warp))^2
      acc = LOSS == TCLB200_L1 ? add2(acc, f2(fabsf(d.x), fabsf(d.y))) : fma2(d, d, acc);
    }
    if (MASK == MASK_GIVEN) {   // (m*d)^2 resp. m*|d| summed over channels
      const float2 m = f2(mk[j0], mk[j1]);
      acc = mul2(LOSS == TCLB200_L1 ? m : mul2(m, m), acc);
    }
    e[j0] = acc.x; e[j1] = acc.y;
    keepbits |= ((keep0 ? 1u : 0u) << j0) | ((keep1 ? 1u : 0u) << j1);
    ambbits |= ((amb0 && ok0 ? 1u : 0u) << j0) | ((amb1 && ok1 ? 1u : 0u) << j1);
    // left for the exact replay from global memory below: out-of-box pixels whose test was too close to call (or, dataset
    // mask, every out-of-box pixel)
    if (MIXED) outbits |= (((amb0 || !kFixInLoop) && in0 && !ok0 ? 1u : 0u) << j0) | (((amb1 || !kFixInLoop) && in1 && !ok1 ? 1u : 0u) << j1);
  }
  // rare, divergent: tests too close to call replay the exact sequences (a few pixels per million)
  if (MASK == MASK_COMPUTED && __builtin_expect(ambbits != 0, 0)) {
#pragma unroll
    for (int k = 0; k < P; ++k)
      if ((ambbits >> k) & 1u) {
        const bool kp = exact_keep<Cfg, true>(s_bu, s_ff, c0 + pix_dy(k) * BFW, xf, yf0 + (float)pix_dy(k), lg, box_xf, box_yf);
        keepbits = (keepbits & ~(1u << k)) | ((kp ? 1u : 0u) << k);
      }
  }
  // ... the same for pixels of a mixed tile whose taps left the boxes: redone from global memory
  if (MIXED && __builtin_expect(outbits != 0, 0)) {
    const size_t plane = (size_t)g.H * g.W;
#pragma unroll
    for (int k = 0; k < P; ++k)
      if ((outbits >> k) & 1u) {
        if (CT == 3) {
          e[k] = pixel_global<FrameT, MASK, false, LOSS>(p.bf + (size_t)t.bfi * p.bf_batch, p.bf_plane, MASK == MASK_COMPUTED ? p.ff + (size_t)t.ffi * p.ff_batch : nullptr, p.ff_plane,
                                                         reinterpret_cast<const FrameT*>(p.prev) + (size_t)t.pf * 3 * plane, g, t.x0 + lx0,
                                                         t.y0 + ly0 + pix_dy(k), cur[k][0], cur[k][CT == 3 ? 1 : 0], cur[k][CT == 3 ? 2 : 0], mk[k]);
          keepbits |= 1u << k;   // the verdict is already applied
        } else {
          const float kp = pixel_global<FrameT, MASK, true, LOSS>(p.bf + (size_t)t.bfi * p.bf_batch, p.bf_plane, p.ff + (size_t)t.ffi * p.ff_batch, p.ff_plane, nullptr, g,
                                                                  t.x0 + lx0, t.y0 + ly0 + pix_dy(k), 0.0f, 0.0f, 0.0f, 0.0f);
          keepbits = (keepbits & ~(1u << k)) | ((kp != 0.0f ? 1u : 0u) << k);
        }
      }
  }
  if (CT == 0) {   // mask-only: store the verdicts (two coalesced 64-byte row segments per warp instruction)
    float* mo = p.mask_out + (size_t)t.pair * gplane + (size_t)(t.y0 + ly0) * g.W + (t.x0 + lx0);
#pragma unroll
    for (int k = 0; k < P; ++k)
      if (!EDGE || (xin && 2 * k < rows_in)) __stcs(mo + (ptrdiff_t)pix_dy(k) * g.W, ((keepbits >> k) & 1u) ? 1.0f : 0.0f);
    return 0.0f;
  }
  float err = 0.0f;
#pragma unroll
  for (int k = 0; k < P; ++k) {
    if (MASK == MASK_GIVEN) err = __fadd_rn(err, e[k]);
    else err = ((keepbits >> k) & 1u) ? __fadd_rn(err, e[k]) : err;
  }
  return err;
}

// ---------------------------------------------------------------------------------------------
// TMA-staged, persistent, warp-specialised forward kernel (the hot kernel)
// ---------------------------------------------------------------------------------------------
// One CTA per SM walks tiles of TW x TH pixels (static round robin, or a global counter for long launches).
//
//   producer warp   keeps NB flow tiles and NS source-box sets in flight with TMA:
//       bf tile k   (TW+16) x (TH+2) x 2, 1 px halo (4 columns on the left for the 16-byte TMA alignment), zero-filled
//                   outside the image = the zero padding of flowtools.gradient
//       ff / prev   BW x BH boxes at the origin the scanner's extent dictates, zero-filled outside the image =
//                   grid_sample's padding_mode='zeros'; tiles whose taps do not fit the box are "mixed", tiles with
//                   non-finite / absurd flow are not staged at all (exact predicated global gathers)
//       when the consumers release a tile: folds their 32 * CW partial sums in a fixed order -> one fp64 per tile
//   scanner warp    as soon as a flow tile lands: extent of x+u, y+v over it (LDS.128) -> box[]; runs NS tiles ahead of
//                   the consumers, off everybody's critical path
//   consumer warps  one pass per pixel: flow + 4 neighbours from the flow tile (vertical strips, see WsCfg),
//                   motion-boundary test, sampling position, 4 x (2 + C) taps from the source boxes, occlusion test,
//                   masked error against `cur` (coalesced global loads issued before the wait for the boxes).
template <typename FrameT, int MASK, bool REDUCE, int CT, int LEAN, typename Cfg>
__global__ void __launch_bounds__(Cfg::kThreads, 1) fused_forward_ws_kernel(const FwdParams p, const __grid_constant__ CUtensorMap tm_bf,
                                                                         const __grid_constant__ CUtensorMap tm_ff,
                                                                         const __grid_constant__ CUtensorMap tm_prev,
                                                                         const __grid_constant__ CUtensorMap tm_cur) {
  constexpr int NB = Cfg::NB, NS = Cfg::NS, P = Cfg::kPPL;
  constexpr int kCWarps = Cfg::CW;
  constexpr int kLoss = LEAN == 2 ? TCLB200_L1 : TCLB200_L2;
  // interior / edge / mixed staged tiles of the reducing hot configurations: packed fp32 arithmetic (lean_tile_packed)
  // ... and fbcCheckTorch on its own (mask_out only)
  constexpr bool kPacked = TCL_PACKED && (((LEAN == 1 || LEAN == 2) && CT == 3 && (MASK == MASK_COMPUTED || (MASK == MASK_GIVEN && TCL_PACKED_GIVEN))) ||
                                          (TCL_PACKED_MASK && LEAN == 1 && CT == 0 && MASK == MASK_COMPUTED && !REDUCE));
  using Ctl = WsCtl<NB, NS, kCWarps>;
  static_assert(sizeof(Ctl) <= Cfg::kCtlBytes, "control block too large");
  extern __shared__ __align__(128) unsigned char smem_raw[];
  unsigned char* smem = smem_raw + ((128u - (smem_u32(smem_raw) & 127u)) & 127u);  // TMA destinations: 128-byte aligned
  Ctl* ctl = reinterpret_cast<Ctl*>(smem + Cfg::kCtlOff);
  auto bf_stage = [&](int s) { return reinterpret_cast<float*>(smem + Cfg::kBfOff + (size_t)s * Cfg::kBfStage); };
  auto ff_stage = [&](int s) { return reinterpret_cast<float*>(smem + Cfg::kSrcOff + (size_t)s * Cfg::kSrcStage); };
  auto prev_stage = [&](int s) { return reinterpret_cast<FrameT*>(smem + Cfg::kSrcOff + (size_t)s * Cfg::kSrcStage + Cfg::kFfStage); };

  const int total_tiles = p.B * p.tiles_per_pair;
  // LEAN: 1 = both mask tests / L2, 2 = both mask tests / L1, 3 = mask-only with the motion-boundary test alone,
  //       4 = as 1 plus the optional per-pixel outputs (warp_out / mask_out / blend_out, whichever are set)
  const bool want_occ = MASK == MASK_COMPUTED && (LEAN ? LEAN != 3 : (p.flags & TCLB200_OCC) != 0);
  const bool want_frames = CT > 0 && (LEAN || p.prev != nullptr);
  const bool want_scan = want_occ || want_frames;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const Geo& g = p.geo;
  // Local tile k of this CTA lives in flow stage k % NB / source stage k % NS.  Which tile that is, is decided when its
  // flow tile is requested: static round robin for short launches, a global atomic counter for long ones, so that all
  // CTAs stay within a few tiles of each other and the overlapping halos of neighbouring boxes still hit in L2 (with a
  // static schedule the CTAs drift apart over ~1000 tiles and the overlaps are re-read from HBM: +21 % traffic measured).
  // The entry after a CTA's last tile carries pair = -1.
  auto real = [&](int k) { return ctl->tinfo[k % NB].pair >= 0; };

  if (REDUCE) asm volatile("griddepcontrol.launch_dependents;" ::: "memory");   // let the fold kernel get resident early
  if (threadIdx.x == 0) {
    for (int i = 0; i < NB; ++i) { mbar_init(&ctl->bf_full[i], 1); mbar_init(&ctl->scanned[i], 1); }
    for (int i = 0; i < NS; ++i) { mbar_init(&ctl->src_full[i], 1); mbar_init(&ctl->done[i], kCWarps); }
    fence_barrier_init();
  }
  __syncthreads();

  if (warp == Cfg::kProducerWarp) {
    // ===================================== producer warp =====================================
    // lane 0 only: next tile of this CTA (prefetched one call ahead so the atomic's latency is off the critical path)
    const bool dynamic = p.scratch.tile_ctr != nullptr;
    int tg_next = (int)blockIdx.x;
    bool exhausted = false;
    auto next_tile = [&]() {
      const int tg = tg_next;
      tg_next = dynamic ? (int)gridDim.x + (int)atomicAdd(p.scratch.tile_ctr, 1u) : tg + (int)gridDim.x;
      return tg;
    };
    auto issue_bf = [&](int k) {   // lane 0: describe local tile k, request its flow tile (or mark the end)
      const int s = k % NB;
      const int tg = exhausted ? total_tiles : next_tile();
      if (tg >= total_tiles) {
        exhausted = true;
        ctl->tinfo[s].pair = -1;
        mbar_arrive(&ctl->bf_full[s]);
        return;
      }
      const TileId t = tile_id(p, tg, Cfg::TW, Cfg::TH);
      ctl->tinfo[s] = t;
      mbar_expect_tx(&ctl->bf_full[s], Cfg::kBfLoad);
      tma_load_4d(bf_stage(s), &tm_bf, &ctl->bf_full[s], t.x0 - Cfg::kHaloL, t.y0 - 1, 0, t.bfi);
      // the consumers read this tile's `cur` values straight from global memory NB tiles from now: have them in L2 by then
      if (LEAN && CT > 0 && p.cur != nullptr) tma_prefetch_l2_4d(&tm_cur, t.x0, t.y0, 0, t.cf);
    };
    // lane 0: the scanner has left the extent of x+u, y+v over local tile k in box[k % NB] -> origin of the source
    // boxes.  The coordinate map is monotone in x+u (every step is a correctly rounded monotone operation), so the
    // extreme taps come from the extreme sums.
    struct Placement { int ox, oy, mode, ffi, pf; };
    auto place_src = [&](int k) -> Placement {
      const int sb = k % NB;
      const TileId t = ctl->tinfo[sb];
      int ox = 0, oy = 0, mode = 0;   // mode: 0 = nothing staged, 1 = every tap inside the boxes, 2 = mixed
#if TCL_DIAG == 3   // tuning aid: boxes at the tile's own position, no scan (results are garbage)
      if (true) { ox = (t.x0 - 8) & ~3; oy = t.y0 - 4; mode = 1; } else
#endif
      if (want_scan) {
        mbar_wait_idle(&ctl->scanned[sb], (k / NB) & 1);
        const float xmin = ord2f(ctl->box[sb][0]), ymin = ord2f(ctl->box[sb][1]), xmax = ord2f(ctl->box[sb][2]), ymax = ord2f(ctl->box[sb][3]);
        const float lim = 30000.0f;   // (keeps the consumers' floating-point box addresses exact, see lean_tile)
        const bool sane = xmin > -lim && xmax < lim && ymin > -lim && ymax < lim && xmin <= xmax && ymin <= ymax;   // false for NaN / Inf
        if (sane) {
          const float i2x = __fmul_rn(2.0f, g.inv_dx), i2y = __fmul_rn(2.0f, g.inv_dy);
          auto coord = [](float a, float i2, float sz) {
            const float tt = __fadd_rn(__fsub_rn(__fmul_rn(a, i2), 1.0f), 1.0f);
            return __fmul_rn(__fmaf_rn(tt, sz, -1.0f), 0.5f);
          };
          const int bx0 = __float2int_rd(coord(xmin, i2x, g.Wf)), bx1 = __float2int_rd(coord(xmax, i2x, g.Wf));
          const int by0 = __float2int_rd(coord(ymin, i2y, g.Hf)), by1 = __float2int_rd(coord(ymax, i2y, g.Hf));
          ox = bx0 & ~(Cfg::kXAlign - 1);   // 16-byte aligned box start (floor, also for negatives)
          oy = by0;
          // taps span [x0, x0+1] x [y0, y0+1]
          const bool fitx = bx1 + 1 - ox < Cfg::BW, fity = by1 + 1 - oy < Cfg::BH;
          mode = (fitx && fity) ? 1 : 2;
          if (mode == 2) {
            // a motion boundary runs through the tile: centre the box on the extent (per axis, where it does not fit);
            // pixels whose taps fall outside take the global path one by one
            if (!fitx) ox = ((bx0 + bx1 + 1 - Cfg::BW) / 2) & ~(Cfg::kXAlign - 1);
            if (!fity) oy = (by0 + by1 + 1 - Cfg::BH) / 2;
          }
        }
        if (mode != 1) atomicAdd(&g_tile_stats[mode == 2 ? 1 : 0], 1ull);
      }
      return Placement{ox, oy, mode, t.ffi, t.pf};
    };
    // ... and, once the source stage is free, the request itself (lane 0)
    auto issue_src = [&](int k, const Placement& pl) {
      const int ss = k % NS;
      ctl->meta[ss][0] = pl.ox; ctl->meta[ss][1] = pl.oy; ctl->meta[ss][2] = pl.mode;
#if TCL_DIAG == 1   // tuning aid: no source-box traffic at all (results are garbage)
      if (false) {
#else
      if (pl.mode != 0) {
#endif
        TCL_STAMP(k, 0);
        mbar_expect_tx(&ctl->src_full[ss], (want_occ ? Cfg::kFfLoad : 0u) + (want_frames ? Cfg::kPrevLoad : 0u));
        if (want_occ) tma_load_4d(ff_stage(ss), &tm_ff, &ctl->src_full[ss], pl.ox, pl.oy, 0, pl.ffi);
        if (want_frames) tma_load_4d(prev_stage(ss), &tm_prev, &ctl->src_full[ss], pl.ox, pl.oy, 0, pl.pf);
      } else {
        mbar_arrive(&ctl->src_full[ss]);
      }
    };

    if (lane == 0) {
      prefetch_tmap(&tm_bf);
      if (want_occ) prefetch_tmap(&tm_ff);
      if (want_frames) prefetch_tmap(&tm_prev);
      for (int j = 0; j < NB; ++j) issue_bf(j);
      for (int j = 0; j < NS && real(j); ++j) issue_src(j, place_src(j));
    }
    __syncwarp();
    for (int j = 0; real(j); ++j) {
      mbar_wait_idle(&ctl->done[j % NS], (j / NS) & 1);   // consumers are finished with tile j: its stages are free
      const TileId t = ctl->tinfo[j % NB];   // (before issue_bf recycles the slot)
      // every consumer lane's sum of this tile: lane l folds the warps' lanes l in warp order (fp64 from here on)
      double ts = 0.0;
      if (REDUCE) {
        const float* r = ctl->red[j % NS] + lane;
#pragma unroll
        for (int w = 0; w < kCWarps; ++w) ts += (double)r[32 * w];
      }
      __syncwarp();   // (all of red[] is in registers before the stage is handed out again)
      if (lane == 0) {
        if (real(j + NS)) issue_src(j + NS, place_src(j + NS));
        issue_bf(j + NB);
      }
      __syncwarp();
      // ... then the lanes in a fixed butterfly: one fp64 partial per tile, independent of the tile schedule
      if (REDUCE) {
        ts = warp_sum(ts);
        if (lane == 0) __stcg(&p.scratch.partials[(size_t)t.pair * p.tiles_per_pair + t.tile], ts);
      }
    }
    // long launches: the last CTA to run out of tiles re-arms the tile counter for the next launch
    if (dynamic && lane == 0) {
      __threadfence();
      if (atomicAdd(p.scratch.tile_ctr + 1, 1u) == gridDim.x - 1) {
        p.scratch.tile_ctr[0] = 0;
        p.scratch.tile_ctr[1] = 0;
      }
    }
    return;
  }

  if (warp >= Cfg::kScannerWarp) {
    // ===================================== scanner warps =====================================
    if (!want_scan || TCL_DIAG == 3) return;
    for (int k = warp - Cfg::kScannerWarp;; k += Cfg::kScanners) {
      const int sb = k % NB;
      mbar_wait_idle(&ctl->bf_full[sb], (k / NB) & 1);
      if (ctl->tinfo[sb].pair < 0) return;
      scan_flow_tile<Cfg>(bf_stage(sb), ctl->tinfo[sb], g, p.row_end, ctl->box[sb], lane);
      __syncwarp();
      if (lane == 0) mbar_arrive(&ctl->scanned[sb]);
    }
  }

  // ======================================= consumer warps =======================================
  unsigned near = 0;
  const size_t plane = (size_t)g.H * g.W;
  int lx0, ly0;
  lane_origin<Cfg>(warp, lane, lx0, ly0);
  const int lane_off = ly0 * g.W + lx0;
  // shared-memory addresses the loop needs every tile, computed once (the empty asm keeps the compiler from
  // re-deriving them from the generic pointers inside the loop)
  uint32_t bf_full_s = smem_u32(&ctl->bf_full[0]), src_full_s = smem_u32(&ctl->src_full[0]), done_s = smem_u32(&ctl->done[0]);
  uint32_t red_s = smem_u32(&ctl->red[0][threadIdx.x]);
  asm volatile("" : "+r"(bf_full_s), "+r"(src_full_s), "+r"(done_s), "+r"(red_s));
  const bool have_cur = CT > 0 && (LEAN ? MASK != MASK_NONE : p.cur != nullptr);   // (the LEAN configurations fix it at compile time)
  for (int k = 0;; ++k) {
    float err = 0.0f;
    const int sb = k % NB, ss = k % NS;   // stage indices of this tile
    mbar_wait_s(bf_full_s + 8u * sb, (k / NB) & 1);
    // (a reference into shared memory, not a register copy: the fields only the rare paths need -- pf, bfi, ffi -- are read
    // there; the slot is rewritten only after this warp has arrived on done[] for the tile)
    const TileId& t = ctl->tinfo[sb];
    if (t.pair < 0) break;
    const bool t_edge = tile_edge<Cfg>(t, g, p.row_end);
    // this tile's `cur` (and dataset mask) values: coalesced 64-byte row segments, streaming; requested before the wait
    // for the source boxes and first used at the very end of the per-pixel work
    float cur[P][Cfg::kC], mk[P];
    {
      const size_t pix = (size_t)(t.y0 * g.W + t.x0) + lane_off;
      const FrameT* cb = reinterpret_cast<const FrameT*>(p.cur) + (size_t)t.cf * Cfg::kC * plane + pix;
      const float* mb = MASK == MASK_GIVEN ? p.mask_in + (size_t)t.pair * plane + pix : nullptr;
      if (!t_edge && p.cur_index != nullptr) {
        // clip mode: this frame is read again as the `prev` of the next pair -- do not mark its lines evict-first
#pragma unroll
        for (int c = 0; c < Cfg::kC; ++c) {
          const FrameT* pc = cb + (size_t)c * plane;
#pragma unroll
          for (int i = 0; i < P; ++i) cur[i][c] = have_cur ? to_f32(__ldg(pc + (ptrdiff_t)pix_dy(i) * g.W)) : 0.0f;
        }
#pragma unroll
        for (int i = 0; i < P; ++i) mk[i] = MASK == MASK_GIVEN ? __ldcs(mb + (ptrdiff_t)pix_dy(i) * g.W) : 0.0f;
      } else if (!t_edge) {
#pragma unroll
        for (int c = 0; c < Cfg::kC; ++c) {
          const FrameT* pc = cb + (size_t)c * plane;
#pragma unroll
          for (int i = 0; i < P; ++i) cur[i][c] = have_cur ? ld_stream(pc + (ptrdiff_t)pix_dy(i) * g.W) : 0.0f;
        }
#pragma unroll
        for (int i = 0; i < P; ++i) mk[i] = MASK == MASK_GIVEN ? __ldcs(mb + (ptrdiff_t)pix_dy(i) * g.W) : 0.0f;
      } else {
#pragma unroll
        for (int i = 0; i < P; ++i) {
          const bool inside = t.x0 + lx0 < g.W && t.y0 + ly0 + pix_dy(i) < p.row_end;
          const ptrdiff_t off = (ptrdiff_t)pix_dy(i) * g.W;
#pragma unroll
          for (int c = 0; c < Cfg::kC; ++c) cur[i][c] = (have_cur && inside) ? ld_stream(cb + off + (size_t)c * plane) : 0.0f;
          mk[i] = (MASK == MASK_GIVEN && inside) ? __ldcs(mb + off) : 0.0f;
        }
      }
    }
    if (threadIdx.x == 0) TCL_STAMP(k, 1);
    mbar_wait_s(src_full_s + 8u * ss, (k / NS) & 1);
    if (threadIdx.x == 0) TCL_STAMP(k, 2);
#if TCL_DIAG == 1
    const int mode = 1;
#else
    const int mode = ctl->meta[ss][2];
#endif
    if (LEAN == 3) {   // nothing staged, nothing sampled: the flow tile alone decides
      if (t_edge) lean_tile<FrameT, MASK, CT, TCLB200_L2, Cfg, true, false, false>(p, bf_stage(sb), ff_stage(ss), ctl->meta[ss], t, lx0, ly0, cur, mk);
      else lean_tile<FrameT, MASK, CT, TCLB200_L2, Cfg, false, false, false>(p, bf_stage(sb), ff_stage(ss), ctl->meta[ss], t, lx0, ly0, cur, mk);
    } else if (LEAN && mode == 1) {
      if constexpr (kPacked) {
        if (t_edge) err = lean_tile_packed<FrameT, MASK, kLoss, Cfg, true, false, CT>(p, bf_stage(sb), ff_stage(ss), ctl->meta[ss], t, lx0, ly0, cur, mk);
        else err = lean_tile_packed<FrameT, MASK, kLoss, Cfg, false, false, CT>(p, bf_stage(sb), ff_stage(ss), ctl->meta[ss], t, lx0, ly0, cur, mk);
      } else {
        if (t_edge) err = lean_tile<FrameT, MASK, CT, kLoss, Cfg, true, false, true, LEAN == 4>(p, bf_stage(sb), ff_stage(ss), ctl->meta[ss], t, lx0, ly0, cur, mk);
        else err = lean_tile<FrameT, MASK, CT, kLoss, Cfg, false, false, true, LEAN == 4>(p, bf_stage(sb), ff_stage(ss), ctl->meta[ss], t, lx0, ly0, cur, mk);
      }
    } else if (LEAN == 4) {   // outputs wanted and the tile is mixed / unstaged: the feature-complete exact path
      err = full_tile<FrameT, MASK, REDUCE, CT, 0, Cfg, true>(p, bf_stage(sb), ff_stage(ss), prev_stage(ss), ctl->meta[ss], t, lx0, ly0, cur, mk, have_cur, near);
    } else if (LEAN && mode == 2) {
      if constexpr (kPacked) err = lean_tile_packed<FrameT, MASK, kLoss, Cfg, true, true, CT>(p, bf_stage(sb), ff_stage(ss), ctl->meta[ss], t, lx0, ly0, cur, mk);
      else err = lean_tile<FrameT, MASK, CT, kLoss, Cfg, true, true>(p, bf_stage(sb), ff_stage(ss), ctl->meta[ss], t, lx0, ly0, cur, mk);
    } else if (LEAN || t_edge) {
      err = full_tile<FrameT, MASK, REDUCE, CT, LEAN, Cfg, true>(p, bf_stage(sb), ff_stage(ss), prev_stage(ss), ctl->meta[ss], t, lx0, ly0, cur, mk, have_cur, near);
    } else {
      err = full_tile<FrameT, MASK, REDUCE, CT, LEAN, Cfg, false>(p, bf_stage(sb), ff_stage(ss), prev_stage(ss), ctl->meta[ss], t, lx0, ly0, cur, mk, have_cur, near);
    }
    // <= 3 * P fp32 terms per lane; the producer folds the lanes (fixed order, fp64)
    if (REDUCE) asm volatile("st.shared.f32 [%0], %1;" ::"r"(red_s + (uint32_t)(ss * kCWarps * 128)), "f"(err) : "memory");
    __syncwarp();   // every lane is done reading the stages of tile k
    if (lane == 0) mbar_arrive_s(done_s + 8u * ss);
    if (threadIdx.x == 0) TCL_STAMP(k, 3);
  }
  if (!LEAN) count_near(near, p.near_threshold);
}

// ---------------------------------------------------------------------------------------------
// gradient(x): zero-padded central differences (flowtools.py:12-16); one pixel per lane, coalesced
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads) gradient_kernel(const float* __restrict__ xin, size_t in_stride, float* __restrict__ out, int B, int H,
                                                            int W, int tiles_x, int tiles_per_img) {
  const size_t plane = (size_t)H * W;
  const int lane = threadIdx.x & 31, wrp = threadIdx.x >> 5;
  const int img = blockIdx.x / tiles_per_img;
  const int tile = blockIdx.x - img * tiles_per_img;
  const int ty = tile / tiles_x, tx = tile - ty * tiles_x;
  const int x = tx * 32 + lane, y = ty * kWarps + wrp;
  if (x >= W || y >= H) return;
  const float* src = xin + (size_t)img * in_stride;
  const size_t o = (size_t)y * W + x;
  const float l = x > 0 ? __ldg(src + o - 1) : 0.0f, r = x + 1 < W ? __ldg(src + o + 1) : 0.0f;
  const float up = y > 0 ? __ldg(src + o - W) : 0.0f, dn = y + 1 < H ? __ldg(src + o + W) : 0.0f;
  __stcs(out + (size_t)img * plane + o, __fmul_rn(__fsub_rn(r, l), 0.5f));
  __stcs(out + ((size_t)B + img) * plane + o, __fmul_rn(__fsub_rn(dn, up), 0.5f));
}

// W % 4 == 0 and 16-byte aligned planes: four pixels per lane.  The centre row's float4 gives every x-difference but
// the two that reach into the neighbouring lanes' quads (warp shuffles; one scalar load at a warp's ends), the rows
// above / below are two more float4 loads (the three reads of a row are L1 / L2 hits); two float4 stores.
// 4 B/px read + 8 B/px written, all 16-byte accesses.
__global__ void __launch_bounds__(kThreads) gradient_vec4_kernel(const float* __restrict__ xin, size_t in_stride, float* __restrict__ out, int B, int H,
                                                                 int W, int tiles_x, int tiles_per_img) {
  const size_t plane = (size_t)H * W;
  const int lane = threadIdx.x & 31, wrp = threadIdx.x >> 5;
  const int img = blockIdx.x / tiles_per_img;
  const int tile = blockIdx.x - img * tiles_per_img;
  const int ty = tile / tiles_x, tx = tile - ty * tiles_x;
  const int x = tx * 128 + 4 * lane, y = ty * kWarps + wrp;   // warp = one 128-pixel row segment
  if (y >= H) return;
  const bool in = x < W;
  const float* src = xin + (size_t)img * in_stride;
  const size_t o = (size_t)y * W + x;
  const float4 z = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
  const float4 c = in ? __ldg(reinterpret_cast<const float4*>(src + o)) : z;
  const float4 up = (in && y > 0) ? __ldg(reinterpret_cast<const float4*>(src + o - W)) : z;
  const float4 dn = (in && y + 1 < H) ? __ldg(reinterpret_cast<const float4*>(src + o + W)) : z;
  float l = __shfl_up_sync(0xffffffffu, c.w, 1), r = __shfl_down_sync(0xffffffffu, c.x, 1);
  if (lane == 0) l = (in && x > 0) ? __ldg(src + o - 1) : 0.0f;
  if (lane == 31) r = (in && x + 4 < W) ? __ldg(src + o + 4) : 0.0f;
  if (in && x + 4 >= W) r = 0.0f;   // the lane right of the image edge holds zeros anyway; explicit for clarity
  if (!in) return;
  float4 dx, dy;
  dx.x = __fmul_rn(__fsub_rn(c.y, l), 0.5f);   dx.y = __fmul_rn(__fsub_rn(c.z, c.x), 0.5f);
  dx.z = __fmul_rn(__fsub_rn(c.w, c.y), 0.5f); dx.w = __fmul_rn(__fsub_rn(r, c.z), 0.5f);
  dy.x = __fmul_rn(__fsub_rn(dn.x, up.x), 0.5f); dy.y = __fmul_rn(__fsub_rn(dn.y, up.y), 0.5f);
  dy.z = __fmul_rn(__fsub_rn(dn.z, up.z), 0.5f); dy.w = __fmul_rn(__fsub_rn(dn.w, up.w), 0.5f);
  __stcs(reinterpret_cast<float4*>(out + (size_t)img * plane + o), dx);
  __stcs(reinterpret_cast<float4*>(out + ((size_t)B + img) * plane + o), dy);
}

// ---------------------------------------------------------------------------------------------
// backward kernels.  One lane per target pixel; grad_prev is a bilinear scatter-add (red.global.add.f32).
// Frames (x / prev, cur, grad_out, grad_cur) are fp32 or bf16; flows, masks and the scatter target are always fp32.
// ---------------------------------------------------------------------------------------------
struct BwdParams {
  const void* grad_out;    // warp_backward: (B,C,H,W) frame dtype; tcl_backward: unused
  const void* x;           // source frame (prev), frame dtype
  const float* f;          // flow
  const float* mask;       // tcl_backward only
  const void* cur;         // tcl_backward only, frame dtype
  const float* grad_scale; // tcl_backward only (device scalar)
  float scale_mul;         // tcl_backward only: host factor applied to *grad_scale (1/(B*C*H*W) for the mean loss)
  float* grad_x;           // fp32 frames: the output itself; bf16 frames: the fp32 accumulator (workspace) it is rounded from
  float* grad_f;
  void* grad_cur;          // frame dtype
  Geo geo;
  int B, C, flags, loss;
};

// Where the time goes (64 Sintel-shape pairs, memset + kernel 527 us = 54 Gpix/s): the real DRAM traffic is 84 B/px
// (36 inputs + 12 read-for-ownership of the scatter target + 24 written + 12 for the zero-fill), i.e. 4.5 TB/s = 0.69 of
// the measured copy peak with reads and writes mixed.  Measured and dropped, none of them moved that number:
//   - 2 / 4 pixels per lane (all flow-independent loads first, then all gathers): 43 / 19-26 Gpix/s (registers, occupancy)
//   - warp-aggregated scatter (lane l adds lane l-1's right-hand taps to its own `red` where the flow is locally uniform,
//     halving the atomics): 53.9 Gpix/s, no change -- the `red` drain is not the limit
//   - the batch in L2-sized slices (memset of a slice, then its kernel) so that the `red`s find zeroed lines resident:
//     556 / 573 / 614 / 712 us with 96 / 64 / 32 / 16 MB slices -- the tails between the short kernels cost more
// FUSED_LOSS: the upstream gradient of warp is derived in-kernel from the masked loss.
// CT > 0 fixes the channel count at compile time: all 4*CT gathers and the CT `cur` / grad_out loads of a pixel are then
// issued back to back (the kernel is latency-bound otherwise: measured 10 long-scoreboard stall cycles per issue).
// FrameT = __nv_bfloat16: frame loads are converted to fp32 and the arithmetic is the fp32 kernel's, so grad_f and the
// fp32 grad_cur are bit for bit those of the fp32 kernel on the upcast frames; grad_cur is rounded once on the store.
// grad_x goes to an fp32 accumulator (red.add.bf16x2 would round on every add) that bwd_acc_to_bf16_kernel rounds behind.
template <bool FUSED_LOSS, int CT, typename FrameT>
#ifndef TCL_BWD_MINB
#define TCL_BWD_MINB 5   // measured: 5 CTAs per SM (48 registers) beats 4 (59) and 6 (40, spills)
#endif
__global__ void __launch_bounds__(256, TCL_BWD_MINB) warp_backward_kernel(const BwdParams p) {
  if constexpr (sizeof(FrameT) == 2) asm volatile("griddepcontrol.launch_dependents;" ::: "memory");   // the bf16 rounding kernel
  const Geo& g = p.geo;
  const FrameT* const frame_x = static_cast<const FrameT*>(p.x);
  const FrameT* const frame_in = static_cast<const FrameT*>(FUSED_LOSS ? p.cur : p.grad_out);
  FrameT* const frame_gc = static_cast<FrameT*>(p.grad_cur);
  const int W = g.W, H = g.H, C = CT > 0 ? CT : p.C;
  const size_t plane = (size_t)H * W;
  // 32 x 8 pixel tiles: lanes along x (coalesced loads / stores, neighbouring lanes scatter into neighbouring addresses)
  const int lane = threadIdx.x & 31, wrp = threadIdx.x >> 5;
  const int b = blockIdx.z;
  const int x = blockIdx.x * 32 + lane, y = blockIdx.y * 8 + wrp;
  if (x >= W || y >= H) return;
  const size_t o = (size_t)y * W + x;
  const float u = __ldg(p.f + (size_t)b * 2 * plane + o), v = __ldg(p.f + ((size_t)b * 2 + 1) * plane + o);

  // taps, with the un-multiplied fractional parts kept for the coordinate gradient
  const float ix = source_coord(x, u, g.Wf, g.dxf, g.inv_dx, kV);
  const float iy = source_coord(y, v, g.Hf, g.dyf, g.inv_dy, kV);
  const int x0 = __float2int_rd(ix), y0 = __float2int_rd(iy);
  const int x1 = (int)((unsigned)x0 + 1u), y1 = (int)((unsigned)y0 + 1u);
  const float fx1 = (float)x1 - ix, fx0 = ix - (float)x0, fy1 = (float)y1 - iy, fy0 = iy - (float)y0;
  const float nw = fx1 * fy1, ne = fx0 * fy1, sw = fx1 * fy0, se = fx0 * fy0;
  const bool xin0 = (unsigned)x0 < (unsigned)W, xin1 = (unsigned)x1 < (unsigned)W;
  const bool yin0 = (unsigned)y0 < (unsigned)H, yin1 = (unsigned)y1 < (unsigned)H;
  const bool p00 = xin0 && yin0, p10 = xin1 && yin0, p01 = xin0 && yin1, p11 = xin1 && yin1;
  const long long o00 = (long long)y0 * W + x0;

  float valid = 1.0f;
  if (p.flags & TCLB200_VALIDITY) {
    Taps t; t.p00 = p00; t.p10 = p10; t.p01 = p01; t.p11 = p11; t.nw = nw; t.ne = ne; t.sw = sw; t.se = se; t.o00 = 0;
    valid = binarise_validity(ones_sample(t, kV));
  }
  float m = 1.0f, scale = 1.0f;
  if (FUSED_LOSS) {
    m = p.mask ? __ldg(p.mask + (size_t)b * plane + o) : 1.0f;
    scale = __fmul_rn(__ldg(p.grad_scale), p.scale_mul);   // (exactly torch's fp32 `grad_out * (1/N)` when the host factor is that)
  }
  const bool need_taps = FUSED_LOSS || p.grad_f != nullptr;   // the source values themselves are only needed for these

  constexpr int CU = CT > 0 ? CT : 1;
  float gix = 0.0f, giy = 0.0f;
  auto channel = [&](int c, float v00, float v10, float v01, float v11, float in) {
    const size_t base = ((size_t)b * C + c) * plane;
    float go;  // d loss / d warp[b,c,y,x]
    if (FUSED_LOSS) {
      float wv = 0.0f;
      if (p00) wv = fmaf(v00, nw, wv);
      if (p10) wv = fmaf(v10, ne, wv);
      if (p01) wv = fmaf(v01, sw, wv);
      if (p11) wv = fmaf(v11, se, wv);
      wv *= valid;
      float gc;  // d loss / d cur
      if (p.loss == TCLB200_L2) {
        gc = 2.0f * scale * m * m * (in - wv);
      } else {
        const float d = wv - in;
        gc = -scale * m * (d > 0.0f ? 1.0f : (d < 0.0f ? -1.0f : 0.0f));
      }
      if (frame_gc) st_stream(frame_gc + base + o, gc);
      go = -gc;
    } else {
      go = in;
    }
    go *= valid;
    if (p.grad_x) {
      float* gp = p.grad_x + base;
      if (p00) atomicAdd(gp + o00, nw * go);
      if (p10) atomicAdd(gp + o00 + 1, ne * go);
      if (p01) atomicAdd(gp + o00 + W, sw * go);
      if (p11) atomicAdd(gp + o00 + W + 1, se * go);
    }
    if (p.grad_f) {
      gix += go * ((v10 - v00) * fy1 + (v11 - v01) * fy0);
      giy += go * ((v01 - v00) * fx1 + (v11 - v10) * fx0);
    }
  };
  if (CT > 0) {
    float v00[CU], v10[CU], v01[CU], v11[CU], in[CU];
#pragma unroll
    for (int c = 0; c < CU; ++c) {   // every load of this pixel in flight before the first use
      const size_t base = ((size_t)b * C + c) * plane;
      const FrameT* xp = frame_x + base;
      v00[c] = (need_taps && p00) ? ld_gather(xp + o00) : 0.0f;
      v10[c] = (need_taps && p10) ? ld_gather(xp + o00 + 1) : 0.0f;
      v01[c] = (need_taps && p01) ? ld_gather(xp + o00 + W) : 0.0f;
      v11[c] = (need_taps && p11) ? ld_gather(xp + o00 + W + 1) : 0.0f;
      in[c] = ld_stream(frame_in + base + o);
    }
#pragma unroll
    for (int c = 0; c < CU; ++c) channel(c, v00[c], v10[c], v01[c], v11[c], in[c]);
  } else {
    for (int c = 0; c < C; ++c) {
      const size_t base = ((size_t)b * C + c) * plane;
      const FrameT* xp = frame_x + base;
      const float a00 = (need_taps && p00) ? ld_gather(xp + o00) : 0.0f, a10 = (need_taps && p10) ? ld_gather(xp + o00 + 1) : 0.0f;
      const float a01 = (need_taps && p01) ? ld_gather(xp + o00 + W) : 0.0f, a11 = (need_taps && p11) ? ld_gather(xp + o00 + W + 1) : 0.0f;
      channel(c, a00, a10, a01, a11, ld_stream(frame_in + base + o));
    }
  }
  if (p.grad_f) {
    // d ix/d gx = W/2 (grid_sampler), d gx/d u = 2/(W-1) (flowtools.py:28)
    p.grad_f[(size_t)b * 2 * plane + o] = 2.0f * (g.Wf * 0.5f * gix) / g.dxf;
    p.grad_f[((size_t)b * 2 + 1) * plane + o] = 2.0f * (g.Hf * 0.5f * giy) / g.dyf;
  }
}

// grad_x of bf16 frames: the fp32 accumulator the scatter-add left, rounded once (__float2bfloat16_rn, what torch's
// .to(torch.bfloat16) does).  Launched behind warp_backward_kernel with programmatic dependent launch.  Four values per
// lane: one 16-byte load, one 8-byte store (vec = the output is 8-byte aligned; the accumulator always is 16-byte aligned).
__global__ void __launch_bounds__(kThreads) bwd_acc_to_bf16_kernel(const float* __restrict__ acc, __nv_bfloat16* __restrict__ out,
                                                                   size_t n, int vec) {
  asm volatile("griddepcontrol.wait;" ::: "memory");   // every red of the scatter has landed after this
  const size_t i = ((size_t)blockIdx.x * kThreads + threadIdx.x) * 4;
  if (i >= n) return;
  if (vec && i + 4 <= n) {
    const float4 v = __ldcs(reinterpret_cast<const float4*>(acc + i));
    const __nv_bfloat162 lo = __floats2bfloat162_rn(v.x, v.y), hi = __floats2bfloat162_rn(v.z, v.w);
    uint2 w;
    w.x = *reinterpret_cast<const unsigned*>(&lo);
    w.y = *reinterpret_cast<const unsigned*>(&hi);
    __stcs(reinterpret_cast<uint2*>(out + i), w);
  } else {
    for (size_t k = i; k < n && k < i + 4; ++k) st_stream(out + k, __ldcs(acc + k));
  }
}

// ---------------------------------------------------------------------------------------------
// dataset ingest: HWC -> planar NCHW de-interleave (the 9-channel FC2 / Hollywood2 .npy blocks and .flo payloads)
// ---------------------------------------------------------------------------------------------
// A CTA moves kSplitPx consecutive pixels of one sample: the interleaved floats are read as one contiguous, fully
// coalesced run into shared memory (pitch Cs | 1 words per pixel: conflict-free for any Cs), then every requested
// channel is written as a coalesced run of its destination plane.  Pure data movement: 4*Cs B/px read, 4*sum(Cd) written.
constexpr int kSplitPx = 256;
constexpr int kSplitMaxOut = 8;
struct SplitParams {
  const float* src;
  float* dst[kSplitMaxOut];
  int c0[kSplitMaxOut], cd[kSplitMaxOut];
  int n_out, Cs;
  long long plane;       // H * W
  int chunks_per_sample; // ceil(plane / kSplitPx)
};

__global__ void __launch_bounds__(kSplitPx) hwc_split_kernel(const SplitParams p) {
  extern __shared__ float s_px[];
  const int Cs = p.Cs, pitch = Cs | 1;
  const int n = blockIdx.x / p.chunks_per_sample;
  const long long px0 = (long long)(blockIdx.x - n * p.chunks_per_sample) * kSplitPx;
  const int npx = (int)min((long long)kSplitPx, p.plane - px0);
  const float* src = p.src + ((long long)n * p.plane + px0) * Cs;
  const int nfl = npx * Cs;
  for (int i = threadIdx.x; i < nfl; i += kSplitPx) {
    const int px = i / Cs, c = i - px * Cs;
    s_px[px * pitch + c] = __ldcs(src + i);
  }
  __syncthreads();
  const int t = threadIdx.x;
  if (t >= npx) return;
  for (int o = 0; o < p.n_out; ++o) {
    float* dst = p.dst[o] + (long long)n * p.cd[o] * p.plane + px0 + t;
    for (int c = 0; c < p.cd[o]; ++c) __stcs(dst + (long long)c * p.plane, s_px[t * pitch + p.c0[o] + c]);
  }
}

// Two interleaved channels (the .flo payload, utils/flowlib.py:33-48: u0 v0 u1 v1 ...): no staging needed.  A lane loads one
// float4 = two pixels (a warp: 512 contiguous bytes) and stores one float2 per plane (256 contiguous bytes each); four
// independent loads per lane are in flight before the first store.  8 B/px read, 8 B/px written.
struct Split2Params {
  const float* src;
  float* dst[2];            // plane of channel 0 / 1 of sample 0 (nullptr: channel not requested)
  long long dstride[2];     // elements between consecutive samples of that destination
  long long plane;          // H * W, even
  long long pairs;          // N * plane / 2 pixel pairs in all
};
__global__ void __launch_bounds__(256) hwc2_split_kernel(const Split2Params p) {
  constexpr int K = 4;
  const long long half = p.plane / 2;
  long long i = ((long long)blockIdx.x * K) * 256 + threadIdx.x;
  float4 v[K];
#pragma unroll
  for (int k = 0; k < K; ++k)
    if (i + k * 256 < p.pairs) v[k] = __ldcs(reinterpret_cast<const float4*>(p.src) + i + k * 256);
#pragma unroll
  for (int k = 0; k < K; ++k) {
    const long long j = i + k * 256;
    if (j >= p.pairs) break;
    const long long n = j / half, q = j - n * half;   // sample, pixel pair within its plane
    if (p.dst[0]) __stcs(reinterpret_cast<float2*>(p.dst[0] + n * p.dstride[0]) + q, make_float2(v[k].x, v[k].z));
    if (p.dst[1]) __stcs(reinterpret_cast<float2*>(p.dst[1] + n * p.dstride[1]) + q, make_float2(v[k].y, v[k].w));
  }
}

// ---------------------------------------------------------------------------------------------
// RAFT's convex 8x flow upsampling (utils/raft/raft/raft.py:72-83), the step right before the path: the flows the
// kernels above consume are produced by it.  softmax over the 9 mask logits, convex combination of the 3x3 coarse
// neighbourhood of 8*flow (zero padded, F.unfold), pixel shuffle to (N,2,8H,8W) -- one pass: the (N,576,H,W) mask is
// read once (2304 B per coarse pixel, coalesced along w), the fine flow is written once (coalesced through a shared tile).
// ---------------------------------------------------------------------------------------------
constexpr int kUpW = 32;   // coarse cells per CTA (one coarse row segment)
__global__ void __launch_bounds__(256) upsample_flow_kernel(const float* __restrict__ flow, const float* __restrict__ mask,
                                                            float* __restrict__ out, int H, int W, int segs) {
  __shared__ float s_fl[2][3][kUpW + 2];          // 8 * coarse flow, rows h-1..h+1, cols w0-1..w0+32 (zero padded)
  __shared__ float s_out[2][8][8 * kUpW + 4];     // fine rows 8h..8h+7, cols 8*w0 .. 8*w0+255
  const int lane = threadIdx.x & 31, wrp = threadIdx.x >> 5;
  const int seg = blockIdx.x % segs, h = (blockIdx.x / segs) % H, n = blockIdx.x / (segs * H);
  const int w0 = seg * kUpW;
  const size_t cplane = (size_t)H * W;
  for (int i = threadIdx.x; i < 2 * 3 * (kUpW + 2); i += 256) {
    const int c = i / (3 * (kUpW + 2)), r = (i / (kUpW + 2)) % 3, x = i % (kUpW + 2);
    const int hh = h + r - 1, ww = w0 + x - 1;
    s_fl[c][r][x] = (hh >= 0 && hh < H && ww >= 0 && ww < W) ? 8.0f * __ldg(flow + ((size_t)n * 2 + c) * cplane + (size_t)hh * W + ww) : 0.0f;
  }
  __syncthreads();
  const int w = w0 + lane;
  if (w < W) {
    const float* mp = mask + (size_t)n * 576 * cplane + (size_t)h * W + w;
#pragma unroll 2
    for (int ij = wrp; ij < 64; ij += 8) {          // sub-pixel (i, j) = (ij / 8, ij % 8); lanes = 32 coarse columns
      float m[9], mx = -3.4e38f;
#pragma unroll
      for (int k = 0; k < 9; ++k) { m[k] = __ldcs(mp + (size_t)(k * 64 + ij) * cplane); mx = fmaxf(mx, m[k]); }
      float sum = 0.0f, au = 0.0f, av = 0.0f;
#pragma unroll
      for (int k = 0; k < 9; ++k) {
        const float e = __expf(m[k] - mx);
        sum += e;
        au = fmaf(e, s_fl[0][k / 3][lane + k % 3], au);   // unfold order: k = 3 * (dy + 1) + (dx + 1)
        av = fmaf(e, s_fl[1][k / 3][lane + k % 3], av);
      }
      const float inv = 1.0f / sum;
      s_out[0][ij >> 3][8 * lane + (ij & 7)] = au * inv;
      s_out[1][ij >> 3][8 * lane + (ij & 7)] = av * inv;
    }
  }
  __syncthreads();
  const int ncol = min(8 * kUpW, 8 * (W - w0));
  const size_t fW = (size_t)8 * W, fplane = (size_t)64 * cplane;
  for (int i = threadIdx.x; i < 2 * 8 * 8 * kUpW; i += 256) {
    const int c = i / (8 * 8 * kUpW), r = (i / (8 * kUpW)) % 8, x = i % (8 * kUpW);
    if (x < ncol) __stcs(out + ((size_t)n * 2 + c) * fplane + (size_t)(8 * h + r) * fW + 8 * w0 + x, s_out[c][r][x]);
  }
}

}  // namespace tcl

// =============================================================================================
// C ABI
// =============================================================================================
using namespace tcl;

static thread_local char g_err[512] = "";
static unsigned long long g_launches = 0;   // kernels of this library launched by this process (diagnostics / bench.py)

namespace tcl {   // for tcl_host.cu / tcl_cv2.cu
void set_last_error(const char* msg) { snprintf(g_err, sizeof(g_err), "%s", msg); }
void count_launch() { ++g_launches; }
}

static int fail(int code, const char* fmt, const char* detail = "") {
  snprintf(g_err, sizeof(g_err), fmt, detail);
  return code;
}
#define CUDA_TRY(expr)                                                                  \
  do {                                                                                  \
    cudaError_t e__ = (expr);                                                           \
    if (e__ != cudaSuccess) return fail(TCLB200_ERR_CUDA, #expr ": %s", cudaGetErrorString(e__)); \
  } while (0)

static bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

extern "C" int tclb200_abi_version(void) { return TCLB200_ABI_VERSION; }
extern "C" const char* tclb200_last_error(void) { return g_err; }

#define TCL_STR2(x) #x
#define TCL_STR(x) TCL_STR2(x)
#ifdef TCL_HOT_ONLY
#define TCL_HOT_ONLY_V 1
#else
#define TCL_HOT_ONLY_V 0
#endif
#ifdef TCL_TRACE
#define TCL_TRACE_V 1
#else
#define TCL_TRACE_V 0
#endif
#ifdef TCL_CWARPS
#define TCL_CWARPS_S TCL_STR(TCL_CWARPS)
#else
#define TCL_CWARPS_S "8/16"
#endif
extern "C" const char* tclb200_build_info(void) {
  return "abi=" TCL_STR(TCLB200_ABI_VERSION) " th=" TCL_STR(TCL_TH) " bh=" TCL_STR(TCL_BH) "/" TCL_STR(TCL_BH8) " bw=" TCL_STR(TCL_BW) " bw16=" TCL_STR(TCL_BW16)
         " ns=" TCL_STR(TCL_NS) "/" TCL_STR(TCL_NS_NOFF) " nb=" TCL_STR(TCL_NB) " cwarps=" TCL_CWARPS_S " scanners=" TCL_STR(TCL_SCANNERS) " packed=" TCL_STR(TCL_PACKED)
         " packed_given=" TCL_STR(TCL_PACKED_GIVEN) " hot_only=" TCL_STR(TCL_HOT_ONLY_V) " diag=" TCL_STR(TCL_DIAG) " trace=" TCL_STR(TCL_TRACE_V);
}

// tile shape of the TMA kernel: 64 x TH pixels per tile, 80 x BH source boxes: after rounding the box origin down
// to a 16-byte boundary the taps may still spread >= 8 px in x and BH-TH-1 px in y beyond the tile's own extent
// before the tile falls back to global gathers
constexpr int kTW = 64, kTH = TCL_TH;
constexpr int box_height(int cw, int esize) { return esize == 2 ? TCL_BH16 : (cw == 8 ? TCL_BH8 : TCL_BH); }
template <typename FrameT> constexpr int box_width() { return sizeof(FrameT) == 4 ? TCL_BW : TCL_BW16; }

static inline int cdiv(int a, int b) { return (a + b - 1) / b; }
// scratch is sized for the finest tiling any kernel uses (32 x 8 generic tiles)
extern "C" size_t tclb200_scratch_bytes(int B, int H, int W) {
  if (B <= 0 || H <= 0 || W <= 0) return 0;
  const size_t tpp = (size_t)cdiv(W, 32) * cdiv(H, kWarps);
  return align_up((size_t)B * tpp * sizeof(double), 256) + align_up(((size_t)B + 3) * sizeof(unsigned), 256);
}

// ---- tensor maps -------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = []() -> EncodeTiledFn {
    void* sym = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &q) != cudaSuccess) return nullptr;
    return q == cudaDriverEntryPointSuccess ? reinterpret_cast<EncodeTiledFn>(sym) : nullptr;
  }();
  return fn;
}

// (W, H, planes, B) view of an NCHW tensor with a (bw, bh, bp, 1) box; plane_stride / batch_stride in elements
// (0 = dense): rows are always dense, planes and images may lie further apart (a cropped view of a padded tensor)
static bool make_map(CUtensorMap* m, const void* base, int esize, int W, int H, int planes, int B, int bw, int bh, int bp,
                     size_t plane_stride = 0, size_t batch_stride = 0) {
  EncodeTiledFn fn = encode_fn();
  if (!fn || !base) return false;
  if (!plane_stride) plane_stride = (size_t)W * H;
  if (!batch_stride) batch_stride = plane_stride * planes;
  const cuuint64_t dims[4] = {(cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)planes, (cuuint64_t)B};
  const cuuint64_t strides[3] = {(cuuint64_t)W * esize, (cuuint64_t)plane_stride * esize, (cuuint64_t)batch_stride * esize};
  const cuuint32_t box[4] = {(cuuint32_t)bw, (cuuint32_t)bh, (cuuint32_t)bp, 1u};
  const cuuint32_t estr[4] = {1u, 1u, 1u, 1u};
  const CUtensorMapDataType dt = esize == 2 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32;
  return fn(m, dt, 4, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
            CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// ---- launches ----------------------------------------------------------------------------------
static int sm_count() {   // of the current device, cached per device index (a process may drive different GPUs / MIG slices)
  static int cache[64] = {};
  int dev = 0, v = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return 148;
  if (dev >= 0 && dev < 64 && cache[dev] > 0) return cache[dev];
  if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || v <= 0) return 148;
  if (dev >= 0 && dev < 64) cache[dev] = v;
  return v;
}

static cudaError_t launch_fold(const FwdParams& p, cudaStream_t s);

template <typename FrameT, int MASK, bool REDUCE, int CT, int LEAN, int CW>
static cudaError_t launch_tma_cw(const FwdParams& p, const CUtensorMap& tb, const CUtensorMap& tf, const CUtensorMap& tp, const CUtensorMap& tc,
                                 cudaStream_t s) {
  constexpr bool has_ff = MASK == MASK_COMPUTED;
  // (mask-only launches stage no frame planes: a third source stage fits beside the flow ring)
  constexpr int NS = has_ff ? (CT == 0 && LEAN == 1 ? TCL_NS_MASK : TCL_NS) : TCL_NS_NOFF, NB = has_ff ? (CT == 0 && LEAN == 1 ? TCL_NS_MASK + 2 : TCL_NB) : TCL_NS_NOFF + 2;
  using Cfg = WsCfg<FrameT, CT, kTW, kTH, box_width<FrameT>(), (has_ff ? box_height(CW, (int)sizeof(FrameT)) : TCL_BH_NOFF), NB, NS, CW, has_ff>;
  auto kern = fused_forward_ws_kernel<FrameT, MASK, REDUCE, CT, LEAN, Cfg>;
  static bool configured[64] = {};  // per instantiation and device (the attribute is a per-device property of the function)
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) dev = 63;   // (an uncached slot: set the attribute every time)
  if (!configured[dev] || dev == 63) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Cfg::kSmemBytes);
    if (e != cudaSuccess) return e;
    configured[dev] = true;
  }
  // persistent: one CTA per SM (or fewer when there are fewer tiles)
  const size_t tiles = (size_t)p.B * p.tiles_per_pair;
  const size_t slots = (size_t)sm_count();
  const unsigned grid = (unsigned)(tiles < slots ? tiles : slots);
  kern<<<grid, Cfg::kThreads, Cfg::kSmemBytes, s>>>(p, tb, tf, tp, tc);
  ++g_launches;
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess || !REDUCE) return e;
  return launch_fold(p, s);
}

// Consumer warps per CTA.  The packed-arithmetic configuration on fp32 frames (computeTCL: both mask tests, C == 3) runs
// best with 8 warps x 8 pixels per lane on large frames (Sintel shape: 130 vs 124 Gpix/s); small frames, where a larger
// share of the tiles straddles a motion boundary and waits for global gathers (256 x 256 training crops: 87 vs 97), bf16
// frames (98 vs 123) and every other configuration run best with 16 warps x 4 pixels.
template <typename FrameT, int MASK, bool REDUCE, int CT, int LEAN>
static cudaError_t launch_tma(const FwdParams& p, const CUtensorMap& tb, const CUtensorMap& tf, const CUtensorMap& tp, const CUtensorMap& tc,
                              cudaStream_t s) {
  // (decided by run_fused, which sized the tensor maps' boxes for it: wants_packed8)
  constexpr bool packed8 = TCL_PACKED && MASK == MASK_COMPUTED && sizeof(FrameT) == 4 &&
                           (((LEAN == 1 || LEAN == 2) && CT == 3) || (TCL_PACKED_MASK && LEAN == 1 && CT == 0 && !REDUCE));
  if constexpr (packed8 && kCWarpsPacked != kCWarpsOther) {
    if (p.cw_packed) return launch_tma_cw<FrameT, MASK, REDUCE, CT, LEAN, kCWarpsPacked>(p, tb, tf, tp, tc, s);
  }
  if (p.cw_packed && kCWarpsPacked != kCWarpsOther) return cudaErrorInvalidConfiguration;   // (tensor maps sized for the other variant)
  return launch_tma_cw<FrameT, MASK, REDUCE, CT, LEAN, kCWarpsOther>(p, tb, tf, tp, tc, s);
}

static cudaError_t launch_fold(const FwdParams& p, cudaStream_t s) {   // behind a kernel that stored one fp64 partial per tile
  ++g_launches;
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  const bool small = p.B <= kFoldSmallPairs && (size_t)p.B * p.tiles_per_pair <= (size_t)kFoldSmallPartials;
  cfg.gridDim = dim3(small ? 1u : (unsigned)p.B); cfg.blockDim = dim3(small ? 1024 : kThreads); cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr; cfg.numAttrs = 1;
  return small ? cudaLaunchKernelEx(&cfg, fold_partials_small_kernel, p) : cudaLaunchKernelEx(&cfg, fold_partials_kernel, p);
}

template <typename FrameT>
static cudaError_t launch_direct(const FwdParams& p, cudaStream_t s) {
  auto kern = p.loss == TCLB200_L1 ? fused_forward_direct_kernel<FrameT, TCLB200_L1> : fused_forward_direct_kernel<FrameT, TCLB200_L2>;
  kern<<<(unsigned)((size_t)p.B * p.tiles_per_pair), kDirectThreads, 0, s>>>(p);
  ++g_launches;
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  return launch_fold(p, s);
}

template <typename FrameT, int MASK, bool REDUCE>
static cudaError_t launch_generic(const FwdParams& p, cudaStream_t s) {
  const unsigned grid = (unsigned)((size_t)p.B * p.tiles_per_pair);
  if (p.C == 3) fused_forward_generic_kernel<FrameT, MASK, REDUCE, 3><<<grid, kThreads, 0, s>>>(p);
  else fused_forward_generic_kernel<FrameT, MASK, REDUCE, 0><<<grid, kThreads, 0, s>>>(p);
  ++g_launches;
  return cudaGetLastError();
}

template <typename FrameT>
static cudaError_t dispatch(const FwdParams& p, int mask_kind, bool reduce, bool tma, const CUtensorMap& tb, const CUtensorMap& tf,
                            const CUtensorMap& tp, const CUtensorMap& tc, cudaStream_t s) {
#ifdef TCL_HOT_ONLY   // tuning builds (tools/sweep_build.py): only the fp32 (1) or bf16 (2) computeTCL configuration, compiles in seconds
  if (sizeof(FrameT) == (TCL_HOT_ONLY == 2 ? 2 : 4) && mask_kind == MASK_COMPUTED && reduce && tma && p.C == 3 && p.prev && p.cur && !p.warp_out && !p.mask_out &&
      !p.blend_out && !p.near_threshold && p.loss == TCLB200_L2)
    return launch_tma<typename std::conditional<TCL_HOT_ONLY == 2, __nv_bfloat16, float>::type, MASK_COMPUTED, true, 3, 1>(p, tb, tf, tp, tc, s);
  if (mask_kind == MASK_COMPUTED && !reduce && !p.prev) return launch_generic<float, MASK_COMPUTED, false>(p, s);
  return cudaErrorNotSupported;
#else
#define TCL_CASE(MK, RD)                                                                       \
  if (mask_kind == MK && reduce == RD) {                                                       \
    if (!tma) return launch_generic<FrameT, MK, RD>(p, s);                                     \
    if (p.C == 3 && lean_out && MK != MASK_NONE) return launch_tma<FrameT, (MK == MASK_NONE ? MASK_GIVEN : MK), RD, 3, 4>(p, tb, tf, tp, tc, s); \
    if (p.C == 3 && lean && RD) return p.loss == TCLB200_L1 ? launch_tma<FrameT, MK, true, 3, 2>(p, tb, tf, tp, tc, s)   \
                                                            : launch_tma<FrameT, MK, true, 3, 1>(p, tb, tf, tp, tc, s);  \
    if (MK == MASK_COMPUTED && !RD && lean_mask) return launch_tma<float, MASK_COMPUTED, false, 0, 1>(p, tb, tf, tp, tc, s); \
    if (MK == MASK_COMPUTED && !RD && lean_mob) return launch_tma<float, MASK_COMPUTED, false, 0, 3>(p, tb, tf, tp, tc, s); \
    if (MK == MASK_NONE && !RD && lean_warp) return launch_tma<FrameT, MASK_NONE, false, 3, 1>(p, tb, tf, tp, tc, s); \
    return p.C == 3 ? launch_tma<FrameT, MK, RD, 3, 0>(p, tb, tf, tp, tc, s) : launch_tma<FrameT, MK, RD, 0, 0>(p, tb, tf, tp, tc, s); \
  }
  // LEAN = the measured hot configurations, fixed at compile time: computeTCL / training loss with C == 3
  const bool lean = reduce && p.prev && p.cur && !p.warp_out && !p.mask_out && !p.blend_out && !p.near_threshold &&
                    !(p.flags & TCLB200_VALIDITY) && mask_kind != MASK_NONE &&
                    (mask_kind != MASK_COMPUTED || (p.flags & (TCLB200_OCC | TCLB200_MOB)) == (TCLB200_OCC | TCLB200_MOB));
  // ... the same with per-pixel outputs (warp / mask / blend), with or without the reduction
  const bool lean_out = p.prev && p.cur && (p.warp_out || p.blend_out || (p.mask_out && mask_kind == MASK_COMPUTED)) &&
                        !(p.mask_out && mask_kind == MASK_GIVEN) && !p.near_threshold && !(p.flags & TCLB200_VALIDITY) &&
                        p.loss == TCLB200_L2 && mask_kind != MASK_NONE &&
                        (mask_kind != MASK_COMPUTED || (p.flags & (TCLB200_OCC | TCLB200_MOB)) == (TCLB200_OCC | TCLB200_MOB));
  // ... and fbcCheckTorch on its own: both tests, mask_out only
  const bool lean_mask = !reduce && !p.prev && p.mask_out && !p.near_threshold && mask_kind == MASK_COMPUTED &&
                         (p.flags & (TCLB200_OCC | TCLB200_MOB)) == (TCLB200_OCC | TCLB200_MOB);
  // ... and its optimisation-based variant: the motion-boundary test alone
  const bool lean_mob = !reduce && !p.prev && p.mask_out && !p.near_threshold && mask_kind == MASK_COMPUTED &&
                        (p.flags & (TCLB200_OCC | TCLB200_MOB)) == TCLB200_MOB;
  // ... and warp() on its own (C == 3, no validity mask): warp_out only
  const bool lean_warp = !reduce && p.prev && p.C == 3 && !p.cur && p.warp_out && !p.mask_out && !p.blend_out && mask_kind == MASK_NONE;
  TCL_CASE(MASK_COMPUTED, true)
  TCL_CASE(MASK_COMPUTED, false)
  TCL_CASE(MASK_GIVEN, true)
  TCL_CASE(MASK_GIVEN, false)
  TCL_CASE(MASK_NONE, true)
  TCL_CASE(MASK_NONE, false)
#undef TCL_CASE
  return cudaErrorInvalidValue;
#endif
}

extern "C" int tclb200_debug_tile_stats(unsigned long long* out2, int reset) {
  unsigned long long zero[2] = {0, 0};
  if (out2) CUDA_TRY(cudaMemcpyFromSymbol(out2, tcl::g_tile_stats, sizeof(zero)));
  if (reset) CUDA_TRY(cudaMemcpyToSymbol(tcl::g_tile_stats, zero, sizeof(zero)));
  return TCLB200_OK;
}

extern "C" unsigned long long tclb200_debug_launch_count(int reset) {
  const unsigned long long n = g_launches;
  if (reset) g_launches = 0;
  return n;
}

#ifdef TCL_TRACE
extern "C" int tclb200_debug_trace(unsigned long long* out, size_t bytes) {
  if (bytes > sizeof(tcl::g_trace)) bytes = sizeof(tcl::g_trace);
  CUDA_TRY(cudaMemcpyFromSymbol(out, tcl::g_trace, bytes));
  return TCLB200_OK;
}
#endif

// test / tuning hook: 1 = the generic kernel on TMA-capable shapes, 2 = never the direct kernel, 3 = the direct kernel whatever the size
static int g_force_generic = 0;
extern "C" void tclb200_debug_force_generic(int on) { g_force_generic = on; }
// launches up to this many pixels go to the direct kernel when their configuration allows (training loss with a dataset
// mask); beyond it the persistent pipeline's steady state wins (measured, tools/small_launch.py)
#ifndef TCL_DIRECT_MAX_PX
#define TCL_DIRECT_MAX_PX (2u << 20)
#endif

static int run_fused(const tclb200_tcl_args* a, cudaStream_t s) {
  if (!a) return fail(TCLB200_ERR_INVALID, "args is NULL");
  if (a->B <= 0 || a->H <= 0 || a->W <= 0) return fail(TCLB200_ERR_INVALID, "B, H, W must be positive");
  if (!a->bf) return fail(TCLB200_ERR_INVALID, "bf (the flow the warp samples with) is required");
  if (a->dtype != TCLB200_F32 && a->dtype != TCLB200_BF16) return fail(TCLB200_ERR_INVALID, "unknown dtype");
  if (a->loss != TCLB200_L2 && a->loss != TCLB200_L1) return fail(TCLB200_ERR_INVALID, "unknown loss");
  if (a->finalize != TCLB200_FIN_MEAN && a->finalize != TCLB200_FIN_RMSE) return fail(TCLB200_ERR_INVALID, "unknown finalize");
  if (a->prev && a->C <= 0) return fail(TCLB200_ERR_INVALID, "C must be positive when frames are given");
  if ((a->cur || a->warp_out || a->blend_out) && !a->prev) return fail(TCLB200_ERR_INVALID, "prev is required with cur / warp_out / blend_out");
  if (a->blend_out && !a->cur) return fail(TCLB200_ERR_INVALID, "blend_out needs cur");
  if ((a->prev_index && a->n_prev_frames <= 0) || (a->cur_index && a->n_cur_frames <= 0))
    return fail(TCLB200_ERR_INVALID, "prev_index / cur_index need n_prev_frames / n_cur_frames");
  if ((a->bf_index && a->n_bf_fields <= 0) || (a->ff && a->ff_index && a->n_ff_fields <= 0))
    return fail(TCLB200_ERR_INVALID, "bf_index / ff_index need n_bf_fields / n_ff_fields");
  if (a->pair_group < 0) return fail(TCLB200_ERR_INVALID, "pair_group must not be negative");
  const bool band = a->row_begin != 0 || a->row_end != 0;
  if (band && (a->row_begin < 0 || a->row_end <= a->row_begin || a->row_end > a->H))
    return fail(TCLB200_ERR_INVALID, "band mode needs 0 <= row_begin < row_end <= H");
  if (band && (a->pair_vals || a->total_val)) return fail(TCLB200_ERR_INVALID, "band mode returns sums only (pair_sums / total_sums): a band's mean is not the frame's");
  if ((size_t)a->H * a->W >= (1u << 30)) return fail(TCLB200_ERR_UNSUPPORTED, "H*W must be below 2^30");
  const bool reduce = a->cur && (a->pair_sums || a->total_sums || a->pair_vals || a->total_val);
  const int mask_kind = a->ff ? MASK_COMPUTED : (a->mask_in ? MASK_GIVEN : MASK_NONE);
  if (mask_kind == MASK_COMPUTED && !(a->flags & (TCLB200_OCC | TCLB200_MOB)))
    return fail(TCLB200_ERR_INVALID, "ff given but neither TCLB200_OCC nor TCLB200_MOB requested");
  if (!a->prev && !a->mask_out) return fail(TCLB200_ERR_INVALID, "nothing to compute: no frames and no mask_out");

  const int esz = a->dtype == TCLB200_BF16 ? 2 : 4;
  // flows may be row-dense views with their own plane / pair strides (RAFT's padded output cropped by
  // InputPadder.unpad or flow_up[:,:,:H,:]); 0 = dense
  const size_t hw = (size_t)a->H * a->W;
  const size_t bf_plane = a->bf_plane_stride ? a->bf_plane_stride : hw, bf_batch = a->bf_batch_stride ? a->bf_batch_stride : 2 * bf_plane;
  const size_t ff_plane = a->ff_plane_stride ? a->ff_plane_stride : hw, ff_batch = a->ff_batch_stride ? a->ff_batch_stride : 2 * ff_plane;
  if (bf_plane < hw || ff_plane < hw || (a->B > 1 && (bf_batch < hw || ff_batch < hw)))
    return fail(TCLB200_ERR_INVALID, "flow plane / pair strides must be at least H*W");
  const bool strides16 = bf_plane % 4 == 0 && bf_batch % 4 == 0 && ff_plane % 4 == 0 && ff_batch % 4 == 0;   // TMA: 16-byte strides
  // TMA needs 16-byte aligned bases and row strides; frames need C == 3 (the compiled box depth)
  bool tma = g_force_generic != 1 && (a->W % 4 == 0) && ((a->W * esz) % 16 == 0) && aligned16(a->bf) && aligned16(a->ff) &&
             aligned16(a->prev) && aligned16(a->cur) && (!a->prev || a->C == 3) && a->B <= 65535 * 16 && strides16 &&
             a->H <= 16384 && a->W <= 16384;   // (box addresses are evaluated in fp32, see lean_tile)
  // the packed-arithmetic configuration on large fp32 frames runs with 8 consumer warps and taller boxes (launch_tma): the
  // same conditions as dispatch()'s `lean` for the computed-mask reductions
  const bool cw_hot = reduce && a->prev && a->cur && a->C == 3 && !a->warp_out && !a->mask_out && !a->blend_out;
  const bool cw_mask = TCL_PACKED_MASK && !reduce && !a->prev && a->mask_out;   // (dispatch()'s `lean_mask`: fbcCheckTorch on its own)
  const bool cw_packed = TCL_PACKED && kCWarpsPacked != kCWarpsOther && tma && a->dtype == TCLB200_F32 && mask_kind == MASK_COMPUTED &&
                         (cw_hot || cw_mask) && !a->near_threshold &&
                         !(a->flags & TCLB200_VALIDITY) && (a->flags & (TCLB200_OCC | TCLB200_MOB)) == (TCLB200_OCC | TCLB200_MOB) &&
                         (size_t)a->H * a->W >= (size_t)384 * 384;
  // short launches of the training loss (dataset mask, reduction only): the direct kernel, no tensor maps needed
  const size_t launch_px = (size_t)a->B * (size_t)((band ? a->row_end - a->row_begin : a->H)) * a->W;
  const bool direct = tma && g_force_generic != 2 && mask_kind == MASK_GIVEN && reduce && a->C == 3 && !a->warp_out && !a->mask_out &&
                      !a->blend_out && !a->near_threshold && !(a->flags & (TCLB200_VALIDITY | TCLB200_THROUGHPUT)) && aligned16(a->mask_in) &&
                      (launch_px <= TCL_DIRECT_MAX_PX || g_force_generic == 3);
  CUtensorMap tb, tf, tp, tc;
  memset(&tb, 0, sizeof(tb)); memset(&tf, 0, sizeof(tf)); memset(&tp, 0, sizeof(tp)); memset(&tc, 0, sizeof(tc));
  if (tma && !direct) {
    const int bw = a->dtype == TCLB200_BF16 ? box_width<__nv_bfloat16>() : box_width<float>();
    const int kBH = mask_kind == MASK_COMPUTED ? box_height(cw_packed ? kCWarpsPacked : kCWarpsOther, esz) : TCL_BH_NOFF;
    tma = make_map(&tb, a->bf, 4, a->W, a->H, 2, a->bf_index ? a->n_bf_fields : a->B, kTW + 16, kTH + 2, 2, bf_plane, bf_batch);
    if (tma && mask_kind == MASK_COMPUTED && (a->flags & TCLB200_OCC))
      tma = make_map(&tf, a->ff, 4, a->W, a->H, 2, a->ff_index ? a->n_ff_fields : a->B, bw, kBH, 2, ff_plane, ff_batch);
    if (tma && a->prev) tma = make_map(&tp, a->prev, esz, a->W, a->H, 3, a->prev_index ? a->n_prev_frames : a->B, bw, kBH, 3);
    if (tma && a->prev && a->cur) tma = make_map(&tc, a->cur, esz, a->W, a->H, 3, a->cur_index ? a->n_cur_frames : a->B, kTW, kTH, 3);
  }

  FwdParams p;
  memset(&p, 0, sizeof(p));
  p.ff = a->ff; p.bf = a->bf; p.mask_in = a->mask_in; p.prev = a->prev; p.cur = a->cur;
  p.ff_plane = ff_plane; p.ff_batch = ff_batch; p.bf_plane = bf_plane; p.bf_batch = bf_batch;
  p.prev_index = a->prev ? a->prev_index : nullptr; p.cur_index = a->cur ? a->cur_index : nullptr;
  p.bf_index = a->bf_index; p.ff_index = a->ff ? a->ff_index : nullptr;
  p.pair_group = a->pair_group > 1 ? a->pair_group : 1;
  p.cw_packed = cw_packed ? 1 : 0;
  p.warp_out = a->warp_out; p.mask_out = a->mask_out; p.blend_out = a->blend_out;
  p.pair_sums = a->pair_sums; p.total_sums = a->total_sums; p.pair_vals = a->pair_vals; p.total_val = a->total_val;
  p.near_threshold = a->near_threshold;
  p.geo = make_geo(a->H, a->W);
  p.B = a->B; p.C = a->prev ? a->C : 0;
  p.row_begin = band ? a->row_begin : 0;
  p.row_end = band ? a->row_end : a->H;
  p.tiles_x = tma ? cdiv(a->W, kTW) : cdiv(a->W, 32);
  p.tiles_per_pair = p.tiles_x * (tma ? cdiv(p.row_end - p.row_begin, kTH) : cdiv(p.row_end - p.row_begin, kWarps));
  if (direct) { p.tiles_x = 0; p.tiles_per_pair = (int)(((size_t)(p.row_end - p.row_begin) * a->W + kDirectChunk - 1) / kDirectChunk); }
  p.flags = a->flags; p.loss = a->loss; p.finalize = a->finalize;
  p.inv_count = a->prev ? 1.0 / ((double)a->C * a->H * a->W) : 0.0;
  if ((size_t)p.B * p.tiles_per_pair >= 0x7fffffffu) return fail(TCLB200_ERR_UNSUPPORTED, "too many tiles for one launch");
  if (reduce) {
    if (!a->scratch || a->scratch_bytes < tclb200_scratch_bytes(a->B, a->H, a->W))
      return fail(TCLB200_ERR_INVALID, "scratch missing or smaller than tclb200_scratch_bytes(B,H,W)");
    char* base = reinterpret_cast<char*>(a->scratch);
    const size_t tpp_max = (size_t)cdiv(a->W, 32) * cdiv(a->H, kWarps);
    p.scratch.partials = reinterpret_cast<double*>(base);
    p.scratch.pair_ticket = reinterpret_cast<unsigned*>(base + align_up((size_t)a->B * tpp_max * sizeof(double), 256));
    p.scratch.batch_ticket = p.scratch.pair_ticket + a->B;
    // long launches of the TMA kernel hand out tiles through a counter (two words behind the tickets)
    const size_t tiles = (size_t)p.B * p.tiles_per_pair;
    p.scratch.tile_ctr = (tma && !direct && tiles > 16 * (size_t)sm_count()) ? p.scratch.batch_ticket + 1 : nullptr;
  }
  if (direct) {
    const cudaError_t e = a->dtype == TCLB200_BF16 ? launch_direct<__nv_bfloat16>(p, s) : launch_direct<float>(p, s);
    if (e != cudaSuccess) return fail(TCLB200_ERR_CUDA, "fused forward (direct) launch: %s", cudaGetErrorString(e));
    return TCLB200_OK;
  }
  const cudaError_t e = a->dtype == TCLB200_BF16 ? dispatch<__nv_bfloat16>(p, mask_kind, reduce, tma, tb, tf, tp, tc, s)
                                                 : dispatch<float>(p, mask_kind, reduce, tma, tb, tf, tp, tc, s);
  if (e != cudaSuccess) return fail(TCLB200_ERR_CUDA, "fused forward launch: %s", cudaGetErrorString(e));
  return TCLB200_OK;
}

extern "C" int tclb200_tcl_forward(const tclb200_tcl_args* args, tclb200_stream_t stream) {
  return run_fused(args, reinterpret_cast<cudaStream_t>(stream));
}

extern "C" int tclb200_warp(const void* x, const float* f, void* out, int B, int C, int H, int W, int dtype, int flags,
                            tclb200_stream_t stream) {
  if (!x || !f || !out) return fail(TCLB200_ERR_INVALID, "x, f and out are required");
  tclb200_tcl_args a;
  memset(&a, 0, sizeof(a));
  a.bf = f; a.prev = x; a.warp_out = out;
  a.B = B; a.C = C; a.H = H; a.W = W; a.dtype = dtype; a.flags = flags & TCLB200_VALIDITY;
  return run_fused(&a, reinterpret_cast<cudaStream_t>(stream));
}

extern "C" int tclb200_fbcheck(const float* ff, const float* bf, float* mask_out, int B, int H, int W, int flags,
                               unsigned long long* near_threshold, tclb200_stream_t stream) {
  if (!bf || !mask_out) return fail(TCLB200_ERR_INVALID, "bf and mask_out are required");
  if ((flags & TCLB200_OCC) && !ff) return fail(TCLB200_ERR_INVALID, "ff is required for the occlusion test");
  if (!(flags & (TCLB200_OCC | TCLB200_MOB))) return fail(TCLB200_ERR_INVALID, "flags must request TCLB200_OCC and/or TCLB200_MOB");
  tclb200_tcl_args a;
  memset(&a, 0, sizeof(a));
  a.ff = ff ? ff : bf;  // the motion-boundary-only variant never reads ff
  a.bf = bf; a.mask_out = mask_out; a.near_threshold = near_threshold;
  a.B = B; a.C = 0; a.H = H; a.W = W; a.flags = flags & (TCLB200_OCC | TCLB200_MOB);
  return run_fused(&a, reinterpret_cast<cudaStream_t>(stream));
}

static int run_gradient(const float* x, size_t in_stride, float* out, int B, int H, int W, cudaStream_t s) {
  if (!x || !out) return fail(TCLB200_ERR_INVALID, "x and out are required");
  if (B <= 0 || H <= 0 || W <= 0) return fail(TCLB200_ERR_INVALID, "B, H, W must be positive");
  if (in_stride < (size_t)H * W) return fail(TCLB200_ERR_INVALID, "x_batch_stride must be at least H*W");
  const bool vec4 = !g_force_generic && W % 4 == 0 && aligned16(x) && aligned16(out) && ((size_t)H * W) % 4 == 0 && in_stride % 4 == 0;
  const int tx = cdiv(W, vec4 ? 128 : 32), tpi = tx * cdiv(H, kWarps);
  if ((size_t)B * tpi >= 0x7fffffffu) return fail(TCLB200_ERR_UNSUPPORTED, "too many tiles for one launch");
  if (vec4) gradient_vec4_kernel<<<(unsigned)((size_t)B * tpi), kThreads, 0, s>>>(x, in_stride, out, B, H, W, tx, tpi);
  else gradient_kernel<<<(unsigned)((size_t)B * tpi), kThreads, 0, s>>>(x, in_stride, out, B, H, W, tx, tpi);
  ++g_launches;
  CUDA_TRY(cudaGetLastError());
  return TCLB200_OK;
}

extern "C" int tclb200_gradient(const float* x, float* out, int B, int H, int W, tclb200_stream_t stream) {
  return run_gradient(x, (size_t)(H > 0 && W > 0 ? (size_t)H * W : 0), out, B, H, W, reinterpret_cast<cudaStream_t>(stream));
}

extern "C" int tclb200_gradient_strided(const float* x, size_t x_batch_stride, float* out, int B, int H, int W, tclb200_stream_t stream) {
  return run_gradient(x, x_batch_stride, out, B, H, W, reinterpret_cast<cudaStream_t>(stream));
}

template <typename FrameT>
static void launch_backward(const BwdParams& p, bool fused, dim3 grid, cudaStream_t s) {
  if (fused) {
    if (p.C == 3) warp_backward_kernel<true, 3, FrameT><<<grid, 256, 0, s>>>(p);
    else warp_backward_kernel<true, 0, FrameT><<<grid, 256, 0, s>>>(p);
  } else {
    if (p.C == 3) warp_backward_kernel<false, 3, FrameT><<<grid, 256, 0, s>>>(p);
    else if (p.C == 2) warp_backward_kernel<false, 2, FrameT><<<grid, 256, 0, s>>>(p);
    else warp_backward_kernel<false, 0, FrameT><<<grid, 256, 0, s>>>(p);
  }
}

// bf16 frames: p.grad_x is the fp32 accumulator and grad_x_bf16 the caller's output it is rounded into
static int run_backward(const BwdParams& p, bool fused, int dtype, __nv_bfloat16* grad_x_bf16, cudaStream_t s) {
  const size_t n = (size_t)p.B * p.geo.H * p.geo.W;
  if (dtype == TCLB200_BF16 && p.grad_x && n * p.C / (4 * kThreads) >= 0x7fffffffu)
    return fail(TCLB200_ERR_UNSUPPORTED, "too many elements for one rounding launch");
  if (p.grad_x) CUDA_TRY(cudaMemsetAsync(p.grad_x, 0, n * p.C * sizeof(float), s));
  if (p.B > 65535) return fail(TCLB200_ERR_UNSUPPORTED, "batch too large for one backward launch");
  const dim3 grid((unsigned)cdiv(p.geo.W, 32), (unsigned)cdiv(p.geo.H, 8), (unsigned)p.B);
  if (grid.y > 65535) return fail(TCLB200_ERR_UNSUPPORTED, "image too tall for one backward launch");
  if (dtype == TCLB200_BF16) launch_backward<__nv_bfloat16>(p, fused, grid, s);
  else launch_backward<float>(p, fused, grid, s);
  ++g_launches;
  CUDA_TRY(cudaGetLastError());
  if (dtype == TCLB200_BF16 && p.grad_x) {
    const size_t count = n * p.C;
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3((unsigned)((count + 4 * kThreads - 1) / (4 * kThreads))); cfg.blockDim = dim3(kThreads); cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    const int vec = (reinterpret_cast<uintptr_t>(grad_x_bf16) & 7u) == 0;
    ++g_launches;
    CUDA_TRY(cudaLaunchKernelEx(&cfg, bwd_acc_to_bf16_kernel, (const float*)p.grad_x, grad_x_bf16, count, vec));
  }
  return TCLB200_OK;
}

extern "C" size_t tclb200_backward_workspace_bytes(int B, int C, int H, int W, int dtype) {
  if (dtype != TCLB200_BF16 || B <= 0 || C <= 0 || H <= 0 || W <= 0) return 0;
  return align_up((size_t)B * C * H * W * sizeof(float), 256);
}

// the frame dtype and, for bf16 frames with a grad_x / grad_prev, the accumulator workspace: p.grad_x is pointed at it
static int backward_dtype_setup(BwdParams& p, int dtype, void* grad_x, void* workspace, size_t workspace_bytes, const char* what) {
  if (dtype != TCLB200_F32 && dtype != TCLB200_BF16) return fail(TCLB200_ERR_INVALID, "unknown dtype");
  if (dtype == TCLB200_F32 || grad_x == nullptr) {
    p.grad_x = static_cast<float*>(grad_x);
    return TCLB200_OK;
  }
  const size_t need = tclb200_backward_workspace_bytes(p.B, p.C, p.geo.H, p.geo.W, dtype);
  if (workspace == nullptr || workspace_bytes < need) {
    static thread_local char msg[192];
    snprintf(msg, sizeof(msg), "%s of bf16 frames needs a workspace of tclb200_backward_workspace_bytes() = %zu bytes, got %zu",
             what, need, workspace ? workspace_bytes : (size_t)0);
    return fail(TCLB200_ERR_INVALID, "%s", msg);
  }
  if (!aligned16(workspace)) return fail(TCLB200_ERR_INVALID, "workspace must be 16-byte aligned");
  p.grad_x = static_cast<float*>(workspace);
  return TCLB200_OK;
}

extern "C" int tclb200_warp_backward_dt(const void* grad_out, const void* x, const float* f, void* grad_x, float* grad_f,
                                        int B, int C, int H, int W, int dtype, int flags, void* workspace, size_t workspace_bytes,
                                        tclb200_stream_t stream) {
  if (!grad_out || !x || !f) return fail(TCLB200_ERR_INVALID, "grad_out, x and f are required");
  if (B <= 0 || C <= 0 || H <= 0 || W <= 0) return fail(TCLB200_ERR_INVALID, "B, C, H, W must be positive");
  if ((size_t)H * W >= (1u << 30)) return fail(TCLB200_ERR_UNSUPPORTED, "H*W must be below 2^30");
  BwdParams p;
  memset(&p, 0, sizeof(p));
  p.grad_out = grad_out; p.x = x; p.f = f; p.grad_f = grad_f;
  p.geo = make_geo(H, W); p.B = B; p.C = C; p.flags = flags & TCLB200_VALIDITY;
  const int rc = backward_dtype_setup(p, dtype, grad_x, workspace, workspace_bytes, "grad_x");
  if (rc != TCLB200_OK) return rc;
  return run_backward(p, false, dtype, static_cast<__nv_bfloat16*>(grad_x), reinterpret_cast<cudaStream_t>(stream));
}

extern "C" int tclb200_warp_backward(const float* grad_out, const float* x, const float* f, float* grad_x, float* grad_f,
                                     int B, int C, int H, int W, int flags, tclb200_stream_t stream) {
  return tclb200_warp_backward_dt(grad_out, x, f, grad_x, grad_f, B, C, H, W, TCLB200_F32, flags, nullptr, 0, stream);
}

extern "C" int tclb200_tcl_backward_dt(const float* bf, const float* mask, const void* prev, const void* cur, const float* grad_scale,
                                       float scale_mul, void* grad_prev, void* grad_cur, int B, int C, int H, int W, int dtype,
                                       int flags, int loss, void* workspace, size_t workspace_bytes, tclb200_stream_t stream) {
  if (!bf || !prev || !cur || !grad_scale) return fail(TCLB200_ERR_INVALID, "bf, prev, cur and grad_scale are required");
  if (B <= 0 || C <= 0 || H <= 0 || W <= 0) return fail(TCLB200_ERR_INVALID, "B, C, H, W must be positive");
  if (loss != TCLB200_L2 && loss != TCLB200_L1) return fail(TCLB200_ERR_INVALID, "unknown loss");
  if ((size_t)H * W >= (1u << 30)) return fail(TCLB200_ERR_UNSUPPORTED, "H*W must be below 2^30");
  BwdParams p;
  memset(&p, 0, sizeof(p));
  p.x = prev; p.f = bf; p.mask = mask; p.cur = cur; p.grad_scale = grad_scale; p.scale_mul = scale_mul;
  p.grad_cur = grad_cur;
  p.geo = make_geo(H, W); p.B = B; p.C = C; p.flags = flags & TCLB200_VALIDITY; p.loss = loss;
  const int rc = backward_dtype_setup(p, dtype, grad_prev, workspace, workspace_bytes, "grad_prev");
  if (rc != TCLB200_OK) return rc;
  return run_backward(p, true, dtype, static_cast<__nv_bfloat16*>(grad_prev), reinterpret_cast<cudaStream_t>(stream));
}

extern "C" int tclb200_tcl_backward_scaled(const float* bf, const float* mask, const float* prev, const float* cur,
                                           const float* grad_scale, float scale_mul, float* grad_prev, float* grad_cur, int B, int C,
                                           int H, int W, int flags, int loss, tclb200_stream_t stream) {
  return tclb200_tcl_backward_dt(bf, mask, prev, cur, grad_scale, scale_mul, grad_prev, grad_cur, B, C, H, W, TCLB200_F32, flags, loss,
                                 nullptr, 0, stream);
}

extern "C" int tclb200_tcl_backward(const float* bf, const float* mask, const float* prev, const float* cur,
                                    const float* grad_scale, float* grad_prev, float* grad_cur, int B, int C, int H, int W,
                                    int flags, int loss, tclb200_stream_t stream) {
  return tclb200_tcl_backward_scaled(bf, mask, prev, cur, grad_scale, 1.0f, grad_prev, grad_cur, B, C, H, W, flags, loss, stream);
}

extern "C" int tclb200_hwc_split(const float* src, int N, int H, int W, int Cs, int n_out, float* const* dst, const int* c0,
                                 const int* cd, tclb200_stream_t stream) {
  if (!src || !dst || !c0 || !cd) return fail(TCLB200_ERR_INVALID, "src, dst, c0 and cd are required");
  if (N <= 0 || H <= 0 || W <= 0 || Cs <= 0) return fail(TCLB200_ERR_INVALID, "N, H, W, Cs must be positive");
  if (n_out <= 0 || n_out > kSplitMaxOut) return fail(TCLB200_ERR_INVALID, "n_out must be in 1..8");
  if (Cs > 64) return fail(TCLB200_ERR_UNSUPPORTED, "at most 64 interleaved channels");
  SplitParams p;
  memset(&p, 0, sizeof(p));
  p.src = src; p.n_out = n_out; p.Cs = Cs; p.plane = (long long)H * W;
  for (int i = 0; i < n_out; ++i) {
    if (!dst[i] || c0[i] < 0 || cd[i] <= 0 || c0[i] + cd[i] > Cs) return fail(TCLB200_ERR_INVALID, "bad output channel range");
    p.dst[i] = dst[i]; p.c0[i] = c0[i]; p.cd[i] = cd[i];
  }
  if (Cs == 2 && p.plane % 2 == 0 && aligned16(src)) {   // the .flo layout: vector kernel when every plane start is 8-byte aligned
    Split2Params q;
    memset(&q, 0, sizeof(q));
    q.src = src; q.plane = p.plane; q.pairs = (long long)N * p.plane / 2;
    bool ok = true;
    for (int i = 0; i < n_out; ++i)
      for (int c = c0[i]; c < c0[i] + cd[i]; ++c) {
        if (q.dst[c]) ok = false;   // (a channel requested twice: the general kernel handles it)
        q.dst[c] = dst[i] + (long long)(c - c0[i]) * p.plane;
        q.dstride[c] = (long long)cd[i] * p.plane;
        ok = ok && (reinterpret_cast<uintptr_t>(q.dst[c]) & 7u) == 0;
      }
    const long long blocks = (q.pairs + 4 * 256 - 1) / (4 * 256);
    if (ok && blocks < 0x7fffffffLL) {
      hwc2_split_kernel<<<(unsigned)blocks, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(q);
      ++g_launches;
      CUDA_TRY(cudaGetLastError());
      return TCLB200_OK;
    }
  }
  const long long chunks = (p.plane + kSplitPx - 1) / kSplitPx;
  if (chunks * N >= 0x7fffffffLL) return fail(TCLB200_ERR_UNSUPPORTED, "too many chunks for one launch");
  p.chunks_per_sample = (int)chunks;
  const size_t smem = (size_t)kSplitPx * (Cs | 1) * sizeof(float);
  if (smem > 48 * 1024) {
    CUDA_TRY(cudaFuncSetAttribute(hwc_split_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  }
  hwc_split_kernel<<<(unsigned)(chunks * N), kSplitPx, smem, reinterpret_cast<cudaStream_t>(stream)>>>(p);
  ++g_launches;
  CUDA_TRY(cudaGetLastError());
  return TCLB200_OK;
}

extern "C" int tclb200_upsample_flow(const float* flow, const float* mask, float* out, int N, int H, int W, tclb200_stream_t stream) {
  if (!flow || !mask || !out) return fail(TCLB200_ERR_INVALID, "flow, mask and out are required");
  if (N <= 0 || H <= 0 || W <= 0) return fail(TCLB200_ERR_INVALID, "N, H, W must be positive");
  const long long segs = cdiv(W, kUpW), blocks = segs * H * (long long)N;
  if (blocks >= 0x7fffffffLL) return fail(TCLB200_ERR_UNSUPPORTED, "too many blocks for one launch");
  upsample_flow_kernel<<<(unsigned)blocks, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(flow, mask, out, H, W, (int)segs);
  ++g_launches;
  CUDA_TRY(cudaGetLastError());
  return TCLB200_OK;
}
