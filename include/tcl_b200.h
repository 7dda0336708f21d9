/*
 * tcl_b200.h -- C ABI of the B200-native flow-based temporal-consistency path.
 *
 * Drop-in boundary (SURVEY.md section 8b).  The reference (tomstrident/GAN-based-Video-Style-Transfer) is
 * pure Python; its "FFI" for this path is the module-function API
 *     from flowtools import gradient, warp, fbcCheckTorch        (utils/flowtools.py)
 *     from fs_lib import warp                                     (methods/learning-based/fs_lib.py)
 *     from sintel_eval import computeTCL                          (utils/sintel_eval.py)
 * The thin PyTorch wrappers in gan-based-video-style-transfer_b200/ keep those signatures and bind the
 * entry points below with ctypes (INTEGRATION.md shows the stub).  No torch types cross this
 * boundary: plain device pointers owned by the caller, explicit sizes, an explicit cudaStream_t.
 *
 * Conventions
 *   - all tensors NCHW contiguous; flows are (B,2,H,W) fp32 in pixels, channel 0 = u (x), 1 = v (y);
 *     frames are (B,C,H,W) fp32 or bf16 (TCLB200_F32 / TCLB200_BF16); masks are (B,1,H,W) fp32 in {0,1}
 *   - every function returns 0 on success, a TCLB200_ERR_* code otherwise, never throws or aborts;
 *     tclb200_last_error() returns a thread-local message for the last failing call
 *   - no hidden global state: accumulators and scratch are passed in; calls are asynchronous on
 *     `stream` and re-entrant across streams as long as each stream uses its own scratch
 *   - there is NO CPU fallback: without a CUDA device every compute entry returns TCLB200_ERR_CUDA
 */
#ifndef TCL_B200_H_
#define TCL_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TCLB200_ABI_VERSION 6

#define TCLB200_OK 0
#define TCLB200_ERR_INVALID 1     /* bad argument (null pointer, non-positive size, unknown enum) */
#define TCLB200_ERR_CUDA 2        /* a CUDA runtime call failed; see tclb200_last_error() */
#define TCLB200_ERR_UNSUPPORTED 3 /* valid request this build does not implement */

/* frame dtype */
#define TCLB200_F32 0
#define TCLB200_BF16 1

/* mask tests of fbcCheckTorch (utils/flowtools.py:45,53); the optimisation-based variant
 * (methods/optimization-based/flowtools.py:34-58) is TCLB200_MOB alone */
#define TCLB200_OCC 1
#define TCLB200_MOB 2
/* fs_lib.warp validity mask (methods/learning-based/fs_lib.py:29-39) */
#define TCLB200_VALIDITY 4
/* this launch is one chunk of a longer evaluation: always the persistent pipeline (short launches of the training loss
 * otherwise take a latency-optimised kernel with another, equally fixed, summation tree), so that per-pair values do not
 * depend on how the caller chunked the pairs; set by tclb200_tcl_forward_host for its own launches */
#define TCLB200_THROUGHPUT 8

/* masked error */
#define TCLB200_L2 0 /* sum (m*(cur-warp))^2   solver.py:444, sintel_eval.py:110, metrics/eval.py:138 */
#define TCLB200_L1 1 /* sum  m*|warp-cur|      MoGAN/models/cycle_gan_model.py:280-281 */

/* how pair_vals / total_val are derived from the sums (N = C*H*W) */
#define TCLB200_FIN_MEAN 0 /* pair: S_b/N        total: sum_b S_b/(B*N)        (training loss)       */
#define TCLB200_FIN_RMSE 1 /* pair: sqrt(S_b/N)  total: sqrt(sum_b S_b/(B*N))  (computeTCL, tcl_err) */

typedef void* tclb200_stream_t; /* cudaStream_t */

int tclb200_abi_version(void);
const char* tclb200_last_error(void);
/* the compile-time configuration of this build of the library ("abi=6 th=32 bh=40 ... hot_only=0 diag=0 trace=0"): the
 * wrappers refuse a library built with tuning macros (tools/sweep_build.py) unless it was asked for by name   (ABI v5) */
const char* tclb200_build_info(void);

/* bytes of device scratch tclb200_tcl_forward needs for a (B,H,W) problem.  The scratch must be
 * zero-filled once when allocated; every call leaves it zeroed again. */
size_t tclb200_scratch_bytes(int B, int H, int W);

/* gradient(x)  utils/flowtools.py:12-16
 * x (B,H,W) fp32 -> out (2,B,H,W) fp32 = [d/dx, d/dy], zero-padded central differences. */
int tclb200_gradient(const float* x, float* out, int B, int H, int W, tclb200_stream_t stream);
/* the same on B contiguous (H,W) planes that lie x_batch_stride floats apart: the reference calls gradient(bf[:,0,:,:])
 * and gradient(bf[:,1,:,:]) (utils/flowtools.py:47-48), one channel of a (B,2,H,W) flow -- no gather copy needed. */
int tclb200_gradient_strided(const float* x, size_t x_batch_stride, float* out, int B, int H, int W, tclb200_stream_t stream);

/* warp(x, f)  utils/flowtools.py:18-32 (copies: utils/metrics/eval.py:43-57, StarGAN/solver.py:42-56;
 * inline: StarGANv2AdvCon/core/solver.py:427-443, CycleGANCon/models/cycle_gan_model.py:191-203)
 * flags & TCLB200_VALIDITY selects fs_lib.warp (methods/learning-based/fs_lib.py:5-39).
 * x, out (B,C,H,W) of `dtype`; f (B,2,H,W) fp32. */
int tclb200_warp(const void* x, const float* f, void* out, int B, int C, int H, int W, int dtype, int flags,
                 tclb200_stream_t stream);

/* autograd of warp(): what F.grid_sample's backward + the grid normalisation give the reference
 * (solver.py:181 g_loss.backward()).  grad_out, x as in tclb200_warp (fp32; bf16: tclb200_warp_backward_dt); grad_x (B,C,H,W) fp32 is
 * OVERWRITTEN (zero-filled, then bilinear scatter-add); grad_f (B,2,H,W) fp32.  Either output may be NULL. */
int tclb200_warp_backward(const float* grad_out, const float* x, const float* f, float* grad_x, float* grad_f, int B,
                          int C, int H, int W, int flags, tclb200_stream_t stream);

/* fbcCheckTorch(ff, bf)  utils/flowtools.py:34-58
 * mask_out (B,1,H,W) fp32 in {0,1}.  near_threshold (device, optional) is incremented by the number of
 * pixels whose occlusion or motion-boundary margin |lhs-rhs| is below 1e-6 (north_star's exemption band). */
int tclb200_fbcheck(const float* ff, const float* bf, float* mask_out, int B, int H, int W, int flags,
                    unsigned long long* near_threshold, tclb200_stream_t stream);

/* Fused warp + occlusion mask + masked reduction: one pass that reads each pair's flows and frames once.
 *   computeTCL            utils/sintel_eval.py:104-110   (ff,bf given, mask computed, FIN_RMSE)
 *   FC2 tcl_err           utils/metrics/eval.py:137-138  (mask_in given, per-sample FIN_RMSE)
 *   GAN training loss     StarGANv2AdvCon/core/solver.py:427-446 (mask_in given, FIN_MEAN)
 *   MoGAN masked L1       MoGAN/models/cycle_gan_model.py:276-281 (TCLB200_L1)
 *   warp+mask blend       methods/optimization-based/obst_eval.py:500 (blend_out)
 */
typedef struct tclb200_tcl_args {
  /* inputs (device) */
  const float* ff;      /* (B,2,H,W) forward flow, or NULL when mask_in is given / no mask wanted */
  const float* bf;      /* (B,2,H,W) flow the warp samples with; required */
  const float* mask_in; /* (B,1,H,W) dataset mask, or NULL; ignored when ff is given */
  const void* prev;     /* (B,C,H,W) frame t-1 (stylised), `dtype` */
  const void* cur;      /* (B,C,H,W) frame t, `dtype` */
  /* optional per-pixel outputs (device), NULL to skip */
  void* warp_out;       /* (B,C,H,W) `dtype` */
  float* mask_out;      /* (B,1,H,W) */
  void* blend_out;      /* (B,C,H,W) `dtype`: m*warp + (1-m)*cur */
  /* reductions (device), NULL to skip */
  double* pair_sums;    /* [B]  S_b                                   */
  double* total_sums;   /* [2]  {sum_b S_b, sum_b pair_val_b}          */
  float* pair_vals;     /* [B]  per `finalize`                         */
  float* total_val;     /* [1]  per `finalize`                         */
  unsigned long long* near_threshold; /* [1] += near-threshold pixel count, or NULL */
  void* scratch;        /* >= tclb200_scratch_bytes(B,H,W), zero-filled at allocation */
  size_t scratch_bytes;
  int B, C, H, W;
  int dtype;            /* TCLB200_F32 / TCLB200_BF16 (frames only; flows and masks are fp32) */
  int flags;            /* TCLB200_OCC | TCLB200_MOB tests when ff is given; TCLB200_VALIDITY */
  int loss;             /* TCLB200_L2 / TCLB200_L1 */
  int finalize;         /* TCLB200_FIN_MEAN / TCLB200_FIN_RMSE */
  /* clip mode (optional, NULL = off): `prev` / `cur` hold n_*_frames frames (F,C,H,W) and pair b reads frame
   * prev_index[b] / cur_index[b] (device int32 arrays of B entries, values in [0, n_*_frames)).  A video frame stored
   * once can then be the `cur` of pair t and the `prev` of pair t+1 (utils/sintel_eval.py:206-222 evaluates consecutive
   * frames of a clip): its second read is served by the 126 MB L2 instead of HBM.  Per-pixel outputs stay per pair. */
  const int* prev_index;
  const int* cur_index;
  int n_prev_frames, n_cur_frames;
  /* strided flows (optional, 0 = dense): rows stay dense, but the two components of a flow / consecutive pairs may lie
   * ff_plane_stride / ff_batch_stride (bf_...) floats apart.  That is what the reference hands over: RAFT's output on
   * the /8-padded image cropped by InputPadder.unpad (utils/raft/raft/utils/utils.py:21-24) or flow_up[:,:,:H,:]
   * (methods/GAN-based/ConGAN/sintel_eval.py:61) is such a view -- it is read in place, no gather copy. */
  size_t ff_plane_stride, ff_batch_stride, bf_plane_stride, bf_batch_stride;
  /* window mode (optional, NULL / 0 = off; ABI v5): `bf` / `ff` hold n_bf_fields / n_ff_fields flow fields and pair b reads
   * field bf_index[b] / ff_index[b] (device int32 arrays of B entries).  The evaluations of a temporal window use every
   * field twice -- flow(t -> s) is the `bf` of "warp frame s into t" and the `ff` of "warp frame t into s"
   * (utils/sintel_eval.py:84-86,216-222: long-term pairs of a target frame; BASELINE config 4: 3 source frames x both
   * directions) -- so with clip mode on top a window of 4 frames and 3 flow pairs is stored once and serves 6 evaluations.
   * pair_group > 1 interleaves the tiles of that many consecutive pairs (the evaluations of one target frame), so that
   * their shared `cur` tile, flow tiles and neighbouring source boxes are re-read within microseconds: L2 hits, not HBM. */
  const int* bf_index;
  const int* ff_index;
  int n_bf_fields, n_ff_fields;
  int pair_group;
  /* band mode (optional, 0 / 0 = whole frames; ABI v5): only target rows [row_begin, row_end) of every pair are evaluated
   * (sums, mask_out / warp_out / blend_out rows); the inputs are still whole frames -- the flow gradient reads the rows next
   * to the band and the taps land wherever the flow points.  A job with fewer pairs than GPUs (one 4K pair on eight GPUs,
   * BASELINE config 5) splits every frame into horizontal bands, one per GPU, and adds the bands' pair_sums with the path's
   * one all-reduce.  pair_vals / total_val are refused in this mode (a band's mean is not the frame's). */
  int row_begin, row_end;
} tclb200_tcl_args;

int tclb200_tcl_forward(const tclb200_tcl_args* args, tclb200_stream_t stream);

/* Host-buffer entry: the job of the reference's evaluation loops with the data where those loops hold it -- in HOST
 * memory (utils/sintel_eval.py:206-222 and StarGANv2AdvCon/core/solver.py:336-347 walk a clip frame by frame and pull
 * every pair's value back with .cpu().numpy(); utils/metrics/eval.py:137-149 does the same per FC2 batch).
 * All pointers below are HOST pointers except `workspace` (page-locked memory gives full PCIe speed; pageable works).
 * The call enqueues a software pipeline -- chunks of `chunk_pairs` pairs: H2D of the frames the chunk needs that are
 * not on the device yet (each frame of the bank crosses PCIe once), H2D of its flows into a 3-slot ring on an internal
 * copy stream, one fused launch (clip mode of tclb200_tcl_forward) per chunk on `stream`, one D2H of the per-pair
 * results at the end -- and returns; pair_vals / pair_sums are valid once `stream` has been synchronised, and the host
 * inputs must stay untouched until then. */
typedef struct tclb200_host_args {
  const float* ff;       /* (P,2,H,W) forward flows, or NULL (then mask_in or no mask) */
  const float* bf;       /* (P,2,H,W) flows the warp samples with; required */
  const float* mask_in;  /* (P,1,H,W) dataset masks, or NULL; ignored when ff is given */
  const void* frames;    /* (F,C,H,W) `dtype`: the stylised frames, each stored once */
  const int* prev_index; /* [P] frame warped by pair p's flow, in [0,F) */
  const int* cur_index;  /* [P] frame pair p is compared with */
  float* pair_vals;      /* [P] out, per `finalize`; or NULL */
  double* pair_sums;     /* [P] out, S_p; or NULL */
  void* workspace;       /* DEVICE memory, 256-byte aligned, >= tclb200_host_workspace_bytes(...) */
  size_t workspace_bytes;
  int P, F, C, H, W;
  int dtype, flags, loss, finalize; /* as in tclb200_tcl_args */
  int chunk_pairs;       /* pairs per launch, 0 = as many as make a flow copy of about 256 MB (at most 128) */
  int frame_slots;       /* device frame slots the workspace provides: 0 (or >= F) = the whole bank stays resident; fewer =
                          * a ring -- a slot is reused once every chunk that reads its frame has completed; a window of
                          * (3 + 1) chunks of pairs must fit (TCLB200_ERR_INVALID otherwise)          (ABI v5) */
} tclb200_host_args;

/* F here = the number of device frame slots to provision (tclb200_host_args.frame_slots, or the clip's F for a resident bank) */
size_t tclb200_host_workspace_bytes(int P, int F, int C, int H, int W, int dtype, int chunk_pairs, int with_mask);
int tclb200_tcl_forward_host(const tclb200_host_args* args, tclb200_stream_t stream);

/* Backward of the fused training loss  L = grad_scale * sum (m*(cur-warp(prev,bf)))^2   (L2)
 *                                   or L = grad_scale * sum  m*|warp(prev,bf)-cur|      (L1)
 * (solver.py:444-446 + :181; fs_ruder.py:97-106; MoGAN .. :281,285).  grad_scale is a device scalar
 * (upstream gradient times 1/(B*C*H*W) times lambda).  grad_cur (B,C,H,W) fp32 is written; grad_prev
 * (B,C,H,W) fp32 is OVERWRITTEN with the bilinear scatter-add.  Either may be NULL.  fp32 frames (bf16: tclb200_tcl_backward_dt). */
int tclb200_tcl_backward(const float* bf, const float* mask, const float* prev, const float* cur,
                         const float* grad_scale, float* grad_prev, float* grad_cur, int B, int C, int H, int W,
                         int flags, int loss, tclb200_stream_t stream);
/* The same with a host factor applied to the device scalar inside the kernel (one rounded fp32 product, exactly what
 * `grad_out * (1.0 / N)` gives in torch): the autograd wrapper passes the upstream gradient itself and 1/(B*C*H*W), which
 * saves the one-element multiply launch a mean loss otherwise needs in front of every backward. */
int tclb200_tcl_backward_scaled(const float* bf, const float* mask, const float* prev, const float* cur,
                                const float* grad_scale, float scale_mul, float* grad_prev, float* grad_cur, int B, int C,
                                int H, int W, int flags, int loss, tclb200_stream_t stream);

/* Backward of bf16 frames (ABI v6): the entries above with the frame dtype as an argument.  What they compute is the fp32
 * backward of the upcast frames with each frame gradient rounded to bf16 once (__float2bfloat16_rn, torch's
 * .to(torch.bfloat16)) -- what the reference gives under torch.autocast(..., torch.bfloat16), where grid_sampler runs in
 * fp32 on the upcast frames and autograd casts each frame's gradient back.
 *   x / prev, cur, grad_out, grad_x / grad_prev, grad_cur: `dtype` (TCLB200_F32 / TCLB200_BF16); flows, masks, grad_f and
 *   grad_scale stay fp32.  grad_f and grad_cur are bit for bit the fp32 entries' results on the upcast frames (rounded
 *   for grad_cur); grad_x / grad_prev is scattered into `workspace` as fp32, then rounded into the output by a second
 *   kernel (a bf16 scatter-add would round on every add).
 *   workspace: device memory, 16-byte aligned, >= tclb200_backward_workspace_bytes(B,C,H,W,dtype) bytes; only needed for
 *   bf16 frames with grad_x / grad_prev requested (NULL / 0 otherwise; fp32 frames never use it).  Its contents are
 *   irrelevant; it must stay untouched until the call's work on `stream` has completed.
 *   TCLB200_ERR_INVALID for an unknown dtype or a missing / too small / misaligned workspace, before any CUDA call.
 * With dtype = TCLB200_F32 they are tclb200_warp_backward / tclb200_tcl_backward_scaled. */
size_t tclb200_backward_workspace_bytes(int B, int C, int H, int W, int dtype);  /* 0 for TCLB200_F32 */
int tclb200_warp_backward_dt(const void* grad_out, const void* x, const float* f, void* grad_x, float* grad_f, int B, int C, int H,
                             int W, int dtype, int flags, void* workspace, size_t workspace_bytes, tclb200_stream_t stream);
int tclb200_tcl_backward_dt(const float* bf, const float* mask, const void* prev, const void* cur, const float* grad_scale,
                            float scale_mul, void* grad_prev, void* grad_cur, int B, int C, int H, int W, int dtype, int flags,
                            int loss, void* workspace, size_t workspace_bytes, tclb200_stream_t stream);

/* Dataset ingest ("next" row of the scope table): HWC -> planar NCHW de-interleave on the GPU.
 *   - the 9-channel FlyingChairs2 / Hollywood2 blocks [img1 3 | img2 3 | mask 1 | flow 2]
 *     (StarGANv2AdvCon/core/data_loader.py:243-245, methods/learning-based/datasets.py:52-54: np.moveaxis(np_data[:,:,6:7], 2, 0) ...)
 *   - the payload of a .flo file, H x W x 2 (utils/flowlib.py:33-48 readFlow)
 * src (N,H,W,Cs) fp32; output i, dst[i] (N,cd[i],H,W) fp32, receives channels [c0[i], c0[i]+cd[i]) of src.  The
 * arrays dst / c0 / cd are HOST arrays of n_out <= 8 entries (dst[i] are device pointers). */
int tclb200_hwc_split(const float* src, int N, int H, int W, int Cs, int n_out, float* const* dst, const int* c0,
                      const int* cd, tclb200_stream_t stream);

/* Sintel ground-truth occlusion PNG -> mask (utils/sintel_dataset.py:64-65: mask = 1.0 - imread(png)/255.0 in float64, later
 * .float()): src n bytes (4-byte aligned), dst n floats (16-byte aligned), both device; exact for all 256 inputs. */
int tclb200_occlusion_u8_to_mask(const uint8_t* src, float* dst, size_t n, tclb200_stream_t stream);

/* RAFT's convex 8x upsampling of the coarse flow (utils/raft/raft/raft.py:72-83 upsample_flow), the producer of the
 * flows this path consumes ("next" row of the scope table): softmax over the 9 mask logits, convex combination of the
 * zero-padded 3x3 neighbourhood of 8*flow, pixel shuffle.  flow (N,2,H,W), mask (N,576,H,W) -> out (N,2,8H,8W), fp32. */
int tclb200_upsample_flow(const float* flow, const float* mask, float* out, int N, int H, int W, tclb200_stream_t stream);

/* NumPy / OpenCV flavour of the path ("next" row of the scope table): the reference's dataset generators restate warp and
 * the forward-backward check on HWC arrays with cv2.remap / np.gradient / np.linalg.norm
 * (methods/learning-based/dataset-generation/coco-generation.py:66-113, hollywood2-generation.py:63-111,
 * sintel-generation.py:89-130).  Bit-compatible with OpenCV 4.x's remap(INTER_LINEAR, BORDER_CONSTANT 0) on float32: sample
 * position exactly (x+u, y+v) in 1/32-pixel fixed point, table weights, unfused left-to-right sum.
 *   tclb200_cv2_remap     warp_image / warp_flow: src (N,H,W,C), flow (N,H,W,2) -> out (N,H,W,C), all fp32 HWC
 *   tclb200_cv2_fb_check  fb_check(warp_flow(ff, bf), bf) in one pass (prewarped != 0: ff is already the warped flow, the
 *                         reference's two-argument fb_check); ff, bf (N,H,W,2) -> mask (N,H,W) fp32 in {0,1};
 *                         flags = TCLB200_OCC (the COCO copy, :111 comments the boundary test out) | TCLB200_MOB;
 *                         near_threshold as in tclb200_fbcheck. */
int tclb200_cv2_remap(const float* src, const float* flow, float* out, int N, int H, int W, int C, tclb200_stream_t stream);
int tclb200_cv2_fb_check(const float* ff, const float* bf, float* mask, int N, int H, int W, int flags, int prewarped,
                         unsigned long long* near_threshold, tclb200_stream_t stream);

/* Warp chains of the learning-based trainers ("next" row of the scope table, rank 2), fp32 NCHW, C = 3, device pointers.
 *   tclb200_reconet_loss   ReCoNet's output-level temporal loss, methods/learning-based/fs_reconet.py:63-69:
 *                            mean((mask * ((styled2 - warp(styled1,flow)) - luminance(img2 - warp(img1,flow))))**2)
 *                          with warp = fs_lib.warp (fs_lib.py:5-39); the two warps share the sampling position, weights and
 *                          validity factor of the pixel.  mask (B,1,H,W) or NULL (= ones).  Outputs: loss_out [1] fp32 (the
 *                          mean) and / or sum_out [1] fp64 (the sum of squares); lum_out (B,1,H,W) or NULL receives the
 *                          luminance term (the backward is tclb200_tcl_backward with cur = styled2 - lum, TCLB200_VALIDITY).
 *                          scratch: device memory >= tclb200_reconet_scratch_bytes(B,H,W), contents irrelevant.
 *   tclb200_ruder_input    one step of Ruder's recurrent chain, fs_ruder.py:50-75: cat_out (B,7,H,W) =
 *                          cat((img, mask, warp(styled_prev, flow)), 1) in one pass; warp_out (B,3,H,W) or NULL also receives
 *                          the warped frame (`loss_warped`, fs_ruder.py:97).  mask NULL = ones.                      (ABI v5) */
size_t tclb200_reconet_scratch_bytes(int B, int H, int W);
int tclb200_reconet_loss(const float* flow, const float* mask, const float* styled1, const float* styled2, const float* img1,
                         const float* img2, float* lum_out, float* loss_out, double* sum_out, void* scratch, size_t scratch_bytes,
                         int B, int H, int W, tclb200_stream_t stream);
int tclb200_ruder_input(const float* img, const float* mask, const float* styled_prev, const float* flow, float* cat_out,
                        float* warp_out, int B, int H, int W, tclb200_stream_t stream);

/* Aggregation of the evaluation loop (per-video mean of the per-pair RMSE, StarGANv2AdvCon/core/solver.py:352-354; mean over
 * videos, utils/sintel_eval.py:112-126) around the one all-reduce of the sharded evaluation.  All pointers are device pointers.
 *   pack:   pair_vals [n_pairs] fp32, sum_sq [1] fp64 (sum of squared error of these pairs, or NULL), seq_of_pair [n_pairs] int64
 *           -> packed [2*n_seq + 2] fp64 = { sum of values per sequence | pair count per sequence | sum_sq | n_pairs * elems_per_pair }
 *   unpack: packed (summed over ranks) -> out [n_seq + 4] fp64 = { per-sequence mean ... | mean over sequences that have pairs |
 *           mean over pairs | pooled RMSE | number of pairs } */
int tclb200_pack_sequence_sums(const float* pair_vals, const double* sum_sq, const long long* seq_of_pair, int n_pairs, int n_seq,
                               double elems_per_pair, double* packed, tclb200_stream_t stream);
int tclb200_unpack_sequence_means(const double* packed, int n_seq, double* out, tclb200_stream_t stream);

/* Test hook (process-global, not for production use): pin the forward kernel so that all of them are exercised on the
 * same inputs.  0 = off (default); 1 = the generic global-memory kernel also for TMA-capable shapes; 2 = never the direct
 * kernel of short training-loss launches (always the persistent TMA pipeline); 3 = the direct kernel whatever the size. */
void tclb200_debug_force_generic(int on);

/* Diagnostics (process-global device counters, not for production use): out2[0] = tiles of the TMA kernel that
 * could not stage their source boxes (non-finite or extreme flow) and were gathered from global memory,
 * out2[1] = "mixed" tiles (a motion boundary runs through them: some pixels gathered from global memory).
 * Synchronises the device.  reset != 0 clears the counters afterwards. */
int tclb200_debug_tile_stats(unsigned long long* out2, int reset);

/* Diagnostics: number of kernels this library has launched in this process (the fused TMA path launches two per
 * reducing call: the fused kernel and the fold kernel behind it).  reset != 0 clears the counter. */
unsigned long long tclb200_debug_launch_count(int reset);

#ifdef __cplusplus
}
#endif
#endif /* TCL_B200_H_ */
