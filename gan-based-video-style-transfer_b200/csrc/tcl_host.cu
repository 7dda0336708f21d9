// Host-buffer entry of the C ABI: tclb200_tcl_forward_host (include/tcl_b200.h).
//
// The reference's evaluation loops hold their data on the host side of the boundary: every frame of a clip is loaded,
// stylised and compared pair by pair with a `.cpu().numpy()` per pair (utils/sintel_eval.py:206-222,
// StarGANv2AdvCon/core/solver.py:336-347, utils/metrics/eval.py:137-149).  This entry takes the whole job -- flows,
// the frame bank of the clip(s), which frame each pair warps / compares with -- as HOST pointers and runs it as a
// software pipeline:
//
//   copy streams    chunk k (on copy stream k % 2: two streams keep the link busy across the gaps between one stream's
//                   copies -- with eight ranks sharing one host memory system those gaps are bandwidth nobody else can use):
//                   the frames its pairs need that are not on the device yet (each frame crosses PCIe ONCE: 28 B/px per
//                   pair instead of 40 for a clip of fp32 frames; 19 with uint8 frames), then the two flows of its pairs into ring slot k % 3
//   caller's stream chunk k: one fused launch (tclb200_tcl_forward in clip mode) on that slot, results into the
//                   device result array; after the last chunk one D2H copy of the per-pair results
//
// PCIe is the bound (a 1024x436 pair is 12.5 MB of flows + frames; its kernel time is 4 us): the ring only has to keep
// the copy engine busy.
//
// Device frame slots: the workspace holds `frame_slots` frames (0 = all F of them).  With fewer slots than frames the
// bank becomes a ring: a frame's slot is handed out again once every chunk that reads it has completed (known from the
// flow ring's own events: when chunk k is being staged, chunk k - 3 has finished), so long or 4K clips need device
// memory for a window of frames only -- (3 + 1) chunks' worth -- not for the whole clip.  Pairs reach their frames
// through per-pair slot indices written for each chunk.
//
// Channels-last host data (tclb200_host_args.channels_last): what decoders and .flo readers produce, (F,H,W,C) frames and
// (P,H,W,2) flows, crosses PCIe unchanged (each run of consecutive frames is one contiguous block in either layout) and is
// de-interleaved on the caller's stream right before the fused launch of its chunk:
//   frames  chunk k's runs go into the staging area of ring slot k % 3 (on the copy stream, after the same done[] wait that
//           frees its flow slot); the caller's stream de-interleaves them into their bank slots after ready[].  Chunk k + 3
//           reuses the staging area after done[k % 3], which follows chunk k's conversion and launch; a bank slot is written
//           by the caller's stream behind every launch that could still read its previous frame.
//   flows   the ring slot receives the interleaved chunk; the caller's stream de-interleaves it into ONE planar buffer per
//           field, which the launch reads -- the stream orders convert(k) -> launch(k) -> convert(k + 1).
// The de-interleave permutes elements and nothing else: the fused launches see the planar bank and flows they would
// have seen, chunk for chunk, so the results are bit for bit those of planar inputs.
//
// The copy stream and the events are kept in a per-device pool and reused by later calls (creating a stream and seven
// events costs more than a small job).  On any failure the function drains both streams before it returns, so the
// caller may free or reuse its host buffers as soon as it sees the error.
//
// Kept-pixel sums (tclb200_host_args.pair_kept): each chunk's launch writes its pairs' sums into one device array behind
// the other regions of the workspace, which goes back with one more D2H copy at the end.
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <mutex>
#include <vector>

#include "../../include/tcl_b200.h"

namespace tcl { void set_last_error(const char* msg); }   // tcl_kernels.cu: the message tclb200_last_error() returns

namespace {

constexpr int kRing = 3;
constexpr size_t kDefaultChunkBytes = (size_t)256 << 20;   // default chunk: as many pairs as make one flow copy about this large
constexpr int kMaxDefaultChunk = 128;

inline size_t up256(size_t v) { return (v + 255) & ~(size_t)255; }

constexpr int kClAll = TCLB200_CL_FRAMES | TCLB200_CL_FF | TCLB200_CL_BF;

struct Layout {
  size_t frames, flows[kRing][2], mask[kRing], prev_idx, cur_idx, vals, sums, scratch, scratch_bytes;
  size_t kept;   // pair_kept only (empty otherwise): the per-pair kept-pixel sums
  size_t stage[kRing], planar[2], total;   // channels-last only (empty otherwise): frame staging per ring slot, planar ff / bf
  size_t frame_bytes, flow_bytes, mask_bytes;
  int chunk;
};

// F = device frame slots provisioned; cl = TCLB200_CL_* bits; with_kept: the call sets pair_kept
Layout make_layout(int P, int F, int C, int H, int W, int dtype, int chunk_pairs, bool with_mask, int cl, bool with_kept) {
  Layout L;
  memset(&L, 0, sizeof(L));
  const size_t px = (size_t)H * W;
  // few, large copies keep the link busy (measured, Sintel shape, one GPU: chunks of 16 / 32 / 64 / 128 pairs reach 0.82 /
  // 0.93 / 0.98 / 0.99 of the link's rate); the default is sized in bytes so that 4K pairs do not need a 25 GB ring
  if (chunk_pairs > 0) {
    L.chunk = chunk_pairs;
  } else {
    const size_t by_bytes = kDefaultChunkBytes / (px * 2 * sizeof(float));
    L.chunk = by_bytes < 1 ? 1 : (by_bytes > (size_t)kMaxDefaultChunk ? kMaxDefaultChunk : (int)by_bytes);
  }
  if (L.chunk > P) L.chunk = P;
  L.frame_bytes = px * C * (dtype == TCLB200_U8 ? 1 : dtype == TCLB200_BF16 ? 2 : 4);
  L.flow_bytes = px * 2 * sizeof(float);
  L.mask_bytes = px * sizeof(float);
  size_t o = 0;
  L.frames = o; o += up256(L.frame_bytes * (size_t)F);
  for (int r = 0; r < kRing; ++r) {
    for (int j = 0; j < 2; ++j) { L.flows[r][j] = o; o += up256(L.flow_bytes * (size_t)L.chunk); }
    L.mask[r] = o;
    if (with_mask) o += up256(L.mask_bytes * (size_t)L.chunk);
  }
  L.prev_idx = o; o += up256(sizeof(int) * (size_t)P);
  L.cur_idx = o; o += up256(sizeof(int) * (size_t)P);
  L.vals = o; o += up256(sizeof(float) * (size_t)P);
  L.sums = o; o += up256(sizeof(double) * (size_t)P);
  L.scratch_bytes = with_kept ? tclb200_scratch_bytes_kept(L.chunk, H, W) : tclb200_scratch_bytes(L.chunk, H, W);
  L.scratch = o; o += up256(L.scratch_bytes);
  // a chunk of n pairs uploads at most 2n frames, and never more than there are slots
  const size_t stage_frames = (cl & TCLB200_CL_FRAMES) ? (size_t)(F < 2 * L.chunk ? F : 2 * L.chunk) : 0;
  for (int r = 0; r < kRing; ++r) { L.stage[r] = o; o += up256(L.frame_bytes * stage_frames); }
  for (int j = 0; j < 2; ++j) {
    L.planar[j] = o;
    if (cl & (j == 0 ? TCLB200_CL_FF : TCLB200_CL_BF)) o += up256(L.flow_bytes * (size_t)L.chunk);
  }
  L.kept = o;
  if (with_kept) o += up256(sizeof(double) * (size_t)P);
  L.total = o;
  return L;
}

int hfail(int code, const char* what, const char* detail = "") {
  char msg[512];
  snprintf(msg, sizeof(msg), "%s%s", what, detail);
  tcl::set_last_error(msg);
  return code;
}

// copy stream + ring events of one call in flight; pooled per device and reused (never destroyed: process lifetime)
struct Pipe {
  cudaStream_t copy[2] = {nullptr, nullptr};
  cudaEvent_t ready[kRing] = {}, done[kRing] = {}, fork = nullptr;
  int device = -1;
  cudaError_t init() {
    cudaError_t e;
    for (int i = 0; i < 2; ++i)
      if ((e = cudaStreamCreateWithFlags(&copy[i], cudaStreamNonBlocking)) != cudaSuccess) return e;
    for (int i = 0; i < kRing; ++i) {
      if ((e = cudaEventCreateWithFlags(&ready[i], cudaEventDisableTiming)) != cudaSuccess) return e;
      if ((e = cudaEventCreateWithFlags(&done[i], cudaEventDisableTiming)) != cudaSuccess) return e;
    }
    return cudaEventCreateWithFlags(&fork, cudaEventDisableTiming);
  }
  void destroy() {
    for (int i = 0; i < kRing; ++i) {
      if (ready[i]) cudaEventDestroy(ready[i]);
      if (done[i]) cudaEventDestroy(done[i]);
    }
    if (fork) cudaEventDestroy(fork);
    for (int i = 0; i < 2; ++i)
      if (copy[i]) cudaStreamDestroy(copy[i]);
  }
};

std::mutex g_pool_mutex;
std::vector<Pipe*> g_pool;   // idle pipes of all devices

Pipe* acquire_pipe(cudaError_t* err) {
  int dev = 0;
  if ((*err = cudaGetDevice(&dev)) != cudaSuccess) return nullptr;
  {
    std::lock_guard<std::mutex> lock(g_pool_mutex);
    for (size_t i = 0; i < g_pool.size(); ++i)
      if (g_pool[i]->device == dev) {
        Pipe* p = g_pool[i];
        g_pool.erase(g_pool.begin() + (long)i);
        return p;
      }
  }
  Pipe* p = new Pipe();
  p->device = dev;
  if ((*err = p->init()) != cudaSuccess) { p->destroy(); delete p; return nullptr; }
  return p;
}

void release_pipe(Pipe* p) {
  std::lock_guard<std::mutex> lock(g_pool_mutex);
  g_pool.push_back(p);
}

// (N,H,W,C) -> (N,C,H,W) for 1- and 2-byte elements (uint8 frames; bf16 frames as their bit patterns): hwc_split_kernel's
// scheme.  A CTA reads the interleaved elements of kDeintPx consecutive pixels of one frame as one contiguous, coalesced
// run into shared memory (one word per element, pitch C | 1: conflict-free for any C), then writes each channel as a
// coalesced run of its plane.  Element-wise accesses: any H, W and any start address work (staged runs start wherever the
// previous run ended).
constexpr int kDeintPx = 256;
constexpr int kDeintMaxC = 64;

template <typename T>
__global__ void __launch_bounds__(kDeintPx) hwc_to_chw_kernel(const T* __restrict__ src, T* __restrict__ dst, int C,
                                                               long long plane, int chunks_per_frame) {
  extern __shared__ uint32_t s_el[];
  const int pitch = C | 1;
  const int n = blockIdx.x / chunks_per_frame;
  const long long px0 = (long long)(blockIdx.x - n * chunks_per_frame) * kDeintPx;
  const int npx = (int)min((long long)kDeintPx, plane - px0);
  const T* s = src + ((long long)n * plane + px0) * C;
  const int nel = npx * C;
  for (int i = threadIdx.x; i < nel; i += kDeintPx) {
    const int px = i / C, c = i - px * C;
    s_el[px * pitch + c] = __ldcs(s + i);
  }
  __syncthreads();
  const int t = threadIdx.x;
  if (t >= npx) return;
  T* d = dst + (long long)n * C * plane + px0 + t;
  for (int c = 0; c < C; ++c) __stcs(d + (long long)c * plane, (T)s_el[t * pitch + c]);
}

// N frames (N,H,W,C) of `dtype` at src -> N planar frames (N,C,H,W) at dst, on `s`.  fp32 goes through tclb200_hwc_split.
int frames_to_planar(const void* src, void* dst, int N, int C, int H, int W, int dtype, cudaStream_t s) {
  if (dtype == TCLB200_F32) {
    float* d = reinterpret_cast<float*>(dst);
    const int c0 = 0;
    return tclb200_hwc_split(reinterpret_cast<const float*>(src), N, H, W, C, 1, &d, &c0, &C, s);
  }
  const long long plane = (long long)H * W, chunks = (plane + kDeintPx - 1) / kDeintPx;
  if (chunks * N >= 0x7fffffffLL) return hfail(TCLB200_ERR_UNSUPPORTED, "channels-last frames: too many pixels for one launch");
  const size_t smem = (size_t)kDeintPx * (C | 1) * sizeof(uint32_t);
  const dim3 grid((unsigned)(chunks * N));
  cudaError_t e;
  if (dtype == TCLB200_U8) {
    if (smem > 48 * 1024 &&
        (e = cudaFuncSetAttribute(hwc_to_chw_kernel<uint8_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)) != cudaSuccess)
      return hfail(TCLB200_ERR_CUDA, "channels-last frames: ", cudaGetErrorString(e));
    hwc_to_chw_kernel<uint8_t><<<grid, kDeintPx, smem, s>>>(reinterpret_cast<const uint8_t*>(src), reinterpret_cast<uint8_t*>(dst),
                                                             C, plane, (int)chunks);
  } else {
    if (smem > 48 * 1024 &&
        (e = cudaFuncSetAttribute(hwc_to_chw_kernel<uint16_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)) != cudaSuccess)
      return hfail(TCLB200_ERR_CUDA, "channels-last frames: ", cudaGetErrorString(e));
    hwc_to_chw_kernel<uint16_t><<<grid, kDeintPx, smem, s>>>(reinterpret_cast<const uint16_t*>(src), reinterpret_cast<uint16_t*>(dst),
                                                              C, plane, (int)chunks);
  }
  if ((e = cudaGetLastError()) != cudaSuccess) return hfail(TCLB200_ERR_CUDA, "channels-last frames: ", cudaGetErrorString(e));
  return TCLB200_OK;
}

}  // namespace

extern "C" size_t tclb200_host_workspace_bytes(int P, int F, int C, int H, int W, int dtype, int chunk_pairs, int with_mask) {
  return tclb200_host_workspace_bytes_cl(P, F, C, H, W, dtype, chunk_pairs, with_mask, 0);
}

extern "C" size_t tclb200_host_workspace_bytes_cl(int P, int F, int C, int H, int W, int dtype, int chunk_pairs, int with_mask,
                                                  int channels_last) {
  if (P <= 0 || F <= 0 || C <= 0 || H <= 0 || W <= 0 || (channels_last & ~kClAll)) return 0;
  return make_layout(P, F, C, H, W, dtype, chunk_pairs, with_mask != 0, channels_last, false).total;
}

extern "C" size_t tclb200_host_workspace_bytes_kept(int P, int F, int C, int H, int W, int dtype, int chunk_pairs, int with_mask,
                                                    int channels_last) {
  if (P <= 0 || F <= 0 || C <= 0 || H <= 0 || W <= 0 || (channels_last & ~kClAll)) return 0;
  return make_layout(P, F, C, H, W, dtype, chunk_pairs, with_mask != 0, channels_last, true).total;
}

// on failure: drain both streams (the caller may free its host buffers when it sees the error), give the pipe back
#define HOST_TRY(expr)                                                                         \
  do {                                                                                         \
    cudaError_t e__ = (expr);                                                                  \
    if (e__ != cudaSuccess) return bail(hfail(TCLB200_ERR_CUDA, #expr ": ", cudaGetErrorString(e__))); \
  } while (0)

extern "C" int tclb200_tcl_forward_host(const tclb200_host_args* a, tclb200_stream_t stream) {
  if (!a) return hfail(TCLB200_ERR_INVALID, "args is NULL");
  if (a->channels_last & ~kClAll) return hfail(TCLB200_ERR_INVALID, "channels_last: unknown bits (TCLB200_CL_FRAMES | TCLB200_CL_FF | TCLB200_CL_BF)");
  if (a->P < 0 || a->F < 0) return hfail(TCLB200_ERR_INVALID, "P and F must not be negative");
  if (a->P == 0) return TCLB200_OK;   // a clip of one frame has no pairs: nothing to do, nothing to return
  if (a->F <= 0 || a->C <= 0 || a->H <= 0 || a->W <= 0) return hfail(TCLB200_ERR_INVALID, "F, C, H, W must be positive");
  if (!a->bf || !a->frames || !a->prev_index || !a->cur_index) return hfail(TCLB200_ERR_INVALID, "bf, frames, prev_index and cur_index are required");
  if (!a->pair_vals && !a->pair_sums && !a->pair_kept)
    return hfail(TCLB200_ERR_INVALID, "nothing to return: pair_vals, pair_sums and pair_kept are all NULL");
  if (a->dtype != TCLB200_F32 && a->dtype != TCLB200_BF16 && a->dtype != TCLB200_U8) return hfail(TCLB200_ERR_INVALID, "unknown dtype");
  if (a->dtype == TCLB200_U8) {   // (the fused launches check the same; here nothing has been enqueued yet)
    if (a->C != 3) return hfail(TCLB200_ERR_INVALID, "uint8 frames must have C == 3");
    for (int c = 0; c < 3; ++c)
      if (!isfinite(a->u8_scale[c]) || !isfinite(a->u8_offset[c])) return hfail(TCLB200_ERR_INVALID, "uint8 frames: u8_scale / u8_offset must be finite");
  }
  if (a->frame_slots < 0) return hfail(TCLB200_ERR_INVALID, "frame_slots must not be negative");
  const int cl = a->channels_last;
  if ((cl & TCLB200_CL_FF) && !a->ff) return hfail(TCLB200_ERR_INVALID, "TCLB200_CL_FF without ff");
  if ((cl & TCLB200_CL_FRAMES) && a->C > kDeintMaxC) return hfail(TCLB200_ERR_UNSUPPORTED, "channels-last frames: at most 64 channels");
  for (int p = 0; p < a->P; ++p)
    if (a->prev_index[p] < 0 || a->prev_index[p] >= a->F || a->cur_index[p] < 0 || a->cur_index[p] >= a->F)
      return hfail(TCLB200_ERR_INVALID, "prev_index / cur_index outside [0, F)");
  const bool with_mask = !a->ff && a->mask_in;
  const int S = (a->frame_slots > 0 && a->frame_slots < a->F) ? a->frame_slots : a->F;   // device frame slots
  const bool with_kept = a->pair_kept != nullptr;
  const Layout L = make_layout(a->P, S, a->C, a->H, a->W, a->dtype, a->chunk_pairs, with_mask, cl, with_kept);
  if (!a->workspace || a->workspace_bytes < L.total)
    return hfail(TCLB200_ERR_INVALID, with_kept ? "workspace missing or smaller than tclb200_host_workspace_bytes_kept()"
                                                : "workspace missing or smaller than tclb200_host_workspace_bytes_cl()");
  if ((reinterpret_cast<uintptr_t>(a->workspace) & 255u) != 0) return hfail(TCLB200_ERR_INVALID, "workspace must be 256-byte aligned");

  cudaStream_t comp = reinterpret_cast<cudaStream_t>(stream);
  char* ws = reinterpret_cast<char*>(a->workspace);
  cudaError_t perr = cudaSuccess;
  Pipe* pipe = acquire_pipe(&perr);
  if (!pipe) return hfail(TCLB200_ERR_CUDA, "copy stream / events: ", cudaGetErrorString(perr));
  auto bail = [&](int rc) {
    cudaStreamSynchronize(pipe->copy[0]);
    cudaStreamSynchronize(pipe->copy[1]);
    cudaStreamSynchronize(comp);
    release_pipe(pipe);
    return rc;
  };
  // frame -> device slot; a slot is free again once the last chunk that reads its frame has completed.  The whole schedule
  // (which frames every chunk uploads into which slots, every pair's slot indices) depends on the pair order alone, so it is
  // worked out on the host first and the index arrays go up in ONE copy before the pipeline starts: an asynchronous copy from
  // pageable memory synchronises its stream first, and one such copy per chunk would drain the copy stream at every chunk
  // boundary (measured with eight ranks: 185 of the 232 GB/s the box's host side can feed).
  const int n_chunks = (a->P + L.chunk - 1) / L.chunk;
  std::vector<int> slot_of((size_t)a->F, -1), last_use((size_t)a->F, -1), free_slots, h_idx(2 * (size_t)a->P);
  int* h_prev = h_idx.data();
  int* h_cur = h_idx.data() + a->P;
  std::vector<std::vector<int>> dies((size_t)n_chunks);   // frames whose last reader is chunk k
  struct Run { int frame, slot, count; };
  std::vector<std::vector<Run>> uploads((size_t)n_chunks);
  for (int p = 0; p < a->P; ++p) { last_use[(size_t)a->prev_index[p]] = p / L.chunk; last_use[(size_t)a->cur_index[p]] = p / L.chunk; }
  for (int f = 0; f < a->F; ++f) if (last_use[(size_t)f] >= 0) dies[(size_t)last_use[(size_t)f]].push_back(f);
  free_slots.reserve((size_t)S);
  for (int i = S - 1; i >= 0; --i) free_slots.push_back(i);   // handed out in increasing order: consecutive frames, consecutive slots
  {
    int released = 0;   // chunks whose frames have been released
    std::vector<int> want;
    for (int s = 0, k = 0; s < a->P; s += L.chunk, ++k) {
      const int n = a->P - s < L.chunk ? a->P - s : L.chunk;
      if (k >= kRing)     // when chunk k is staged, chunk k - kRing has been consumed: the frames nobody reads after it are free
        for (; released <= k - kRing; ++released)
          for (int f : dies[(size_t)released]) { free_slots.push_back(slot_of[(size_t)f]); slot_of[(size_t)f] = -1; }
      want.clear();
      for (int p = s; p < s + n; ++p) {
        const int f2[2] = {a->prev_index[p], a->cur_index[p]};
        for (int j = 0; j < 2; ++j)
          if (slot_of[(size_t)f2[j]] < 0) {
            if (free_slots.empty()) {
              release_pipe(pipe);
              return hfail(TCLB200_ERR_INVALID, "frame_slots too small: a window of (3 + 1) chunks of pairs must fit the device frame ring");
            }
            slot_of[(size_t)f2[j]] = free_slots.back(); free_slots.pop_back();
            want.push_back(f2[j]);
          }
        h_prev[p] = slot_of[(size_t)f2[0]]; h_cur[p] = slot_of[(size_t)f2[1]];
      }
      // runs of consecutive frames in consecutive slots go as one copy
      for (size_t i = 0; i < want.size();) {
        size_t j = i + 1;
        while (j < want.size() && want[j] == want[j - 1] + 1 && slot_of[(size_t)want[j]] == slot_of[(size_t)want[j - 1]] + 1) ++j;
        uploads[(size_t)k].push_back(Run{want[i], slot_of[(size_t)want[i]], (int)(j - i)});
        i = j;
      }
    }
  }
  // the workspace may still be in use by earlier work on the caller's stream
  HOST_TRY(cudaEventRecord(pipe->fork, comp));
  HOST_TRY(cudaStreamWaitEvent(pipe->copy[0], pipe->fork, 0));
  HOST_TRY(cudaStreamWaitEvent(pipe->copy[1], pipe->fork, 0));
  HOST_TRY(cudaMemsetAsync(ws + L.scratch, 0, L.scratch_bytes, comp));
  HOST_TRY(cudaMemcpyAsync(ws + L.prev_idx, h_prev, sizeof(int) * (size_t)a->P, cudaMemcpyHostToDevice, comp));
  HOST_TRY(cudaMemcpyAsync(ws + L.cur_idx, h_cur, sizeof(int) * (size_t)a->P, cudaMemcpyHostToDevice, comp));

  const char* h_frames = reinterpret_cast<const char*>(a->frames);
  for (int s = 0, k = 0; s < a->P; s += L.chunk, ++k) {
    const int n = a->P - s < L.chunk ? a->P - s : L.chunk;
    const int slot = k % kRing;
    cudaStream_t cs = pipe->copy[k & 1];
    if (k >= kRing) HOST_TRY(cudaStreamWaitEvent(cs, pipe->done[slot], 0));   // chunk k - kRing has been consumed: its flow slot and the frame slots released with it are free
    size_t staged = 0;   // channels-last frames: runs go one after another into the slot's staging area
    for (const Run& r : uploads[(size_t)k]) {
      char* dst = (cl & TCLB200_CL_FRAMES) ? ws + L.stage[slot] + staged : ws + L.frames + (size_t)r.slot * L.frame_bytes;
      HOST_TRY(cudaMemcpyAsync(dst, h_frames + (size_t)r.frame * L.frame_bytes, (size_t)r.count * L.frame_bytes, cudaMemcpyHostToDevice, cs));
      staged += (size_t)r.count * L.frame_bytes;
    }
    if (a->ff) HOST_TRY(cudaMemcpyAsync(ws + L.flows[slot][0], a->ff + (size_t)s * 2 * a->H * a->W, (size_t)n * L.flow_bytes, cudaMemcpyHostToDevice, cs));
    HOST_TRY(cudaMemcpyAsync(ws + L.flows[slot][1], a->bf + (size_t)s * 2 * a->H * a->W, (size_t)n * L.flow_bytes, cudaMemcpyHostToDevice, cs));
    if (with_mask) HOST_TRY(cudaMemcpyAsync(ws + L.mask[slot], a->mask_in + (size_t)s * a->H * a->W, (size_t)n * L.mask_bytes, cudaMemcpyHostToDevice, cs));
    HOST_TRY(cudaEventRecord(pipe->ready[slot], cs));
    HOST_TRY(cudaStreamWaitEvent(comp, pipe->ready[slot], 0));

    if (cl & TCLB200_CL_FRAMES) {
      staged = 0;
      for (const Run& r : uploads[(size_t)k]) {
        const int rc = frames_to_planar(ws + L.stage[slot] + staged, ws + L.frames + (size_t)r.slot * L.frame_bytes, r.count, a->C,
                                        a->H, a->W, a->dtype, comp);
        if (rc != TCLB200_OK) return bail(rc);
        staged += (size_t)r.count * L.frame_bytes;
      }
    }
    const float* flow[2] = {reinterpret_cast<const float*>(ws + L.flows[slot][0]), reinterpret_cast<const float*>(ws + L.flows[slot][1])};
    for (int j = 0; j < 2; ++j)
      if (cl & (j == 0 ? TCLB200_CL_FF : TCLB200_CL_BF)) {
        float* planar = reinterpret_cast<float*>(ws + L.planar[j]);
        const int c0 = 0, cd = 2;
        const int rc = tclb200_hwc_split(flow[j], n, a->H, a->W, 2, 1, &planar, &c0, &cd, stream);
        if (rc != TCLB200_OK) return bail(rc);
        flow[j] = planar;
      }

    tclb200_tcl_args t;
    memset(&t, 0, sizeof(t));
    t.ff = a->ff ? flow[0] : nullptr;
    t.bf = flow[1];
    t.mask_in = with_mask ? reinterpret_cast<const float*>(ws + L.mask[slot]) : nullptr;
    t.prev = ws + L.frames; t.cur = ws + L.frames;
    t.prev_index = reinterpret_cast<const int*>(ws + L.prev_idx) + s;
    t.cur_index = reinterpret_cast<const int*>(ws + L.cur_idx) + s;
    t.n_prev_frames = S; t.n_cur_frames = S;
    t.pair_vals = reinterpret_cast<float*>(ws + L.vals) + s;
    t.pair_sums = reinterpret_cast<double*>(ws + L.sums) + s;
    if (with_kept) t.pair_kept = reinterpret_cast<double*>(ws + L.kept) + s;
    t.scratch = ws + L.scratch; t.scratch_bytes = L.scratch_bytes;
    t.B = n; t.C = a->C; t.H = a->H; t.W = a->W;
    t.dtype = a->dtype; t.flags = a->flags | TCLB200_THROUGHPUT; t.loss = a->loss; t.finalize = a->finalize;
    memcpy(t.u8_scale, a->u8_scale, sizeof(t.u8_scale)); memcpy(t.u8_offset, a->u8_offset, sizeof(t.u8_offset));
    const int rc = tclb200_tcl_forward(&t, stream);
    if (rc != TCLB200_OK) return bail(rc);   // tclb200_last_error() already holds the message
    HOST_TRY(cudaEventRecord(pipe->done[slot], comp));
  }
  if (a->pair_vals) HOST_TRY(cudaMemcpyAsync(a->pair_vals, ws + L.vals, sizeof(float) * (size_t)a->P, cudaMemcpyDeviceToHost, comp));
  if (a->pair_sums) HOST_TRY(cudaMemcpyAsync(a->pair_sums, ws + L.sums, sizeof(double) * (size_t)a->P, cudaMemcpyDeviceToHost, comp));
  if (with_kept) HOST_TRY(cudaMemcpyAsync(a->pair_kept, ws + L.kept, sizeof(double) * (size_t)a->P, cudaMemcpyDeviceToHost, comp));
  // the pipe goes back to the pool once its last use (the final ready event the caller's stream waits for) is enqueued;
  // a later call's work on the copy stream is ordered behind this call's by the stream itself
  release_pipe(pipe);
  return TCLB200_OK;
}
