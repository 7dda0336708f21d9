"""Sharding of frame pairs over the GPUs of one box + the single sum all-reduce (SURVEY.md section 8e).

``pack_local`` / ``unpack`` also accept CPU tensors and then do the same fp64 arithmetic with torch ops: that branch is host
logic of the aggregation (a few dozen numbers), exercised by the world-size-2 gloo tests on the GPU-less build box; it is not
a CPU path of the warp / mask / error computation -- there is none.

Pairs are independent (each reads only its own two flows and two frames), so the path shards by
pair with no data-path collective.  The only cross-GPU step is the final aggregation of the
reference's evaluation loop (per-video mean of per-pair RMSE, then the mean over videos:
StarGANv2AdvCon/core/solver.py:352-354, utils/sintel_eval.py:112-126): ONE ``all_reduce(SUM)`` of a
packed float64 vector ``[sum_rmse per sequence | pair count per sequence | sum of squared error | element count]``.
One process per GPU; ``torch.distributed`` (NCCL over NVLink on the GPU box, gloo in CPU tests).
"""
from dataclasses import dataclass
from typing import List, Optional, Sequence

import torch
import torch.distributed as dist


@dataclass
class ShardPlan:
    rank: int
    world: int
    start: int  # first global pair index owned by this rank
    stop: int   # one past the last
    seq_of_pair: List[int]  # sequence id of each LOCAL pair

    @property
    def n_local(self):
        return self.stop - self.start


def pairs_per_sequence(frames_per_sequence: Sequence[int], gap: int = 1) -> List[int]:
    """Number of (t-gap, t) pairs each clip yields: short-term gap=1, long-term gap=5 (utils/sintel_eval.py:63)."""
    return [max(0, n - gap) for n in frames_per_sequence]


def plan_shards(pairs_in_sequence: Sequence[int], world: int, rank: int) -> ShardPlan:
    """Contiguous, balanced blocks of pairs; a clip's pairs stay on one GPU where the split allows."""
    if not (0 <= rank < world):
        raise ValueError(f"rank {rank} outside world of {world}")
    total = sum(pairs_in_sequence)
    base, rem = divmod(total, world)
    start = rank * base + min(rank, rem)
    stop = start + base + (1 if rank < rem else 0)
    seq_of_pair, g = [], 0
    for s, n in enumerate(pairs_in_sequence):
        lo, hi = max(g, start), min(g + n, stop)
        seq_of_pair.extend([s] * max(0, hi - lo))
        g += n
    return ShardPlan(rank, world, start, stop, seq_of_pair)


def pack_local(pair_vals: torch.Tensor, sum_sq: torch.Tensor, seq_of_pair: torch.Tensor, n_seq: int,
               elems_per_pair: int) -> torch.Tensor:
    """Local contribution to the packed vector (float64, on the tensors' device).  CUDA tensors: one launch of
    ``tclb200_pack_sequence_sums``; CPU tensors (the gloo tests of the host logic): the same arithmetic as torch ops."""
    n = pair_vals.numel()
    if pair_vals.is_cuda:
        import ctypes
        from . import _cabi
        packed = torch.empty(2 * n_seq + 2, dtype=torch.float64, device=pair_vals.device)
        # (the evaluation calls this every step with tensors that already have the right form: no copies, no dispatcher calls then)
        vals = pair_vals if (pair_vals.dtype == torch.float32 and pair_vals.is_contiguous()) else pair_vals.float().contiguous()
        seq = seq_of_pair if (seq_of_pair.dtype == torch.long and seq_of_pair.device == pair_vals.device and seq_of_pair.is_contiguous()) \
            else seq_of_pair.to(device=pair_vals.device, dtype=torch.long).contiguous()
        if not n:
            ssq = None
        elif sum_sq.dtype == torch.float64 and sum_sq.is_contiguous():
            ssq = sum_sq          # (one element: a 0-dim tensor or a view of the launch's total_sums)
        else:
            ssq = sum_sq.double().reshape(1).contiguous()
        ptr = lambda t: ctypes.c_void_p(t.data_ptr()) if t is not None else None
        with torch.cuda.device(pair_vals.device):
            _cabi.check(_cabi.lib().tclb200_pack_sequence_sums(ptr(vals), ptr(ssq), ptr(seq), n, n_seq, float(elems_per_pair), ptr(packed),
                                                               ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)))
        return packed
    packed = torch.zeros(2 * n_seq + 2, dtype=torch.float64, device=pair_vals.device)
    if n:
        packed[:n_seq].index_add_(0, seq_of_pair, pair_vals.double())
        packed[n_seq:2 * n_seq].index_add_(0, seq_of_pair, torch.ones(n, dtype=torch.float64, device=pair_vals.device))
        packed[2 * n_seq] = sum_sq.double().reshape(())
    packed[2 * n_seq + 1] = float(n) * float(elems_per_pair)
    return packed


def allreduce_sums(packed: torch.Tensor, group: Optional[dist.ProcessGroup] = None) -> torch.Tensor:
    """The path's single collective; a no-op when not running distributed."""
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(packed, op=dist.ReduceOp.SUM, group=group)
    return packed


def unpack(packed: torch.Tensor, n_seq: int) -> dict:
    """Per-sequence mean RMSE, the reference's mean over sequences, pooled RMSE. Device tensors, no sync.
    CUDA: one launch of ``tclb200_unpack_sequence_means``; CPU (gloo tests): torch ops."""
    if packed.is_cuda:
        import ctypes
        from . import _cabi
        packed = packed.contiguous()
        out = torch.empty(n_seq + 4, dtype=torch.float64, device=packed.device)
        with torch.cuda.device(packed.device):
            _cabi.check(_cabi.lib().tclb200_unpack_sequence_means(ctypes.c_void_p(packed.data_ptr()), n_seq, ctypes.c_void_p(out.data_ptr()),
                                                                  ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)))
        return {"per_sequence_mean": out[:n_seq], "mean_over_sequences": out[n_seq], "mean_over_pairs": out[n_seq + 1],
                "pooled_rmse": out[n_seq + 2], "n_pairs": out[n_seq + 3]}
    sums, cnt = packed[:n_seq], packed[n_seq:2 * n_seq]
    per_seq = sums / cnt.clamp(min=1.0)
    present = (cnt > 0).double()
    return {
        "per_sequence_mean": per_seq,
        "mean_over_sequences": (per_seq * present).sum() / present.sum().clamp(min=1.0),
        "mean_over_pairs": sums.sum() / cnt.sum().clamp(min=1.0),
        "pooled_rmse": (packed[2 * n_seq] / packed[2 * n_seq + 1].clamp(min=1.0)).sqrt(),
        "n_pairs": cnt.sum(),
    }


def evaluate_sharded(ff, bf, prev, cur, seq_of_pair: torch.Tensor, n_seq: int,
                     group: Optional[dist.ProcessGroup] = None, chunk: Optional[int] = None, kernel_events=None,
                     u8_scale=None, u8_offset=None) -> dict:
    """Temporal error of this rank's shard of pairs (already resident on its GPU) + the one all-reduce.

    ``chunk`` bounds the pairs per launch (None = one launch for the shard).  Returns ``unpack``'s dict.
    ``kernel_events``: optional list; a (start, end) pair of CUDA timing events recorded around every fused launch is
    appended to it (bench.py times the dominant kernel inside its timed region this way).
    uint8 frames: ``u8_scale`` / ``u8_offset`` as in ``ops.fused_forward`` (here and in the two functions below).
    """
    from . import ops
    n = bf.shape[0]
    C, H, W = prev.shape[1:]
    if n == 0:
        packed = torch.zeros(2 * n_seq + 2, dtype=torch.float64, device=seq_of_pair.device)
    else:
        step = n if not chunk else chunk
        packed = None
        for s in range(0, n, step):
            e = min(n, s + step)
            if kernel_events is not None:
                ev = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
                ev[0].record()
            res = ops.fused_forward(bf[s:e], prev[s:e], cur[s:e], ff=ff[s:e], finalize=ops.FIN_RMSE, u8_scale=u8_scale,
                                    u8_offset=u8_offset)
            if kernel_events is not None:
                ev[1].record()
                kernel_events.append(ev)
            part = pack_local(res.pair_vals, res.total_sums[0], seq_of_pair[s:e], n_seq, C * H * W)
            packed = part if packed is None else packed + part
    return unpack(allreduce_sums(packed, group), n_seq)


def band_rows(H: int, world: int, rank: int, align: int = 32):
    """Rows [r0, r1) of an H-row frame that ``rank`` of ``world`` evaluates: contiguous bands of whole 32-row tile rows,
    balanced to within one tile row (the last band takes the frame's ragged end; a band may be empty when world > H/32)."""
    blocks = (H + align - 1) // align
    base, rem = divmod(blocks, world)
    b0 = rank * base + min(rank, rem)
    b1 = b0 + base + (1 if rank < rem else 0)
    return min(H, b0 * align), min(H, b1 * align)


def evaluate_banded(ff, bf, prev, cur, group: Optional[dist.ProcessGroup] = None, rank: Optional[int] = None,
                    world: Optional[int] = None, u8_scale=None, u8_offset=None) -> dict:
    """Fewer pairs than GPUs (one 4K pair on eight GPUs, BASELINE config 5; SURVEY.md section 8e): every rank holds the same
    whole pairs, evaluates one horizontal band of target rows of each (the flow gradient and the bilinear taps read beyond
    the band: the inputs are replicated, nothing is exchanged), and the bands' fp64 sums of squares are added with the path's
    one all-reduce.  Returns ``pair_sums`` (B,) fp64 and ``pair_rmse`` (B,) fp32, identical on every rank."""
    from . import ops
    if world is None:
        world = dist.get_world_size(group) if dist.is_available() and dist.is_initialized() else 1
    if rank is None:
        rank = dist.get_rank(group) if dist.is_available() and dist.is_initialized() else 0
    B, _, H, W = bf.shape
    C = prev.shape[1]
    r0, r1 = band_rows(H, world, rank)
    if r1 > r0:
        sums = ops.fused_forward(bf, prev, cur, ff=ff, rows=(r0, r1), u8_scale=u8_scale, u8_offset=u8_offset).pair_sums.clone()
    else:
        sums = torch.zeros(B, dtype=torch.float64, device=bf.device)
    sums = allreduce_sums(sums, group)
    return {"pair_sums": sums, "pair_rmse": (sums / float(C * H * W)).sqrt().float(), "rows": (r0, r1)}


def evaluate_sharded_host(frames, ff, bf, prev_index, cur_index, seq_of_pair, n_seq: int,
                          group: Optional[dist.ProcessGroup] = None, device=None, chunk_pairs: int = 0, u8_scale=None,
                          u8_offset=None) -> dict:
    """The same evaluation with this rank's shard in HOST memory (``ops.temporal_error_host``: frames of the rank's clips
    stored once, pairs index them) + the one all-reduce.  ``seq_of_pair``: sequence id of each local pair (CPU or CUDA
    long tensor).  Returns ``unpack``'s dict of device tensors."""
    from . import ops
    dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    P = bf.shape[0]
    C, H, W = frames.shape[1:]
    if P == 0:
        packed = torch.zeros(2 * n_seq + 2, dtype=torch.float64, device=dev)
    else:
        vals, sums = ops.temporal_error_host(frames, ff, bf, prev_index, cur_index, chunk_pairs=chunk_pairs, device=dev,
                                             return_sums=True, u8_scale=u8_scale, u8_offset=u8_offset)
        packed = pack_local(vals.to(dev, non_blocking=True), sums.to(dev, non_blocking=True).sum(),
                            torch.as_tensor(seq_of_pair).to(dev), n_seq, C * H * W)
    return unpack(allreduce_sums(packed, group), n_seq)
