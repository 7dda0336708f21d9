#!/usr/bin/env python
"""Benchmark of the flow-based temporal-consistency hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME] [--dump-outputs DIR]

A step = one pass of the fused warp + occlusion-mask + masked-error kernel over this rank's shard
of synthetic frame pairs (default workload: the full Sintel-shape evaluation, 23 sequences /
1041 pairs of 1024x436 fp32 per GPU -- weak scaling, pairs sharded by rank, ONE all-reduce of the
packed sums per step when N > 1).  Prints ONE JSON line (see README / DESIGN.md for the keys).

`--impl reference` times the reference's own CPU implementation of the path: the op-for-op ATen
restatement in oracle/torch_port.py (the Python reference itself cannot travel to the GPU box),
on all host cores, on a bounded sample of the same workload.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True     # the benchmark leaves the tree as it found it (it may be read-only)

BYTES_PER_PX = {"fp32": 40, "bf16": 28}  # SURVEY.md 8(d): ff 8 + bf 8 + prev 4C|2C + cur 4C|2C, C = 3


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="sintel_full")
    ap.add_argument("--pairs", type=int, default=None, help="pairs per GPU per step (default: the workload's)")
    ap.add_argument("--frames", default="smooth", choices=["smooth", "white"])
    ap.add_argument("--no-extras", action="store_true", help="skip e2e / cpu_baseline / other workloads")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step returned as DIR/<name>.npy (float64)")
    return ap.parse_args()


def dump_outputs(out_dir, out):
    """The arrays the timed call (tcl_b200.evaluate_sharded) returned in its last step, one DIR/<name>.npy each.  The inputs
    are seeded, so two builds run with the same arguments can be compared output for output."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, t in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().cpu().numpy().astype(np.float64))


# ------------------------------------------------------------------------------------------------
def kernel_source_hash():
    """Hash of the CUDA sources the library is built from: ties an ncu capture to the kernel it was taken from."""
    import hashlib
    h = hashlib.sha256()
    d = os.path.join(ROOT, "gan-based-video-style-transfer_b200", "csrc")
    for f in ("tcl_kernels.cu", "tcl_common.cuh", "tcl_math.cuh"):
        h.update(open(os.path.join(d, f), "rb").read())
    return h.hexdigest()[:16]


def load_traffic(workload, n_pairs):
    """dram__bytes_read+write of the dominant kernel per launch, from the committed ncu capture of this very
    command (profiles/r02_bench_traffic.json, written by tools/ncu_traffic.py).  None when there is no capture of
    this workload or when the kernel sources changed since it was taken (a stale capture is not reported)."""
    p = os.path.join(ROOT, "profiles", "r02_bench_traffic.json")
    try:
        rec = json.load(open(p))
        if (rec.get("workload") == workload and int(rec.get("pairs_per_launch", -1)) == int(n_pairs)
                and rec.get("kernel_source_hash") == kernel_source_hash()):
            return float(rec["dram_bytes_per_launch"])
    except Exception:
        pass
    return None


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = sorted(int(r[0]) for r in self.rows if r and r[0].isdigit())
        mx = [int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 2 + i and r[2 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def bind_to_gpu_numa_node(index):
    """Pin this rank's host threads to the CPUs next to its GPU (NVML's ideal affinity), so that the pinned host buffers
    of the e2e leg are first-touched on the GPU's own NUMA node.  Best effort: silently skipped where NVML says no."""
    try:
        import pynvml
        pynvml.nvmlInit()
        visible = os.environ.get("CUDA_VISIBLE_DEVICES")
        phys = int(visible.split(",")[index]) if visible and visible.split(",")[index].isdigit() else index
        pynvml.nvmlDeviceSetCpuAffinity(pynvml.nvmlDeviceGetHandleByIndex(phys))
    except Exception:
        pass


def make_shard(tcl, cfg_name, n_pairs, seed, device, frames, chunk=32, start=0, stop=None):
    """Synthetic pairs [start, stop) of the `n_pairs`-pair data set `seed` names, resident in HBM: dict of
    (n,2,H,W)/(n,3,H,W) tensors.  The data set is defined chunk-wise (pairs [s, s + chunk) come from seed + s), so any
    rank can generate exactly its slice of it: the strong-scaling leg shards the SAME pairs N ways."""
    cfg = tcl.synth.CONFIGS[cfg_name]
    H, W, C = cfg["H"], cfg["W"], cfg["C"]
    dt = torch.bfloat16 if cfg["dtype"] == "bf16" else torch.float32
    stop = n_pairs if stop is None else stop
    n = stop - start
    out = dict(ff=torch.empty(n, 2, H, W, device=device), bf=torch.empty(n, 2, H, W, device=device),
               prev=torch.empty(n, C, H, W, device=device, dtype=dt),
               cur=torch.empty(n, C, H, W, device=device, dtype=dt))
    for s in range(start // chunk * chunk, stop, chunk):
        e = min(n_pairs, s + chunk)
        ff, bf = tcl.synth.make_flows(e - s, H, W, seed=seed + s, max_shift=cfg["max_shift"],
                                      max_rot_deg=cfg["max_rot_deg"], device=device)
        prev, cur = tcl.synth.make_frames(e - s, C, H, W, seed=seed + s, kind=frames, device=device, dtype=dt)
        lo, hi = max(s, start), min(e, stop)      # the part of this chunk the slice owns
        for k, t in (("ff", ff), ("bf", bf), ("prev", prev), ("cur", cur)):
            out[k][lo - start:hi - start] = t[lo - s:hi - s]
    return out


def time_kernel(fn, steps, warmup):
    """CUDA-event timing on the current stream; returns (total_ms, per-step ms list)."""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for a, b in evs:
        a.record()
        fn()
        b.record()
    torch.cuda.synchronize()
    per = [a.elapsed_time(b) for a, b in evs]
    return evs[0][0].elapsed_time(evs[-1][1]), per


# ------------------------------------------------------------------------------------------------
def cpu_reference_rate(tcl, cfg_name, frames, budget_s, max_pairs=64):
    """The reference's CPU path (ATen-op port, all host threads) on a bounded sample: pairs/s."""
    from oracle import torch_port as tp
    import oracle
    cfg = tcl.synth.CONFIGS[cfg_name]
    H, W, C = cfg["H"], cfg["W"], cfg["C"]
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    ff, bf = tcl.synth.make_flows(2, H, W, seed=4321, max_shift=cfg["max_shift"], max_rot_deg=cfg["max_rot_deg"])
    prev, cur = tcl.synth.make_frames(2, C, H, W, seed=4321, kind=frames)
    with torch.no_grad():
        tp.temporal_error(ff[:1], bf[:1], prev[:1], cur[:1])  # warm-up
        n, t0 = 0, time.perf_counter()
        while True:
            i = n % 2
            tp.temporal_error(ff[i:i + 1], bf[i:i + 1], prev[i:i + 1], cur[i:i + 1])
            n += 1
            el = time.perf_counter() - t0
            if el >= budget_s or n >= max_pairs:
                break
    rate = n / el
    # the plain-C restatement (OpenMP) for context: a tighter CPU implementation than the ATen op chain
    oracle.build()
    a = [t.numpy() for t in (ff[:1], bf[:1], prev[:1], cur[:1])]
    oracle.temporal_error_sums(*a)
    m, t0 = 0, time.perf_counter()
    while time.perf_counter() - t0 < min(3.0, budget_s / 3) and m < 200:
        oracle.temporal_error_sums(*a)
        m += 1
    c_rate = m / (time.perf_counter() - t0)
    return dict(value=rate, unit="pairs/s", cores=cores, kind="port",
                sample=f"{n} {W}x{H} fp32 pairs of the same synthetic workload in {el:.1f} s; oracle/torch_port.py = the "
                       f"reference's ATen op sequence (bit-identical to utils/flowtools.py on CPU), torch threads={cores}",
                gpix_per_s=rate * H * W / 1e9, c_port_pairs_per_s=c_rate,
                c_port_note="oracle/tcl_oracle.c fused restatement, OpenMP over rows, same sample")


def run_reference(args, tcl):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cfg = tcl.synth.CONFIGS[args.workload]
    H, W, C = cfg["H"], cfg["W"], cfg["C"]
    from oracle import torch_port as tp
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    sample_pairs = 2
    ff, bf = tcl.synth.make_flows(sample_pairs, H, W, seed=4321, max_shift=cfg["max_shift"], max_rot_deg=cfg["max_rot_deg"])
    prev, cur = tcl.synth.make_frames(sample_pairs, C, H, W, seed=4321, kind=args.frames)
    prev, cur = prev.float(), cur.float()

    def step():
        with torch.no_grad():
            for i in range(sample_pairs):
                tp.temporal_error(ff[i:i + 1], bf[i:i + 1], prev[i:i + 1], cur[i:i + 1])
    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    el = time.perf_counter() - t0
    rate = args.steps * sample_pairs / el
    line = {"impl": "reference", "metric": "warped frame-pairs/sec", "value": rate, "unit": "pairs/s",
            "gpix_per_s": rate * H * W / 1e9, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": el / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": args.workload, "shape": f"{W}x{H}", "channels": C,
                       "pairs_per_gpu_per_step": cfg["pairs"], "frames": args.frames,
                       "reference_sample_pairs_per_step": sample_pairs,
                       "note": "same workload as the GPU arm; each reference step = a bounded sample of it "
                               "(fbcCheckTorch + warp + masked RMSE per pair, all host threads)"},
            "cpu_baseline": {"value": rate, "unit": "pairs/s", "cores": cores, "kind": "port",
                             "sample": f"{sample_pairs} pairs/step x {args.steps} steps, oracle/torch_port.py (ATen op sequence of "
                                       f"utils/flowtools.py + sintel_eval.py:110), torch threads={cores}"},
            "e2e": {"value": rate, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
def cuda_eager_rate(tcl, cfg_name, frames, device, n_pairs=8, reps=3):
    """The reference's own op sequence run eagerly on THIS GPU (utils/flowtools.py:18-58 + utils/sintel_eval.py:110 as
    ATen ops, oracle/torch_port.py: per pair the CPU-built pixel grid is uploaded, ~150 kernels run, the scalar is read
    back -- the way the reference's evaluation loop does, core/solver.py:343): the honest "before" number on the B200."""
    from oracle import torch_port as tp
    cfg = tcl.synth.CONFIGS[cfg_name]
    H, W, C = cfg["H"], cfg["W"], cfg["C"]
    ff, bf = tcl.synth.make_flows(n_pairs, H, W, seed=4321, max_shift=cfg["max_shift"], max_rot_deg=cfg["max_rot_deg"], device=device)
    prev, cur = tcl.synth.make_frames(n_pairs, C, H, W, seed=4321, kind=frames, device=device)
    prev, cur = prev.float(), cur.float()

    def one(i):
        with torch.no_grad():
            return float(tp.temporal_error(ff[i:i + 1], bf[i:i + 1], prev[i:i + 1], cur[i:i + 1]).cpu())   # .cpu() per pair: solver.py:343
    vals = [one(i) for i in range(n_pairs)]   # warm-up (and the values, for the cross-check below)
    torch.cuda.synchronize()
    best = float("inf")
    for _ in range(reps):
        t0 = time.perf_counter()
        for i in range(n_pairs):
            one(i)
        torch.cuda.synchronize()
        best = min(best, time.perf_counter() - t0)
    launches = None
    try:
        from torch.profiler import profile, ProfilerActivity
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            one(0)
            torch.cuda.synchronize()
        evs = prof.events()
        launches = sum(1 for e in evs if e.device_type == torch.autograd.DeviceType.CUDA and "memcpy" not in e.name.lower() and "memset" not in e.name.lower())
        copies = sum(1 for e in evs if e.device_type == torch.autograd.DeviceType.CUDA and "memcpy" in e.name.lower())
    except Exception:
        copies = None
    ours = tcl.fused_forward(bf, prev, cur, ff=ff)
    rel = max(abs(float(v) - o) / max(abs(o), 1e-12) for v, o in zip(ours.pair_vals.cpu(), vals))
    return dict(value=n_pairs / best, unit="pairs/s", gpix_per_s=n_pairs * H * W / best / 1e9, kernels_per_pair=launches, memcpys_per_pair=copies,
                sample=f"{n_pairs} {W}x{H} fp32 pairs, one pair per call, best of {reps} passes; oracle/torch_port.temporal_error on cuda:{device.index} "
                       "(the reference's eager op sequence incl. its per-call host-built grid upload and the per-pair .cpu() read-back)",
                max_rel_diff_vs_fused_kernel=rel)


def strong_scaling_leg(tcl, args, dist, device, rank, world, pairs_in_seq, seed, steps):
    """BASELINE config 3 as stated: the SAME global pairs (data set `seed`, the one rank 0's weak shard holds) sharded over
    the ranks with sharding.plan_shards, per-sequence means + mean over sequences through the one all-reduce
    (StarGANv2AdvCon/core/solver.py:352-354).  The aggregate must not depend on N: fp64 sums of fp32 per-pair values are exact."""
    n_seq, total = len(pairs_in_seq), sum(pairs_in_seq)
    plan = tcl.sharding.plan_shards(pairs_in_seq, world, rank)
    shard = make_shard(tcl, args.workload, total, seed, device, args.frames, start=plan.start, stop=plan.stop)
    seq = torch.tensor(plan.seq_of_pair, dtype=torch.long, device=device)
    out = {}

    def step():
        out["r"] = tcl.evaluate_sharded(shard["ff"], shard["bf"], shard["prev"], shard["cur"], seq, n_seq)

    def kernel_only():
        tcl.fused_forward(shard["bf"], shard["prev"], shard["cur"], ff=shard["ff"])
    for _ in range(5):
        step()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(5):
        step()
    torch.cuda.synchronize()
    t = torch.tensor([(time.perf_counter() - t0) / 5 * 1e3], device=device, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    pre = int(1000.0 / max(float(t[0]), 1e-3)) + 1      # ~1 s of the same load first (sustained clocks), same count on every rank
    for _ in range(pre):
        step()
    torch.cuda.synchronize()
    dist.barrier()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps):
        step()
    b.record()
    kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for x, y in kev:
        x.record(); kernel_only(); y.record()
    torch.cuda.synchronize()
    dist.barrier()
    torch.cuda.synchronize()
    t = torch.tensor([a.elapsed_time(b) / steps, sum(x.elapsed_time(y) for x, y in kev) / steps], device=device, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, k_ms = float(t[0]), float(t[1])
    r = out["r"]
    res = dict(scaling="strong", pairs_total=total, pairs_per_gpu=[tcl.sharding.plan_shards(pairs_in_seq, world, q).n_local for q in range(world)],
               value=total / (ms / 1e3), unit="pairs/s", ms_per_step=ms, fused_kernel_ms_per_step=k_ms,
               share_outside_fused_kernel=max(0.0, 1.0 - k_ms / ms),
               share_note="1 - (fused kernel alone, max over ranks) / (step, max over ranks): the fold / pack / unpack launches + the all-reduce",
               result_check={"mean_over_sequences_rmse": float(r["mean_over_sequences"]), "mean_over_sequences_rmse_hex": float(r["mean_over_sequences"]).hex(),
                             "pooled_rmse": float(r["pooled_rmse"]), "n_pairs": int(r["n_pairs"])},
               note="same global data set as the N = 1 line (seed %d): result_check.mean_over_sequences_rmse_hex must be identical at every N" % seed)
    del shard
    torch.cuda.empty_cache()
    return res


def band_split_leg(tcl, args, dist, device, rank, world, seed, steps):
    """Fewer pairs than GPUs (BASELINE config 5: one 4K pair on eight GPUs; SURVEY.md 8e): the same pair on every rank, one
    horizontal band of target rows each, the bands' sums added by the path's one all-reduce (sharding.evaluate_banded)."""
    cfg = tcl.synth.CONFIGS[args.workload]
    H, W, C = cfg["H"], cfg["W"], cfg["C"]
    d = make_shard(tcl, args.workload, 1, seed, device, args.frames, chunk=1)
    out = {}

    def step():
        out["r"] = tcl.evaluate_banded(d["ff"], d["bf"], d["prev"], d["cur"])
    for _ in range(10):
        step()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(20):
        step()
    torch.cuda.synchronize()
    t = torch.tensor([(time.perf_counter() - t0) / 20 * 1e3], device=device, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    pre = int(1000.0 / max(float(t[0]), 1e-3)) + 1
    for _ in range(pre):
        step()
    torch.cuda.synchronize()
    dist.barrier()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps):
        step()
    b.record()
    torch.cuda.synchronize()
    dist.barrier()
    t = torch.tensor([a.elapsed_time(b) / steps], device=device, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t[0])
    whole = tcl.fused_forward(d["bf"], d["prev"], d["cur"], ff=d["ff"])
    _, per = time_kernel(lambda: tcl.fused_forward(d["bf"], d["prev"], d["cur"], ff=d["ff"]), 20, 5)
    rel = abs(float(out["r"]["pair_sums"][0]) - float(whole.pair_sums[0])) / float(whole.pair_sums[0])
    return dict(pairs=1, shape=f"{W}x{H}", bands=[list(tcl.band_rows(H, world, q)) for q in range(world)], ms_per_evaluation=ms,
                gpix_per_s=H * W / ms / 1e6, single_gpu_ms_per_evaluation=sorted(per)[len(per) // 2],
                rmse=float(out["r"]["pair_rmse"][0]), single_gpu_rmse=float(whole.pair_vals[0]), sum_rel_diff_vs_single_gpu=rel,
                note="eager calls: one banded launch + fold + one all-reduce of the pair's fp64 sum per evaluation, max over ranks")


def h2d_ceiling(device, bufs, dist=None, reps=2):
    """Concurrent pinned-host -> device copy rate of this box, measured in the same run over the SAME bytes the evaluation
    moves: every rank streams its whole pinned staging set (`bufs`: frames and flows, ~13 GB for the Sintel workload) to the
    device with plain cudaMemcpyAsync calls of up to 2 GiB, one after the other on one stream, all ranks at the same time
    (barrier-aligned).  Returns (GB/s over the whole set, best of `reps`; GB/s of the first 2 GiB piece alone, best) for this
    rank: the short copy runs faster than the host can sustain over the full set when eight ranks pull at once."""
    piece = 2 << 30
    flats = [b.view(-1).view(torch.uint8) for b in bufs]
    dst = torch.empty(min(piece, max(f.numel() for f in flats)), dtype=torch.uint8, device=device)
    total = sum(f.numel() for f in flats)
    best_all, best_first = 0.0, 0.0
    for _ in range(reps):
        torch.cuda.synchronize()
        if dist:
            dist.barrier()
        a, f1, b = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        a.record()
        first = True
        for f in flats:
            for o in range(0, f.numel(), piece):
                n = min(piece, f.numel() - o)
                dst[:n].copy_(f[o:o + n], non_blocking=True)
                if first:
                    f1.record()
                    first_bytes, first = n, False
        b.record()
        torch.cuda.synchronize()
        best_all = max(best_all, total / (a.elapsed_time(b) / 1e3) / 1e9)
        best_first = max(best_first, first_bytes / (a.elapsed_time(f1) / 1e3) / 1e9)
    del dst
    return best_all, best_first


def h2d_pattern_rate(device, frames_h, ff_h, bf_h, dist=None, chunk=64, reps=2):
    """The bytes of one step in the ORDER the host entry needs them (per chunk of pairs: the run of frames it adds, its ff
    block, its bf block -- three host arrays read in turn), as plain cudaMemcpyAsync calls on one stream with no kernels and no
    events, all ranks at the same time: the rate the copy pattern itself allows.  With several ranks on one host memory system
    it sits below the big-sequential-copy ceiling (measured at N = 8: 186 vs 233 GB/s); the evaluation should sit on it."""
    P = ff_h.shape[0]
    d_fr = torch.empty((chunk + 1,) + tuple(frames_h.shape[1:]), dtype=frames_h.dtype, device=device)
    d_f = [torch.empty((chunk,) + tuple(ff_h.shape[1:]), dtype=ff_h.dtype, device=device) for _ in range(2)]
    total = (frames_h.numel() * frames_h.element_size() + 2 * ff_h.numel() * 4)
    best = 0.0
    for _ in range(reps):
        torch.cuda.synchronize()
        if dist:
            dist.barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        d_fr[:1].copy_(frames_h[:1], non_blocking=True)
        for s0 in range(0, P, chunk):
            n = min(chunk, P - s0)
            d_fr[:n].copy_(frames_h[s0 + 1:s0 + 1 + n], non_blocking=True)   # (clip boundaries ignored: same bytes, same order)
            d_f[0][:n].copy_(ff_h[s0:s0 + n], non_blocking=True)
            d_f[1][:n].copy_(bf_h[s0:s0 + n], non_blocking=True)
        b.record()
        torch.cuda.synchronize()
        best = max(best, total / (a.elapsed_time(b) / 1e3) / 1e9)
    return best


# ------------------------------------------------------------------------------------------------
def e2e_rate(tcl, shard, pairs_in_seq, steps, warmup, device, chunk=0):
    """Same metric through the public host-buffer API (`tcl_b200.temporal_error_host` = ONE C-ABI call,
    tclb200_tcl_forward_host): the clips' frames and flows start in pinned HOST memory, every step copies them to the
    device inside the call (each stylised frame once -- it is the `cur` of pair t and the `prev` of pair t+1, the way
    utils/sintel_eval.py:206-222 walks a clip), runs the fused launches and reads the per-pair values back to the host."""
    import psutil
    import torch.distributed as tdist
    multi = tdist.is_available() and tdist.is_initialized() and tdist.get_world_size() > 1

    def all_ranks_ok(ok):   # the step below contains a collective: either every rank runs it or none does
        if not multi:
            return ok
        flag = torch.tensor([1 if ok else 0], device=device, dtype=torch.int32)
        tdist.all_reduce(flag, op=tdist.ReduceOp.MIN)
        return bool(int(flag[0]))
    H, W = shard["bf"].shape[2:]
    C = shard["cur"].shape[1]
    esz = shard["cur"].element_size()
    frame_b, flow_b = C * H * W * esz, 2 * H * W * 4
    world = int(os.environ.get("WORLD_SIZE", "1"))
    budget = psutil.virtual_memory().available * 0.5 / world     # pinned host memory this rank may take
    seqs, need = [], 0
    for n in pairs_in_seq:      # as many whole sequences as fit (all of them on the boxes this was measured on)
        b = (n + 1) * frame_b + 2 * n * flow_b
        if seqs and need + b > budget:
            break
        seqs.append(n)
        need += b
    P, F = sum(seqs), sum(seqs) + len(seqs)
    if multi:   # every rank evaluates the same number of sequences (the smallest any rank has room for)
        t = torch.tensor([len(seqs)], device=device, dtype=torch.int32)
        tdist.all_reduce(t, op=tdist.ReduceOp.MIN)
        seqs = seqs[:int(t[0])]
        P, F = sum(seqs), sum(seqs) + len(seqs)
    saved_affinity = os.sched_getaffinity(0)
    if world > 1 and not os.environ.get("TCL_BENCH_NO_BIND"):   # (N = 1 measured 55 GB/s unbound; the cpu_baseline leg that follows must see every host core)
        bind_to_gpu_numa_node(device.index)
    setup_error = None
    try:
        frames_h = torch.empty((F, C, H, W), dtype=shard["cur"].dtype, pin_memory=True)
        ff_h = torch.empty((P, 2, H, W), dtype=torch.float32, pin_memory=True)
        bf_h = torch.empty((P, 2, H, W), dtype=torch.float32, pin_memory=True)
    except Exception as ex:
        setup_error = ex
    if not all_ranks_ok(setup_error is None):
        os.sched_setaffinity(0, saved_affinity)
        raise RuntimeError(f"pinned host buffers for the e2e leg could not be allocated on every rank: {setup_error!r}")
    ff_h.copy_(shard["ff"][:P]); bf_h.copy_(shard["bf"][:P])
    prev_i, cur_i, p0, f0 = [], [], 0, 0
    for n in seqs:    # frame bank of a clip: its first frame, then the frame each pair is compared with
        frames_h[f0].copy_(shard["prev"][p0])
        frames_h[f0 + 1:f0 + 1 + n].copy_(shard["cur"][p0:p0 + n])
        prev_i += list(range(f0, f0 + n)); cur_i += list(range(f0 + 1, f0 + 1 + n))
        p0 += n; f0 += n + 1
    prev_i, cur_i = torch.tensor(prev_i, dtype=torch.int32), torch.tensor(cur_i, dtype=torch.int32)
    torch.cuda.synchronize()
    lib = tcl._cabi.lib()

    seq_ids = torch.tensor([si for si, n in enumerate(seqs) for _ in range(n)], dtype=torch.long)
    ceiling, ceiling_2g = h2d_ceiling(device, [frames_h, ff_h, bf_h], tdist if multi else None)
    pattern = h2d_pattern_rate(device, frames_h, ff_h, bf_h, tdist if multi else None)

    def step():
        # one C-ABI call for the shard (synchronises its stream), the packed sums, ONE all-reduce when N > 1, result on the host
        res = tcl.evaluate_sharded_host(frames_h, ff_h, bf_h, prev_i, cur_i, seq_ids, len(pairs_in_seq), chunk_pairs=chunk)
        return float(res["mean_over_pairs"])

    # short steps (config 4: 286 MB, ~6 ms per rank) are timed over ~2 s worth of them: measured on 2 GPUs, single steps of such a
    # run take 9-99 ms instead of 6 (host-side stalls of lock-stepped ranks), and ten steps would report whichever outliers they caught.
    # Every rank derives the same count from the step's bytes (the step contains a collective).
    h2d = F * frame_b + 2 * P * flow_b + 2 * 4 * P
    steps = max(steps, min(400, int(2.0 / (h2d / 50e9))))
    import gc
    for _ in range(warmup):
        step()
    torch.cuda.synchronize()
    lib.tclb200_debug_launch_count(1)
    gc.collect()
    gc.disable()           # (no collector pauses inside the timed region; nothing here creates reference cycles)
    t0 = time.perf_counter()
    step_ms = []
    for _ in range(steps):
        ts = time.perf_counter()
        mean_rmse = step()
        step_ms.append((time.perf_counter() - ts) * 1e3)
    torch.cuda.synchronize()
    el = time.perf_counter() - t0
    gc.enable()
    step_ms.sort()
    launches = int(lib.tclb200_debug_launch_count(0))
    os.sched_setaffinity(0, saved_affinity)
    return dict(value=steps * P / el, unit="pairs/s", h2d_bytes_per_step=h2d, d2h_bytes_per_step=12 * P + 8,
                ms_per_step=el / steps * 1e3, h2d_gb_per_s=h2d * steps / el / 1e9, pairs_per_step=P, frames_per_step=F,
                sequences_per_step=len(seqs), gpu_launches_per_step=launches // max(steps, 1), mean_rmse=mean_rmse, steps=steps,
                step_ms_rank0=dict(median=round(step_ms[len(step_ms) // 2], 3), p90=round(step_ms[int(len(step_ms) * 0.9)], 3), max=round(step_ms[-1], 3)),
                h2d_ceiling_gb_per_s=ceiling, h2d_first_2gib_gb_per_s=ceiling_2g, h2d_pattern_gb_per_s=pattern,
                note=f"tcl_b200.evaluate_sharded_host = temporal_error_host (C ABI tclb200_tcl_forward_host) + packed sums + one all-reduce when N > 1: pinned host clips -> chunks of pairs ({chunk or 'library default: ~256 MB per flow copy'}), "
                     "3-slot device ring, two internal copy streams; every frame crosses PCIe once per step (28.3 B/px per pair "
                     "instead of 40), per-pair values and sums copied back to the host (12 B per pair), the aggregate read on the host")


def other_workloads(tcl, device, frames, peak):
    """Secondary configs of BASELINE.json (not bench lines; context for the roofline)."""
    out = []
    specs = [("train_b16_256", 16, 12, "mask_in"), ("hd1080_window", 6, 4, "ff"), ("uhd4k_stress", 1, 4, "ff"),
             ("sintel_clip", 49, 1, "ff")]
    for name, n, nbuf, mode in specs:
        try:
            cfg = tcl.synth.CONFIGS[name]
            bufs = [make_shard(tcl, name, n, 9000 + 97 * i, device, frames, chunk=8) for i in range(nbuf)]
            masks = [tcl.fbcCheckTorch(b["ff"], b["bf"]) for b in bufs] if mode == "mask_in" else None
            def launch(i):
                b = bufs[i % nbuf]
                if mode == "mask_in":
                    tcl.fused_forward(b["bf"], b["prev"], b["cur"], mask=masks[i % nbuf], finalize=tcl.ops.FIN_MEAN)
                else:
                    tcl.fused_forward(b["bf"], b["prev"], b["cur"], ff=b["ff"])
            # launch-bound sizes: capture one launch per rotating buffer in a CUDA graph and time replays
            side = torch.cuda.Stream(device)
            with torch.cuda.stream(side):
                for i in range(nbuf):
                    launch(i)
            torch.cuda.synchronize()
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                for i in range(nbuf):
                    launch(i)
            total, per = time_kernel(graph.replay, 20, 5)
            per.sort()
            ms = per[len(per) // 2] / nbuf
            px = n * cfg["H"] * cfg["W"]
            bpp = (36 if mode == "mask_in" else 40) if cfg["dtype"] == "fp32" else 28
            out.append(dict(workload=name, pairs=n, shape=f'{cfg["W"]}x{cfg["H"]}', dtype=cfg["dtype"], mask=mode,
                            ms_per_launch_median=ms, timing="CUDA graph of one launch per rotating buffer, median of 20 replays", gpix_per_s=px / ms / 1e6, bytes_per_px=bpp,
                            achieved_gbs=px * bpp / ms / 1e6, frac_of_measured_peak=px * bpp / ms / 1e6 / peak,
                            rotating_buffers=nbuf, working_set_mb=px * bpp * nbuf / 1e6,
                            kernel=("fused_forward_direct_kernel (dataset mask, launch <= 2 Mpx) + fold_partials_small_kernel" if mode == "mask_in" and px <= (2 << 20)
                                    else "fused_forward_ws_kernel + fold kernel")))
            del bufs, masks
            torch.cuda.empty_cache()
        except Exception as ex:  # report, never hide
            out.append(dict(workload=name, error=repr(ex)))
    out.append(training_step(tcl, device, frames, peak))
    return out


def training_step(tcl, device, frames, peak):
    """BASELINE configs[1] as the trainer runs it (StarGANv2AdvCon/core/solver.py:427-446 + :181): the temporal loss
    forward AND its backward to both frames, batch 16 at 256x256 fp32, dataset mask.  Device time of the two library
    launches (+ the memset of grad_prev) from a CUDA graph over rotating buffers; the eager autograd call is timed
    beside it (host-bound: Python + autograd bookkeeping of a 30 us job)."""
    import ctypes
    name, n, nbuf = "train_b16_256", 16, 12
    try:
        cfg = tcl.synth.CONFIGS[name]
        H, W, C = cfg["H"], cfg["W"], cfg["C"]
        bufs = [make_shard(tcl, name, n, 9500 + 97 * i, device, frames, chunk=8) for i in range(nbuf)]
        masks = [tcl.fbcCheckTorch(b["ff"], b["bf"]) for b in bufs]
        gp, gc = torch.empty_like(bufs[0]["prev"]), torch.empty_like(bufs[0]["cur"])
        scale = torch.full((1,), 100.0 / (n * C * H * W), device=device)     # lambda_tcl = 100 (main.py:94) times 1/N
        lib = tcl._cabi.lib()
        ptr = lambda t: ctypes.c_void_p(t.data_ptr())

        def launch(i):
            b, m = bufs[i % nbuf], masks[i % nbuf]
            tcl.fused_forward(b["bf"], b["prev"], b["cur"], mask=m, finalize=tcl.ops.FIN_MEAN)
            tcl._cabi.check(lib.tclb200_tcl_backward(ptr(b["bf"]), ptr(m), ptr(b["prev"]), ptr(b["cur"]), ptr(scale), ptr(gp), ptr(gc),
                                                     n, C, H, W, 0, tcl.ops.L2, ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)))
        side = torch.cuda.Stream(device)
        with torch.cuda.stream(side):
            for i in range(nbuf):
                launch(i)
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            for i in range(nbuf):
                launch(i)
        _, per = time_kernel(graph.replay, 20, 5)
        per.sort()
        ms = per[len(per) // 2] / nbuf
        # the eager public call: tcl.temporal_loss(...).backward()
        p2, c2 = bufs[0]["prev"].clone().requires_grad_(True), bufs[0]["cur"].clone().requires_grad_(True)

        def eager():
            p2.grad = None
            c2.grad = None
            (tcl.temporal_loss(masks[0], c2, p2, bufs[0]["bf"]) * 100.0).backward()
        _, per_e = time_kernel(eager, 50, 10)
        per_e.sort()
        px = n * H * W
        bpp = 36 + 36 + 24 + 12    # fwd reads; bwd reads again, writes grad_cur + grad_prev (zero-fill), + the scatter's read-for-ownership
        return dict(workload=name + "_fwd_bwd", pairs=n, shape=f"{W}x{H}", dtype="fp32", mask="mask_in", loss="L2 mean, grads to prev and cur",
                    ms_per_step_device=ms, ms_per_step_eager_autograd=per_e[len(per_e) // 2], gpix_per_s=px / ms / 1e6, bytes_per_px=bpp,
                    achieved_gbs=px * bpp / ms / 1e6, frac_of_measured_peak=px * bpp / ms / 1e6 / peak, rotating_buffers=nbuf,
                    timing="CUDA graph of fwd + bwd launches per rotating buffer, median of 20 replays; eager = public autograd call, median of 50")
    except Exception as ex:
        return dict(workload=name + "_fwd_bwd", error=repr(ex))


def main():
    args = parse()
    import tcl_b200 as tcl
    if args.impl == "reference":
        return run_reference(args, tcl)

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the product path has no CPU fallback (use --impl reference for the CPU arm)")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    device = torch.device("cuda", local)
    torch.cuda.set_device(device)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=device)
    tcl._cabi.lib()  # fail loudly now if the CUDA extension is missing

    cfg = tcl.synth.CONFIGS[args.workload]
    H, W, C = cfg["H"], cfg["W"], cfg["C"]
    dtype = cfg["dtype"]
    # weak scaling: every rank owns one workload-sized shard of pairs (for sintel_full: all 23 sequences)
    if args.workload == "sintel_full":
        pairs_in_seq = tcl.sharding.pairs_per_sequence(tcl.synth.SINTEL_TRAIN_FRAMES)
    else:
        pairs_in_seq = [cfg["pairs"]]
    n_local = args.pairs or sum(pairs_in_seq)
    if args.pairs:
        pairs_in_seq = [args.pairs]
    n_seq = len(pairs_in_seq)
    seq_of_pair = torch.tensor([s for s, n in enumerate(pairs_in_seq) for _ in range(n)], dtype=torch.long, device=device)
    GLOBAL_SEED = 1234 + 2000     # rank 0's weak shard = the global data set the strong-scaling leg shards N ways
    shard = make_shard(tcl, args.workload, n_local, GLOBAL_SEED + 100000 * rank, device, args.frames)
    torch.cuda.synchronize()

    last = {}
    lib = tcl._cabi.lib()

    kernel_events = []      # (start, end) events around the fused launch of every timed step

    def step(events=None):
        out = tcl.evaluate_sharded(shard["ff"], shard["bf"], shard["prev"], shard["cur"], seq_of_pair, n_seq, kernel_events=events)
        last["out"] = out

    def kernel_only():
        tcl.fused_forward(shard["bf"], shard["prev"], shard["cur"], ff=shard["ff"])

    def sync_max(v):   # max over ranks of a host number (every rank must then run the same number of steps)
        if not dist:
            return v
        t = torch.tensor([v], device=device, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0])

    for _ in range(max(args.warmup, 3)):
        step()
    torch.cuda.synchronize()
    # Steady state before anything is timed: the board reaches its 1000 W power cap within ~100 ms of this load and the
    # SM clock then settles ~15 % below its maximum.  Run the same step untimed for >= PREHEAT_S so that the timed region,
    # the kernel-only timing behind it and the clock samples all see the capped (sustained) clock, not the burst one.
    PREHEAT_S = 1.5
    t0 = time.perf_counter()
    for _ in range(3):
        step()
    torch.cuda.synchronize()
    est_ms = sync_max((time.perf_counter() - t0) / 3 * 1e3)
    preheat_steps = int(PREHEAT_S * 1e3 / max(est_ms, 1e-3)) + 1
    sampler = ClockSampler(local)
    for i in range(preheat_steps):
        if rank == 0 and i == preheat_steps // 2:
            sampler.start()          # clocks are sampled from the second half of the pre-heat to the end of the timed region
        step()
    torch.cuda.synchronize()
    if dist:
        dist.barrier()
    torch.cuda.synchronize()
    lib.tclb200_debug_launch_count(1)
    lib.tclb200_debug_tile_stats(None, 1)
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.cudart().cudaProfilerStart()   # no-op unless run under `ncu --profile-from-start off` (profiles/ launch lists)
    start.record()
    for _ in range(args.steps):
        step(kernel_events)     # the fused launch of every step is bracketed by its own pair of events: the roofline numerator
    end.record()                # is the dominant kernel's time INSIDE the timed region (kernel_ms_per_launch <= ms_per_step)
    torch.cuda.synchronize()
    torch.cuda.cudart().cudaProfilerStop()
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:     # (the aggregate is all-reduced: every rank holds the same arrays)
        dump_outputs(args.dump_outputs, last["out"])
    n_launches = int(lib.tclb200_debug_launch_count(0))   # kernels of libtcl_b200.so launched inside the timed region
    import ctypes
    tile_stats = (ctypes.c_ulonglong * 2)()
    lib.tclb200_debug_tile_stats(tile_stats, 1)
    tile_stats = [int(tile_stats[0]), int(tile_stats[1])]
    if dist:
        dist.barrier()
    torch.cuda.synchronize()
    elapsed_ms = sync_max(start.elapsed_time(end))   # max over ranks
    per = [ka.elapsed_time(kb) for ka, kb in kernel_events]
    k_ms = sync_max(sum(per) / len(per))
    # the same kernel after a one-second pause: the first launches run before the power cap pulls the SM clock down (what
    # MEASURED_PEAKS' best-of-10 copy peak is: a burst figure).  Reported beside the sustained number, never as `value`.
    time.sleep(1.0)
    _, per_b = time_kernel(kernel_only, 3, 0)
    burst_ms = min(per_b)
    total_pairs = n_local * world * args.steps
    pairs_per_s = total_pairs / (elapsed_ms / 1e3)
    peak, peak_src = load_peaks()
    bpp = BYTES_PER_PX[dtype]
    alg_bytes = n_local * H * W * bpp
    achieved = alg_bytes / (k_ms / 1e3) / 1e9
    res = last["out"]
    # mask statistics of the workload (SURVEY.md 8d: keep fraction and near-threshold pixel count with every run);
    # outside the timed region, on a bounded sample of this rank's pairs, through the exact (counting) path
    ns = min(64, n_local)
    m_s, near_s = tcl.fbcheck_with_near_count(shard["ff"][:ns], shard["bf"][:ns])
    mask_stats = {"sample_pairs": ns, "keep_fraction": float(m_s.mean()), "near_threshold_px": int(near_s),
                  "sample_px": int(m_s.numel()),
                  "note": "pixels whose occlusion / motion-boundary margin is within 1e-6 of the threshold (the north-star exemption band)"}
    del m_s
    line = {
        "metric": "warped frame-pairs/sec", "value": pairs_per_s, "unit": "pairs/s",
        "gpix_per_s": pairs_per_s * H * W / 1e9,
        "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "preheat_steps": preheat_steps,
        "ms_per_step": elapsed_ms / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32" if dtype == "fp32" else "bf16 frames / f32 flows+math", "data": "synthetic",
        "config": {"workload": args.workload, "shape": f"{W}x{H}", "channels": C, "pairs_per_gpu_per_step": n_local,
                   "sequences": n_seq, "frames": args.frames, "sharding": "by frame pair, one all-reduce of packed sums per step",
                   "l2": "inputs (%.1f GB per GPU) are larger than L2, no flush needed" % (alg_bytes / 1e9)},
        "gpu_launches": n_launches,
        "gpu_launches_note": "kernels of libtcl_b200.so inside the timed region: per step one fused_forward_ws_kernel + one "
                             "fold_partials_kernel (programmatic dependent launch) + the two single-CTA aggregation kernels "
                             "(pack / unpack of the per-sequence sums around the all-reduce)",
        "tiles": {"per_step": n_local * ((W + 63) // 64) * ((H + 31) // 32),
                  "mixed_per_step": tile_stats[1] // max(args.steps, 1), "global_per_step": tile_stats[0] // max(args.steps, 1),
                  "note": "mixed = a motion boundary runs through the 64x32 tile, some pixels gather from global memory"},
        "mask_stats": mask_stats,
        "result_check": {"mean_over_sequences_rmse": float(res["mean_over_sequences"]), "mean_over_sequences_rmse_hex": float(res["mean_over_sequences"]).hex(),
                         "pooled_rmse": float(res["pooled_rmse"]), "n_pairs": int(res["n_pairs"]),
                         "note": "aggregate of all ranks' weak shards (rank r holds data set seed + 100000 r); at N = 1 this is the value "
                                 "strong_scaling.result_check must reproduce at every N"},
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": load_traffic(args.workload, n_local), "peak_source": peak_src,
                     "kernel": "tcl::fused_forward_ws_kernel<float, MASK_COMPUTED, reduce, C=3, lean> (+ fold_partials_kernel, <0.1 % of the time)",
                     "kernel_ms_per_launch": k_ms, "algorithmic_bytes_per_launch": alg_bytes, "bytes_per_px": bpp,
                     "frac_of_nominal_8TBs": achieved / 8000.0,
                     "timing": "CUDA events around the fused launch of every timed step (inside the timed region: sustained, power-capped clock); "
                               "the interval also holds the fold_partials_kernel launched behind it with programmatic dependent launch",
                     "burst": {"kernel_ms_per_launch": burst_ms, "achieved": alg_bytes / (burst_ms / 1e3) / 1e9,
                               "frac": alg_bytes / (burst_ms / 1e3) / 1e9 / peak,
                               "note": "side figure: best of 3 launches after a 1 s pause (before the power cap lowers the SM clock); "
                                       "`value`, `achieved` and `frac` are all steady-state (>= 1.5 s of the same load before the timed region)"}},
        "clocks": clocks,
    }
    if clocks is not None:
        line["clocks"]["note"] = (f"sampled (100 ms period) over the second half of the {preheat_steps}-step untimed pre-heat and the timed region "
                                  f"({elapsed_ms:.0f} ms): one uninterrupted run of the same step")
    if not args.no_extras:
        if dist:
            dist.barrier()
        try:
            e = e2e_rate(tcl, shard, pairs_in_seq, max(3, min(args.steps // 2, 10)), 2, device)
        except Exception as ex:   # report, never hide; keep the collectives below symmetric across ranks
            e = {"error": repr(ex), "ms_per_step": float("inf")}
        if dist:  # whole-job rate = all ranks' pairs over the slowest rank's time
            t = torch.tensor([e["ms_per_step"]], device=device, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            if "error" not in e and float(t[0]) != float("inf"):
                e["ms_per_step"] = float(t[0])
                e["value"] = e["pairs_per_step"] * world / (e["ms_per_step"] / 1e3)
                e["h2d_bytes_per_step"] *= world
                e["d2h_bytes_per_step"] *= world
                e["h2d_gb_per_s"] = e["h2d_bytes_per_step"] / (e["ms_per_step"] / 1e3) / 1e9
            c = torch.tensor([e.get("h2d_ceiling_gb_per_s", 0.0), e.get("h2d_first_2gib_gb_per_s", 0.0), e.get("h2d_pattern_gb_per_s", 0.0)],
                             device=device, dtype=torch.float64)
            dist.all_reduce(c, op=dist.ReduceOp.SUM)     # all ranks copied at the same time: the box's aggregate rate
            if "error" not in e:
                e["h2d_ceiling_gb_per_s"], e["h2d_first_2gib_gb_per_s"], e["h2d_pattern_gb_per_s"] = float(c[0]), float(c[1]), float(c[2])
        if "error" not in e and e.get("h2d_ceiling_gb_per_s"):
            e["h2d_frac_of_ceiling"] = e["h2d_gb_per_s"] / e["h2d_ceiling_gb_per_s"]
            if e.get("h2d_pattern_gb_per_s"):
                e["h2d_frac_of_pattern"] = e["h2d_gb_per_s"] / e["h2d_pattern_gb_per_s"]
                e["h2d_pattern_note"] = ("h2d_pattern_gb_per_s = the same bytes in the order the host entry needs them (per chunk of pairs: frames, ff block, "
                                         "bf block, from the caller's three host arrays) as plain cudaMemcpyAsync calls, no kernels, no events, all ranks at once: "
                                         "the evaluation runs at that rate; the gap to h2d_ceiling at N > 1 is the host memory system's, not the pipeline's")
            e["h2d_ceiling_note"] = ("every rank streams its whole pinned staging set (the bytes one step moves) with plain cudaMemcpyAsync calls of "
                                     "<= 2 GiB at the same time (best of 2, summed over ranks): what this box's host side can feed its GPUs; "
                                     "h2d_first_2gib_gb_per_s = the first piece alone (a short copy runs above the sustained rate)")
        line["e2e"] = e
        del shard
        torch.cuda.empty_cache()
        if world > 1 and args.workload == "sintel_full" and not args.pairs:
            try:
                line["strong_scaling"] = strong_scaling_leg(tcl, args, dist, device, rank, world, pairs_in_seq, GLOBAL_SEED, max(args.steps, 20))
            except Exception as ex:
                line["strong_scaling"] = {"error": repr(ex)}
        if world > 1 and args.workload == "uhd4k_stress":
            try:
                line["band_split"] = band_split_leg(tcl, args, dist, device, rank, world, GLOBAL_SEED, max(args.steps, 20))
            except Exception as ex:
                line["band_split"] = {"error": repr(ex)}
        if world == 1:
            try:
                line["cuda_eager_baseline"] = cuda_eager_rate(tcl, args.workload, args.frames, device)
            except Exception as ex:
                line["cuda_eager_baseline"] = {"error": repr(ex)}
            line["cpu_baseline"] = cpu_reference_rate(tcl, args.workload, args.frames, args.cpu_seconds)
            line["other_workloads"] = other_workloads(tcl, device, args.frames, peak)
    if rank == 0:
        print(json.dumps(line), flush=True)
    if dist:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
