"""Device time of the temporal-loss backward with bf16 frames against fp32 frames, measured in the same run, alternating.

  1. training step (BASELINE config 2: 16 pairs at 256x256, dataset mask, L2 mean): forward + backward to both frames, and
     the backward alone, per dtype; plus the backward without grad_prev (no scatter, no accumulator) to show where its time goes
  2. backward alone on 64 Sintel-shape pairs (436x1024): Gpix/s and the DRAM bytes per pixel the launches need, from shapes
  3. --profile: one torch.profiler pass per dtype over the training-shape backward, device time per kernel / memset

Every timing is a CUDA graph of one step per buffer set over sets that together exceed the 126 MB L2 (the first pass does
not warm the next), replayed; the per-step time is the median over replays.  The GPU's name, power limit and max SM clock
are read with nvidia-smi in the same run.

usage: python tools/bf16_backward_bench.py [--rounds 5] [--replays 20] [--profile] [--out OUT.json]
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import tcl_b200 as tcl  # noqa: E402

DT = {"fp32": (torch.float32, tcl._cabi.F32), "bf16": (torch.bfloat16, tcl._cabi.BF16)}


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else f"nvidia-smi failed: {q.stderr.strip()}"


def make_sets(n_sets, B, H, W, seed, shift, rot, dev):
    sets = []
    for i in range(n_sets):
        ff, bf = [], []
        prev, cur = [], []
        for s in range(0, B, 8):
            n = min(8, B - s)
            f_, b_ = tcl.synth.make_flows(n, H, W, seed=seed + 97 * i + s, max_shift=shift, max_rot_deg=rot, device=dev)
            p_, c_ = tcl.synth.make_frames(n, 3, H, W, seed=seed + 97 * i + s, kind="smooth", device=dev)
            ff.append(f_); bf.append(b_); prev.append(p_); cur.append(c_)
        ff, bf = torch.cat(ff), torch.cat(bf)
        d = dict(bf=bf, mask=tcl.fbcCheckTorch(ff, bf), prev32=torch.cat(prev), cur32=torch.cat(cur))
        del ff
        for name, (tdt, _) in DT.items():
            d["prev_" + name] = d["prev32"].to(tdt)
            d["cur_" + name] = d["cur32"].to(tdt)
        del d["prev32"], d["cur32"]
        sets.append(d)
    return sets


class Step:
    """Library launches of one training-loss step on one buffer set: fused forward (FIN_MEAN) and / or the backward."""

    def __init__(self, sets, dtype, B, H, W, fwd=True, bwd=True, grad_prev=True):
        self.sets, self.dt, self.fwd, self.bwd = sets, dtype, fwd, bwd
        self.B, self.H, self.W = B, H, W
        tdt, code = DT[dtype]
        self.code = code
        self.gp = torch.empty((B, 3, H, W), dtype=tdt, device="cuda") if grad_prev else None
        self.gc = torch.empty((B, 3, H, W), dtype=tdt, device="cuda")
        self.scale = torch.full((1,), 100.0, device="cuda")
        self.nbytes = tcl._cabi.lib().tclb200_backward_workspace_bytes(B, 3, H, W, code) if grad_prev else 0
        self.ws = torch.empty(max(self.nbytes, 1), dtype=torch.uint8, device="cuda")

    def __call__(self, i):
        s = self.sets[i % len(self.sets)]
        prev, cur = s["prev_" + self.dt], s["cur_" + self.dt]
        if self.fwd:
            tcl.fused_forward(s["bf"], prev, cur, mask=s["mask"], finalize=tcl.ops.FIN_MEAN)
        if self.bwd:
            p = lambda t: ctypes.c_void_p(t.data_ptr()) if t is not None else None
            lib = tcl._cabi.lib()
            tcl._cabi.check(lib.tclb200_tcl_backward_dt(
                p(s["bf"]), p(s["mask"]), p(prev), p(cur), p(self.scale), 1.0 / (self.B * 3 * self.H * self.W), p(self.gp), p(self.gc),
                self.B, 3, self.H, self.W, self.code, 0, tcl.ops.L2, p(self.ws) if self.nbytes else None, self.nbytes,
                ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)))


_keep = []   # the steps' output and workspace tensors must outlive the graphs that write them


def graph_of(step, n):
    _keep.append(step)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for i in range(n):
            step(i)
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for i in range(n):
            step(i)
    for _ in range(3):
        g.replay()
    torch.cuda.synchronize()
    return g


def time_graph(g, n, replays):
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(replays)]
    for a, b in evs:
        a.record()
        g.replay()
        b.record()
    torch.cuda.synchronize()
    per = sorted(a.elapsed_time(b) / n for a, b in evs)
    return per[len(per) // 2] * 1e3   # us per step


def run_alternating(cases, rounds, replays):
    """cases: {label: (graph, steps per replay)} -> {label: {median_us, min_us, max_us, rounds}} over alternating rounds."""
    res = {k: [] for k in cases}
    for _ in range(rounds):
        for k, (g, n) in cases.items():
            res[k].append(time_graph(g, n, replays))
    return {k: dict(median_us=sorted(v)[len(v) // 2], min_us=min(v), max_us=max(v), rounds=[round(x, 2) for x in v]) for k, v in res.items()}


def bwd_bytes_per_px(dtype, acc_in_l2):
    """DRAM bytes per pixel of the fused backward with both frame gradients, from shapes (3 channels).  fp32: inputs (flow 8,
    mask 4, prev 12, cur 12), grad_cur 12, grad_prev 12 written by the zero-fill, 12 read-for-ownership and 12 written back by
    the scatter.  bf16: inputs 8 + 4 + 6 + 6, grad_cur 6; the fp32 accumulator: zero-fill 12, read-for-ownership 12, write-back
    12, read by the rounding kernel 12; grad_prev 6.  With the accumulator resident in L2 its zero-fill, read-for-ownership and
    second read stay on chip and only the write-back of its dirty lines reaches DRAM."""
    if dtype == "fp32":
        parts = dict(inputs=36, grad_cur=12, memset=12, scatter_rfo=12, scatter_writeback=12)
    else:
        parts = dict(inputs=24, grad_cur=6, memset=12, scatter_rfo=12, scatter_writeback=12, round_read=12, grad_prev_bf16=6)
        if acc_in_l2:
            parts.update(memset=0, scatter_rfo=0, round_read=0)
    return sum(parts.values()), parts


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--replays", type=int, default=20)
    ap.add_argument("--profile", action="store_true")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bf16_backward_bench.py needs a CUDA device")
    torch.cuda.set_device(0)
    out = dict(gpu=gpu_info(), torch=torch.__version__)

    # 1. training shape
    B, H, W, nset = 16, 256, 256, 12
    sets = make_sets(nset, B, H, W, 9500, 24.0, 6.0, "cuda")
    cases = {}
    for dt in DT:
        cases[f"train_fwd_bwd_{dt}"] = (graph_of(Step(sets, dt, B, H, W), nset), nset)
        cases[f"train_bwd_{dt}"] = (graph_of(Step(sets, dt, B, H, W, fwd=False), nset), nset)
        cases[f"train_bwd_grad_cur_only_{dt}"] = (graph_of(Step(sets, dt, B, H, W, fwd=False, grad_prev=False), nset), nset)
    t = run_alternating(cases, args.rounds, args.replays)
    px = B * H * W
    out["train_b16_256"] = dict(pairs=B, shape=f"{W}x{H}", mask="dataset (mask_in)", loss="L2 mean, lambda 100", buffer_sets=nset,
                                accumulator_mb=B * 3 * H * W * 4 / 1e6, times=t,
                                gpix_per_s={k: px / v["median_us"] / 1e3 for k, v in t.items()})
    if args.profile:
        out["train_b16_256"]["profile_us_per_step"] = profile(sets, B, H, W, nset)
    del cases, sets
    torch.cuda.empty_cache()

    # 2. backward alone, 64 Sintel-shape pairs (the accumulator, 343 MB, does not fit L2)
    B, H, W, nset = 64, 436, 1024, 2
    sets = make_sets(nset, B, H, W, 7100, 32.0, 3.0, "cuda")
    cases = {f"sintel64_bwd_{dt}": (graph_of(Step(sets, dt, B, H, W, fwd=False), nset), nset) for dt in DT}
    t = run_alternating(cases, args.rounds, max(5, args.replays // 2))
    px = B * H * W
    rows = {}
    for dt in DT:
        v = t[f"sintel64_bwd_{dt}"]
        bpp, parts = bwd_bytes_per_px(dt, acc_in_l2=False)
        rows[dt] = dict(times=v, gpix_per_s=px / v["median_us"] / 1e3, dram_bytes_per_px=bpp, bytes_parts=parts,
                        achieved_gbs=px * bpp / v["median_us"] / 1e3)
    out["sintel64_bwd"] = dict(pairs=B, shape=f"{W}x{H}", **rows)
    out["bytes_model_train_shape"] = {dt: bwd_bytes_per_px(dt, acc_in_l2=(dt == "bf16"))[0] for dt in DT}
    line = json.dumps(out, indent=1)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


def profile(sets, B, H, W, nset):
    """Device time per kernel (and memset) of the backward alone, per dtype, from torch.profiler (eager launches)."""
    from torch.profiler import ProfilerActivity, profile as tprof
    res = {}
    for dt in DT:
        step = Step(sets, dt, B, H, W, fwd=False)
        for i in range(nset):
            step(i)
        torch.cuda.synchronize()
        reps = 4
        with tprof(activities=[ProfilerActivity.CUDA]) as prof:
            for r in range(reps):
                for i in range(nset):
                    step(i)
            torch.cuda.synchronize()
        acc = {}
        for e in prof.key_averages():
            if e.self_device_time_total > 0:
                name = "memset" if "memset" in e.key.lower() else e.key.split("(")[0].replace("void ", "").replace("tcl::", "")
                acc[name] = acc.get(name, 0.0) + e.self_device_time_total
        res[dt] = {k: v / (reps * nset) for k, v in sorted(acc.items())}
    return res


if __name__ == "__main__":
    main()
