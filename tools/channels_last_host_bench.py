"""Scoring interleaved host clips: channels-last frames and flows through the host-buffer entry, against planar ones and
against a host transpose in front of the planar entry.

  python tools/channels_last_host_bench.py [--out profiles/r05_channels_last_host.json] [--frames 65] [--rounds 5]

Sintel shape (1024 x 436), `--frames` frames (consecutive pairs), computed mask, seeded synthetic inputs, uint8 and fp32
frames, one call per step (`temporal_error_host`, synchronised), in one chunk and in chunks of 8 pairs.  Three arms, alternated
round by round:
  planar       (a) planar pinned frames and flows -- the best case before channels-last input was taken
  cl           (b) the same values as channels-last views of pinned (F,H,W,C) / (P,H,W,2) memory, de-interleaved on the GPU
  host_copy    (c) those channels-last tensors made `.contiguous()` on the host (pageable results) and passed to the planar
               entry, the transpose inside the timed step
pairs/s per arm (median, min, max over the rounds), whether the arms' results are bit-identical, the pinned H2D ceiling of
the same run (tools/u8_frames_bench.py's measurement), the card's name, power limit and SM clocks, the host's core count.
A separate profiled call per frame type gives the device time of the conversion kernels per chunk, next to the fused
kernel's."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import torch

sys.dont_write_bytecode = True
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import tcl_b200 as tcl  # noqa: E402
from u8_frames_bench import h2d_ceiling  # noqa: E402  (tools/ is this script's directory)

H, W = 436, 1024
CONVERT = ("hwc_to_chw_kernel", "hwc_split_kernel", "hwc2_split_kernel")


def gpu_info():
    q = "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm"
    out = subprocess.run(["nvidia-smi", q, "--format=csv"], capture_output=True, text=True, timeout=30).stdout.strip()
    return out.splitlines()


def clip(T, d):
    ff, bf = tcl.synth.make_flows(T - 1, H, W, seed=7, max_shift=32.0, device=d)
    g = torch.Generator(device=d).manual_seed(7)
    u8 = torch.randint(0, 256, (T, 3, H, W), device=d, dtype=torch.uint8, generator=g)
    return ff, bf, {"u8": u8, "fp32": u8.float().mul(torch.tensor(1 / 255, dtype=torch.float32, device=d))}


def pinned_hwc(t):
    """A channels-last view of pinned interleaved memory holding t's values."""
    return t.permute(0, 2, 3, 1).contiguous().cpu().pin_memory().permute(0, 3, 1, 2)


def host_clips(T, d):
    """Per frame type: the three arms' calls on pinned host copies of one seeded clip (the flows are shared)."""
    ff, bf, frames = clip(T, d)
    flows_planar = (ff.cpu().pin_memory(), bf.cpu().pin_memory())
    flows_cl = (pinned_hwc(ff), pinned_hwc(bf))
    runs, pinned = {}, {}
    for kind, fr in frames.items():
        planar = (fr.cpu().pin_memory(),) + flows_planar
        cl = (pinned_hwc(fr),) + flows_cl
        pinned[kind] = planar
        runs[kind] = {"planar": lambda planar=planar, **kw: tcl.temporal_error_host(*planar, **kw),
                      "cl": lambda cl=cl, **kw: tcl.temporal_error_host(*cl, **kw),
                      "host_copy": lambda cl=cl, **kw: tcl.temporal_error_host(*(t.contiguous() for t in cl), **kw)}
    return runs, frames, ff, list(pinned["fp32"])   # (the last: what the H2D ceiling copies, the largest set)


def timed(T, rounds, d, chunk_pairs):
    runs, frames, ff, ceiling_bufs = host_clips(T, d)
    P = T - 1
    out = {}
    ceiling = h2d_ceiling(d, ceiling_bufs)
    t = {kind: {arm: [] for arm in fns} for kind, fns in runs.items()}
    res = {kind: {} for kind in runs}
    for kind, fns in runs.items():      # pre-heat every arm (workspace sized for the largest, modules loaded, clocks up)
        for arm, fn in fns.items():
            res[kind][arm] = fn(chunk_pairs=chunk_pairs, return_sums=True)
    for _ in range(rounds):
        for kind, fns in runs.items():
            for arm, fn in fns.items():
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                fn(chunk_pairs=chunk_pairs)        # (synchronises)
                t[kind][arm].append(time.perf_counter() - t0)
    for kind, fns in runs.items():
        nbytes = frames[kind].numel() * frames[kind].element_size() + 2 * ff.numel() * 4
        ref = res[kind]["planar"]
        o = {}
        for arm, v in t[kind].items():
            m = statistics.median(v)
            o[arm] = {"pairs_per_s_median": P / m, "pairs_per_s_min": P / max(v), "pairs_per_s_max": P / min(v),
                      "step_ms": [x * 1e3 for x in v], "h2d_gb_per_s": nbytes / m / 1e9, "h2d_frac_of_ceiling": nbytes / m / 1e9 / ceiling,
                      "bit_identical_to_planar": bool(torch.equal(res[kind][arm][0], ref[0]) and torch.equal(res[kind][arm][1], ref[1]))}
        o["cl_over_planar"] = o["cl"]["pairs_per_s_median"] / o["planar"]["pairs_per_s_median"]
        o["host_copy_over_planar"] = o["host_copy"]["pairs_per_s_median"] / o["planar"]["pairs_per_s_median"]
        o["h2d_bytes"] = nbytes
        out[kind] = o
    return out, {"pairs": P, "frames": T, "chunk_pairs": chunk_pairs or P, "rounds": rounds, "h2d_ceiling_gb_per_s": ceiling}


def profiled(T, d, chunk_pairs):
    """Device time of the conversion kernels and of the fused launches, one channels-last call per frame type."""
    runs = host_clips(T, d)[0]
    n_chunks = -(-(T - 1) // (chunk_pairs or (T - 1)))
    out = {}
    for kind, fns in runs.items():
        fns["cl"](chunk_pairs=chunk_pairs)
        torch.cuda.synchronize()
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            fns["cl"](chunk_pairs=chunk_pairs)
        per = {}
        for e in prof.key_averages():
            dt = getattr(e, "device_time_total", None)
            if dt is None:
                dt = e.cuda_time_total
            if dt > 0 and ("kernel" in e.key or "Memcpy" in e.key):
                per[e.key[:120]] = {"count": e.count, "device_us": dt}
        conv = sum(v["device_us"] for k, v in per.items() if any(c in k for c in CONVERT))
        fused = sum(v["device_us"] for k, v in per.items() if "fused_forward" in k)
        out[kind] = {"chunks": n_chunks, "convert_us_per_chunk": conv / n_chunks, "fused_us_per_chunk": fused / n_chunks,
                     "events": per}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--frames", type=int, default=65)
    ap.add_argument("--rounds", type=int, default=5)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    d = torch.device("cuda:0")
    r = {"gpu": gpu_info(), "host_cores": os.cpu_count(), "torch_threads": torch.get_num_threads(), "shape": [H, W],
         "mask": "computed (OCC | MOB)"}
    r["one_chunk"], r["one_chunk_setup"] = timed(args.frames, args.rounds, d, 0)
    r["chunks_of_8"], r["chunks_of_8_setup"] = timed(args.frames, args.rounds, d, 8)
    r["profile_chunks_of_8"] = profiled(args.frames, d, 8)
    r["gpu_after"] = gpu_info()
    text = json.dumps(r, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
