"""Scoring stored 8-bit video: uint8 frames against fp32 / bf16 frames, on the device and through the host-buffer entry.

  python tools/u8_frames_bench.py [--out profiles/r04_u8_frames.json] [--frames 65] [--repeats 5]

Sintel shape (1024 x 436), clip mode with a computed mask (computeTCL over consecutive frames), seeded synthetic inputs.
  resident   temporal_error_clip on a device-resident clip of `--frames` frames (working set > 126 MB of L2 for every frame
             type: the flows alone are 7.1 MB a pair); fp32 / bf16 / uint8 alternate, `--repeats` rounds after a pre-heat,
             Gpix/s = pairs * H * W / kernel time
  host       temporal_error_host on pinned CPU clips: pairs/s, the H2D bytes the entry moves per pair (one new frame + two
             flows) over the time, and the pinned H2D copy ceiling measured in the same run the way bench.py measures it; once as
             one chunk of pairs (the launch after the copies) and once in chunks of 8 pairs (launches under the next copies)
  default    whether torch-CUDA's u.float() / 255 rounds like u.float() * fp32(1/255) (the default normalisation), all 256 values
The card name and power limit are read in the same run."""
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

H, W = 436, 1024


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else torch.cuda.get_device_name(0)
    except Exception:
        return torch.cuda.get_device_name(0)


def clip(T, d):
    ff, bf = tcl.synth.make_flows(T - 1, H, W, seed=7, max_shift=32.0, device=d)
    g = torch.Generator(device=d).manual_seed(7)
    u8 = torch.randint(0, 256, (T, 3, H, W), device=d, dtype=torch.uint8, generator=g)
    scale = torch.tensor(1 / 255, dtype=torch.float32, device=d)
    f32 = u8.float().mul(scale)
    return ff, bf, {"fp32": f32, "bf16": f32.to(torch.bfloat16), "u8": u8}


def resident(T, repeats, d):
    ff, bf, frames = clip(T, d)
    P = T - 1
    iters = 20
    res = {k: [] for k in frames}
    outs = {}
    for k, fr in frames.items():   # pre-heat every frame type (module load, allocator, clocks)
        for _ in range(5):
            outs[k] = tcl.temporal_error_clip(fr, ff, bf)
    torch.cuda.synchronize()
    for _ in range(repeats):
        for k, fr in frames.items():
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(iters):
                tcl.temporal_error_clip(fr, ff, bf)
            b.record()
            torch.cuda.synchronize()
            res[k].append(P * H * W * iters / (a.elapsed_time(b) / 1e3) / 1e9)
    ref = outs["fp32"].double()
    return {k: {"gpix_per_s_median": statistics.median(v), "gpix_per_s_min": min(v), "gpix_per_s_max": max(v), "runs": v,
                "max_rel_diff_vs_fp32": float(((outs[k].double() - ref).abs() / ref.abs()).max())} for k, v in res.items()}, \
        {"pairs": P, "frames": T, "iters_per_run": iters,
         "working_set_mb": {k: (fr.numel() * fr.element_size() + 2 * ff.numel() * 4) / 1e6 for k, fr in frames.items()}}


def h2d_ceiling(d, bufs, reps=2):
    """bench.py's measurement for one rank: the whole pinned set, copies of up to 2 GiB back to back on one stream."""
    piece = 2 << 30
    flats = [b.view(-1).view(torch.uint8) for b in bufs]
    dst = torch.empty(min(piece, max(f.numel() for f in flats)), dtype=torch.uint8, device=d)
    total, best = sum(f.numel() for f in flats), 0.0
    for _ in range(reps):
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for f in flats:
            for o in range(0, f.numel(), piece):
                n = min(piece, f.numel() - o)
                dst[:n].copy_(f[o:o + n], non_blocking=True)
        b.record()
        torch.cuda.synchronize()
        best = max(best, total / (a.elapsed_time(b) / 1e3) / 1e9)
    return best


def host(T, repeats, d, chunk_pairs=0):
    ff, bf, frames = clip(T, d)
    P = T - 1
    ffh, bfh = ff.cpu().pin_memory(), bf.cpu().pin_memory()
    fh = {k: v.cpu().pin_memory() for k, v in frames.items()}
    ceiling = h2d_ceiling(d, [fh["fp32"], ffh, bfh])
    res = {k: [] for k in fh}
    for k in ("fp32", "bf16", "u8"):   # pre-heat (the workspace is sized for the largest bank first)
        tcl.temporal_error_host(fh[k], ffh, bfh, chunk_pairs=chunk_pairs)
    for _ in range(repeats):
        for k, fr in fh.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            tcl.temporal_error_host(fr, ffh, bfh, chunk_pairs=chunk_pairs)   # (synchronises)
            res[k].append(time.perf_counter() - t0)
    out = {}
    for k, v in res.items():
        t = statistics.median(v)
        nbytes = fh[k].numel() * fh[k].element_size() + ffh.numel() * 4 + bfh.numel() * 4
        out[k] = {"pairs_per_s_median": P / t, "pairs_per_s_min": P / max(v), "pairs_per_s_max": P / min(v),
                  "h2d_bytes": nbytes, "h2d_bytes_per_pair": nbytes / P, "h2d_gb_per_s": nbytes / t / 1e9,
                  "h2d_frac_of_ceiling": nbytes / t / 1e9 / ceiling}
    for k in ("bf16", "u8"):
        out[k]["speedup_vs_fp32"] = out[k]["pairs_per_s_median"] / out["fp32"]["pairs_per_s_median"]
        out[k]["byte_model_speedup_vs_fp32"] = out["fp32"]["h2d_bytes_per_pair"] / out[k]["h2d_bytes_per_pair"]
    return out, {"pairs": P, "frames": T, "chunk_pairs": chunk_pairs or P, "h2d_ceiling_gb_per_s": ceiling}


def default_scale_check(d):
    u = torch.arange(256, dtype=torch.uint8, device=d)
    div = u.float() / 255
    mul = u.float().mul(torch.tensor(1 / 255, dtype=torch.float32, device=d))
    return {"values": 256, "div_255_differs_from_mul_fp32_recip": int((div != mul).sum()),
            "div_255_differs_from_true_quotient": int((div.double() != (u.double() / 255).float().double()).sum())}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--frames", type=int, default=65)
    ap.add_argument("--repeats", type=int, default=5)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    d = torch.device("cuda:0")
    r = {"gpu": gpu_info(), "shape": [H, W], "mask": "computed (OCC | MOB)", "default_scale": default_scale_check(d)}
    r["resident"], r["resident_setup"] = resident(args.frames, args.repeats, d)
    torch.cuda.empty_cache()
    r["host"], r["host_setup"] = host(args.frames, args.repeats, d)
    # the same clip in chunks of 8 pairs: each chunk's launch runs under the next chunk's copies (the pipeline's steady state)
    r["host_chunked"], r["host_chunked_setup"] = host(args.frames, args.repeats, d, chunk_pairs=8)
    text = json.dumps(r, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
