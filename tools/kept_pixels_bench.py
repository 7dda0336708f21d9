"""Cost of the kept-pixel sums: the fused evaluation with `want_kept=True` against the same call without, on the device and
through the host-buffer entry.

  python tools/kept_pixels_bench.py [--out profiles/r06_kept_pixels.json] [--pairs 1041] [--rounds 7] [--host-pairs 64]

Sintel shape (1024 x 436), computed mask (computeTCL), fp32 frames, seeded synthetic inputs.
  resident   bench.py's workload: `--pairs` independent device-resident pairs (26 GB: nothing of it stays in the 126 MB L2), one
             fused launch per call; the kept row and today's row alternate, `--rounds` rounds of 10 calls each after a pre-heat;
             Gpix/s = pairs * H * W / time between CUDA events.  Also checks that pair_sums are bit-identical between the arms and
             that the kept sums equal fbcCheckTorch's mask summed in fp64 on a sample of pairs.
  host       temporal_error_host on a pinned clip of `--host-pairs` + 1 frames, with and without return_kept, alternating:
             pairs/s from a host clock around the synchronising call.
The card name, power limit and SM clocks are read in the same run."""
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
    q = "name,power.limit,clocks.max.sm,clocks.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=30).stdout.strip().splitlines()
        return {"query": q, "value": out[0] if out else torch.cuda.get_device_name(0)}
    except Exception:
        return {"query": "torch.cuda.get_device_name", "value": torch.cuda.get_device_name(0)}


def pairs(P, d, batch=64):
    ff = torch.empty(P, 2, H, W, device=d)
    bf = torch.empty_like(ff)
    prev = torch.empty(P, 3, H, W, device=d)
    cur = torch.empty_like(prev)
    for s in range(0, P, batch):
        n = min(batch, P - s)
        ff[s:s + n], bf[s:s + n] = tcl.synth.make_flows(n, H, W, seed=100 + s, max_shift=32.0, device=d)
        prev[s:s + n], cur[s:s + n] = tcl.synth.make_frames(n, 3, H, W, seed=100 + s, kind="smooth", device=d)
    return ff, bf, prev, cur


def resident(P, rounds, d):
    ff, bf, prev, cur = pairs(P, d)
    iters = 10
    arms = {"today": lambda: tcl.fused_forward(bf, prev, cur, ff=ff),
            "kept": lambda: tcl.fused_forward(bf, prev, cur, ff=ff, want_kept=True)}
    outs = {}
    for k, fn in arms.items():   # pre-heat both rows (module load, shared-memory attribute, clocks)
        for _ in range(3):
            outs[k] = fn()
    torch.cuda.synchronize()
    runs = {k: [] for k in arms}
    for _ in range(rounds):
        for k, fn in arms.items():
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(iters):
                fn()
            b.record()
            torch.cuda.synchronize()
            runs[k].append(P * H * W * iters / (a.elapsed_time(b) / 1e3) / 1e9)
    sample = list(range(0, P, max(1, P // 16)))[:16]
    want_kept = torch.stack([tcl.fbcCheckTorch(ff[i:i + 1], bf[i:i + 1]).double().sum() for i in sample])
    res = {k: {"gpix_per_s_median": statistics.median(v), "gpix_per_s_min": min(v), "gpix_per_s_max": max(v), "runs": v}
           for k, v in runs.items()}
    res["kept_over_today_median"] = res["kept"]["gpix_per_s_median"] / res["today"]["gpix_per_s_median"]
    res["pair_sums_bit_identical"] = bool(torch.equal(outs["kept"].pair_sums, outs["today"].pair_sums))
    res["kept_equals_mask_sum_on_sample"] = bool(torch.equal(outs["kept"].pair_kept[sample], want_kept))
    res["keep_fraction_mean"] = float(outs["kept"].pair_kept.mean()) / (H * W)
    return res, {"pairs": P, "iters_per_run": iters, "rounds": rounds, "working_set_gb": (ff.numel() * 2 + prev.numel() * 2) * 4 / 1e9}


def host(P, rounds, d):
    T = P + 1
    ff, bf = tcl.synth.make_flows(P, H, W, seed=7, max_shift=32.0, device=d)
    frames, _ = tcl.synth.make_frames(T, 3, H, W, seed=7, kind="smooth", device=d)
    ffh, bfh, fh = ff.cpu().pin_memory(), bf.cpu().pin_memory(), frames.cpu().pin_memory()
    arms = {"today": lambda: tcl.temporal_error_host(fh, ffh, bfh, return_sums=True),
            "kept": lambda: tcl.temporal_error_host(fh, ffh, bfh, return_sums=True, return_kept=True)}
    outs = {k: fn() for k, fn in arms.items()}   # pre-heat (the workspace is sized for the kept call from here on)
    runs = {k: [] for k in arms}
    for _ in range(rounds):
        for k, fn in arms.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            fn()   # (synchronises)
            runs[k].append(P / (time.perf_counter() - t0))
    res = {k: {"pairs_per_s_median": statistics.median(v), "pairs_per_s_min": min(v), "pairs_per_s_max": max(v), "runs": v}
           for k, v in runs.items()}
    res["kept_over_today_median"] = res["kept"]["pairs_per_s_median"] / res["today"]["pairs_per_s_median"]
    res["values_and_sums_bit_identical"] = bool(torch.equal(outs["kept"][0], outs["today"][0]) and torch.equal(outs["kept"][1], outs["today"][1]))
    dev = tcl.fused_forward(bf, frames[:-1], frames[1:], ff=ff, want_kept=True)
    res["kept_equals_device_path"] = bool(torch.equal(outs["kept"][2], dev.pair_kept.cpu()))
    return res, {"pairs": P, "frames": T, "rounds": rounds}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--pairs", type=int, default=1041)
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--host-pairs", type=int, default=64)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    d = torch.device("cuda:0")
    r = {"gpu": gpu_info(), "shape": [H, W], "mask": "computed (OCC | MOB)", "frames": "fp32"}
    r["resident"], r["resident_setup"] = resident(args.pairs, args.rounds, d)
    torch.cuda.empty_cache()
    r["host"], r["host_setup"] = host(args.host_pairs, args.rounds, d)
    r["gpu_after"] = gpu_info()
    text = json.dumps(r, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
