"""The training loss under torch.compile: host and device time of its forward + backward per route, and a stand-in training
step eager vs reduce-overhead (CUDA graphs), alternated over rounds in one run.

  1. training-loss forward + backward alone (BASELINE config 2: 16 pairs at 256x256, dataset mask, L2 mean), fp32 and bf16
     frames; arms: ``eager`` (the public function's direct route), ``eager_ops`` (the same call forced through the
     ``torch.ops.tcl_b200`` operators: the routing decision of DESIGN.md section 5 rests on this pair), ``compile``
     (torch.compile default) and ``reduce_overhead`` (torch.compile mode="reduce-overhead").  Host clock around a
     synchronised loop of >= --seconds per arm, device time from CUDA events around the same loop.  Each iteration takes the
     next of --sets buffer sets, which together exceed the 126 MB L2.
  2. the stand-in training step of tests/test_gpu_under_compile.py (two-layer conv generator producing both frames,
     ``loss_tcl * 100``, SGD), eager vs reduce-overhead, steps/s.
  3. --parent DIR: ``bench.py`` of the tree in DIR and of this tree, alternated, with their result_check and pairs/s.

Medians with min-max over --rounds rounds; card name, power limit and SM clocks of the same run (nvidia-smi).

usage: python tools/compile_bench.py [--rounds 5] [--seconds 2] [--parent DIR] [--out profiles/r07_compile.json]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import tcl_b200 as tcl  # noqa: E402

B, C, H, W = 16, 3, 256, 256


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else f"nvidia-smi failed: {q.stderr.strip()}"


def make_sets(n, dtype, dev):
    sets = []
    for i in range(n):
        ff, bf = tcl.synth.make_flows(B, H, W, seed=11 + 97 * i, max_shift=12.0, device=dev)
        prev, cur = (t.to(dev).to(dtype) for t in tcl.synth.make_frames(B, C, H, W, seed=11 + 97 * i, kind="smooth"))
        sets.append(dict(bf=bf, mask=tcl.fbcCheckTorch(ff, bf), prev=prev.requires_grad_(), cur=cur.requires_grad_()))
    return sets


def loss_public(prev, cur, flow, mask):
    return tcl.temporal_loss(mask, cur, prev, flow)


def loss_ops(prev, cur, flow, mask):
    # what temporal_loss does after its validation on the traced route
    return torch.ops.tcl_b200.temporal_loss(prev, cur, flow, mask, tcl.ops.L2, 0)


def timed_loop(fn, sets, seconds):
    """-> (host us per iteration, device us per iteration) over a synchronised loop of >= seconds."""
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n, t0 = 0, time.perf_counter()
    e0.record()
    while True:
        for _ in range(50):
            fn(sets[n % len(sets)])
            n += 1
        if time.perf_counter() - t0 >= seconds:
            break
    e1.record()
    torch.cuda.synchronize()
    host = time.perf_counter() - t0
    return host / n * 1e6, e0.elapsed_time(e1) / n * 1e3


def fwd_bwd(loss_fn):
    def step(s):
        s["prev"].grad = s["cur"].grad = None
        loss_fn(s["prev"], s["cur"], s["bf"], s["mask"]).backward()
    return step


def summary(xs):
    return dict(median=statistics.median(xs), min=min(xs), max=max(xs), n=len(xs))


class StandIn(torch.nn.Module):
    def __init__(self):
        super().__init__()
        self.c1 = torch.nn.Conv2d(3, 8, 3, padding=1)
        self.c2 = torch.nn.Conv2d(8, 3, 3, padding=1)

    def forward(self, x):
        return torch.sigmoid(self.c2(torch.relu(self.c1(x))))


def tcl_step_loss(G, x_prev, x_cur, flow, mask):
    return tcl.temporal_loss(mask, G(x_cur), G(x_prev), flow) * 100.0


def bench_line(tree, steps, warmup):
    r = subprocess.run([sys.executable, "bench.py", "--gpus", "1", "--steps", str(steps), "--warmup", str(warmup)], cwd=tree,
                       capture_output=True, text=True)
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    if r.returncode != 0 or not lines:
        raise RuntimeError(f"bench.py in {tree} failed ({r.returncode}): {r.stderr[-2000:]}")
    return json.loads(lines[-1])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--seconds", type=float, default=2.0)
    ap.add_argument("--sets", type=int, default=8)
    ap.add_argument("--parent", default=None)
    ap.add_argument("--bench-steps", type=int, default=100)
    ap.add_argument("--bench-warmup", type=int, default=20)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("compile_bench needs a CUDA device")
    dev = torch.device("cuda:0")
    out = dict(gpu_before=gpu_info(), torch=torch.__version__, shape=f"{B}x{C}x{H}x{W}, dataset mask, L2 mean", rounds=a.rounds,
               seconds_per_arm=a.seconds, buffer_sets=a.sets, loss={}, step={})

    # 1. the training loss alone
    for name, dtype in (("fp32", torch.float32), ("bf16", torch.bfloat16)):
        sets = make_sets(a.sets, dtype, dev)
        arms = dict(eager=fwd_bwd(loss_public), eager_ops=fwd_bwd(loss_ops),
                    compile=fwd_bwd(torch.compile(loss_public, fullgraph=True)),
                    reduce_overhead=fwd_bwd(torch.compile(loss_public, mode="reduce-overhead", fullgraph=True)))
        for fn in arms.values():   # warm-up: compiles, cudagraph recording, allocator
            for s in sets * 3:
                fn(s)
        res = {k: dict(host_us=[], device_us=[]) for k in arms}
        for r in range(a.rounds):
            for k in (list(arms) if r % 2 == 0 else list(arms)[::-1]):
                h, d = timed_loop(arms[k], sets, a.seconds)
                res[k]["host_us"].append(h)
                res[k]["device_us"].append(d)
        out["loss"][name] = {k: dict(host_us=summary(v["host_us"]), device_us=summary(v["device_us"])) for k, v in res.items()}
        print(name, {k: round(statistics.median(v["host_us"]), 1) for k, v in res.items()}, flush=True)
        del sets, arms
        torch._dynamo.reset()

    # 2. the stand-in training step
    torch.manual_seed(0)
    data = []
    for i in range(a.sets):
        ff, bf = tcl.synth.make_flows(B, H, W, seed=300 + i, max_shift=12.0, device=dev)
        xp, xc = (t.to(dev) for t in tcl.synth.make_frames(B, C, H, W, seed=300 + i, kind="smooth"))
        data.append((xp, xc, bf, tcl.fbcCheckTorch(ff, bf)))
    arms = {}
    for k, fn in (("eager", tcl_step_loss), ("reduce_overhead", torch.compile(tcl_step_loss, mode="reduce-overhead", fullgraph=True))):
        G = StandIn().to(dev)
        opt = torch.optim.SGD(G.parameters(), lr=1e-3)

        def step(d, G=G, opt=opt, fn=fn):
            opt.zero_grad(set_to_none=True)
            fn(G, *d).backward()
            opt.step()
        arms[k] = step
        for d in data * 3:
            step(d)
    res = {k: [] for k in arms}
    for r in range(a.rounds):
        for k in (list(arms) if r % 2 == 0 else list(arms)[::-1]):
            h, _ = timed_loop(arms[k], data, a.seconds)
            res[k].append(1e6 / h)
    out["step"] = dict(what="conv(3->8) relu conv(8->3) sigmoid on both frames + temporal_loss * 100 + SGD, 16x3x256x256",
                       steps_per_s={k: summary(v) for k, v in res.items()})
    print("step", {k: round(statistics.median(v), 1) for k, v in res.items()}, flush=True)

    # 3. bench.py, parent tree and this tree, alternated
    if a.parent:
        lines = {"parent": [], "this": []}
        for r in range(2):
            for k in (("parent", "this") if r % 2 == 0 else ("this", "parent")):
                lines[k].append(bench_line(a.parent if k == "parent" else ROOT, a.bench_steps, a.bench_warmup))
        out["bench"] = {k: dict(result_check=[l.get("result_check") for l in v], value=[l.get("value") for l in v],
                                unit=v[0].get("unit")) for k, v in lines.items()}
        print("bench", json.dumps(out["bench"]), flush=True)
    out["gpu_after"] = gpu_info()
    s = json.dumps(out, indent=1)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(s + "\n")
    print(s)


if __name__ == "__main__":
    main()
