"""Instruction-text comparison of kernels between two builds (cuobjdump -sass, no GPU needed).

Template parameters change mangled names, so kernels are matched by a key the caller derives from the demangled name, and
compared by their instruction text alone (opcode and operands; addresses and encodings dropped).

  python tools/sass_diff.py OLD.so|.o NEW.so|.o [--match warp_backward_kernel]
      prints one line per matched kernel: identical / DIFFERENT (+ the first differing instruction); exit code 1 on any difference
  python tools/sass_diff.py --exact OLD.so|.o NEW.so|.o [--match ""]
      the same over every matched kernel, bf16 ones included, keyed by its full demangled name (no fp32 key folding)
  python tools/sass_diff.py --digest LIB [--match ...]
      prints a SHA-256 of each matched kernel's instruction text (what tests/test_bf16_backward_cpu.py pins)
"""
import argparse
import hashlib
import re
import subprocess
import sys


def kernels(path, match):
    """{demangled name: [instruction text, ...]} of every kernel whose demangled name contains `match`."""
    sass = subprocess.run(["cuobjdump", "-sass", path], capture_output=True, text=True, check=True).stdout
    funcs, cur = {}, None
    for line in sass.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            cur = m.group(1)
            funcs[cur] = []
            continue
        m = re.match(r"\s*/\*[0-9a-f]{4,}\*/\s+(.*?)\s*;", line)
        if cur and m:
            funcs[cur].append(re.sub(r"\s+", " ", m.group(1)))
    names = list(funcs)
    demangled = subprocess.run(["c++filt"] + names, capture_output=True, text=True, check=True).stdout.splitlines() if names else []
    return {d: funcs[n] for n, d in zip(names, demangled) if match in d}


def fp32_key(name):
    """Demangled name without a trailing fp32 frame-type template argument: `k<true, 3, float>` and `k<true, 3>` -> `k<true, 3>`."""
    return re.sub(r",\s*float>", ">", name)


def digest(instrs):
    return hashlib.sha256("\n".join(instrs).encode()).hexdigest()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("old", nargs="?")
    ap.add_argument("new")
    ap.add_argument("--match", default="warp_backward_kernel")
    ap.add_argument("--digest", action="store_true")
    ap.add_argument("--exact", action="store_true", help="key every kernel by its full demangled name")
    args = ap.parse_args()
    if args.digest:
        for name, instrs in sorted(kernels(args.new, args.match).items()):
            if "__nv_bfloat16" not in name:
                print(f"{fp32_key(name)}  {len(instrs)}  {digest(instrs)}")
        return 0
    if args.exact:
        old, new = kernels(args.old, args.match), kernels(args.new, args.match)
    else:
        old = {fp32_key(k): v for k, v in kernels(args.old, args.match).items()}
        new = {fp32_key(k): v for k, v in kernels(args.new, args.match).items() if "__nv_bfloat16" not in k}
    bad = 0
    for key in sorted(set(old) | set(new)):
        if key not in old or key not in new:
            print(f"{key}: only in {'new' if key in new else 'old'}")
            bad += 1
            continue
        a, b = old[key], new[key]
        if a == b:
            print(f"{key}: identical ({len(a)} instructions)")
            continue
        bad += 1
        i = next((i for i, (x, y) in enumerate(zip(a, b)) if x != y), min(len(a), len(b)))
        print(f"{key}: DIFFERENT ({len(a)} vs {len(b)} instructions; first at {i}: {a[i] if i < len(a) else '-'} | {b[i] if i < len(b) else '-'})")
    return 1 if bad else 0


if __name__ == "__main__":
    sys.exit(main())
