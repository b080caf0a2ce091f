"""Time of every kernel launch of one `bench.py --workload render` step, and of each specular lattice pass (GPU).

    python scripts/spec_pass_times.py [--batch B] [--footprint auto|S] [--repeats R] [--json FILE]

The inputs are the bench's own (`bench.wl_render`: same seeds, footprints and sizes).  After a warm-up, R steps run under
torch.profiler with CUDA activities; each launch's time is the median over the steps.  The pass of a specular launch is
read from its template argument (`tree_spec_pass_kernel<P>`) or, for a library with one kernel for all passes, from its
position after the diffuse launch of its chunk of renders.
"""
from __future__ import annotations

import argparse
import json
import re
import statistics
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.dont_write_bytecode = True


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except Exception as e:  # the times stand without it; say why it is missing
        return f"unknown ({e})"


def short_name(name):
    m = re.search(r"drm::(\w+)(<[^>]*>)?", name)
    return (m.group(1) + (m.group(2) or "")) if m else name[:60]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=0)
    ap.add_argument("--footprint", default="auto")
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--json", help="also write the result as JSON to this file")
    args = ap.parse_args()

    import torch
    from torch.profiler import ProfilerActivity, profile

    import bench
    from drmnet_b200 import _lib
    assert torch.cuda.is_available(), "spec_pass_times.py needs a CUDA device"
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    W = bench.wl_render(argparse.Namespace(batch=args.batch, footprint=args.footprint), 0, dev)
    for _ in range(3):
        W["step"]()
    torch.cuda.synchronize()

    steps = []
    for _ in range(args.repeats):
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            W["step"]()
            torch.cuda.synchronize()
        kern = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA and "drm::" in e.name]
        kern.sort(key=lambda e: e.time_range.start)
        launches, pass_idx = [], -1
        for e in kern:
            name = short_name(e.name)
            p = None
            if name.startswith("tree_diff_kernel"):
                pass_idx = -1
            elif re.match(r"tree_spec_pass2?_kernel", name):
                pass_idx += 1
                m = re.search(r"<(\d+)>", name)
                p = int(m.group(1)) if m else pass_idx
            launches.append((name, p, e.time_range.elapsed_us() / 1e3))
        steps.append(launches)

    n = min(len(s) for s in steps)
    rows = []
    for i in range(n):
        name, p, _ = steps[0][i]
        rows.append({"kernel": name, "pass": p, "ms": statistics.median(s[i][2] for s in steps)})
    total = sum(r["ms"] for r in rows)
    passes = {}
    for r in rows:
        if r["pass"] is not None:
            passes[r["pass"]] = passes.get(r["pass"], 0.0) + r["ms"]
    info = gpu_info()
    print(f"GPU (name, power limit, max SM clock): {info}")
    print(f"torch {torch.__version__}, library {_lib.SO_PATH}, {W['units']} renders, footprints "
          f"{W['config']['footprint_S_histogram']}, median of {args.repeats} profiled steps")
    for r in rows:
        tag = f"pass {r['pass']}" if r["pass"] is not None else ""
        print(f"  {r['kernel']:40s} {tag:7s} {r['ms']:9.3f} ms")
    print(f"kernels in all: {total:.3f} ms")
    for p in sorted(passes):
        print(f"  specular pass {p}: {passes[p]:9.3f} ms  ({100 * passes[p] / total:5.1f} %)")
    diff = sum(r["ms"] for r in rows if r["kernel"].startswith("tree_diff_kernel"))
    print(f"  diffuse pass:    {diff:9.3f} ms  ({100 * diff / total:5.1f} %)")
    if args.json:
        Path(args.json).parent.mkdir(parents=True, exist_ok=True)
        Path(args.json).write_text(json.dumps({"gpu": info, "launches": rows, "passes_ms": passes, "diffuse_ms": diff,
                                               "kernels_ms": total}, indent=1))


if __name__ == "__main__":
    main()
