"""A/B of the specular lattice pass instances on the bench's render inputs, in one process (GPU).

    python scripts/spec_eval_ab.py [--rounds R] [--steps K] [--json FILE]

Renders the inputs of `bench.py --workload render` (64 synthetic 2000x1000 envmaps, the bench's BRDF and view draws and
auto footprints, 128^2 refmaps) with the default pass instances (DrmRenderOptions::spec_kernels = 0) and the pinned ones
(spec_kernels = 1), alternated R times.  Per round and path: the step time from CUDA events over K steps, and the time
of each specular pass and of the diffuse pass in one step under torch.profiler (the method of spec_pass_times.py).  Then
the difference of the two outputs per refmap (relative L2, worst cell over the refmap's peak).  The card's name, power
limit and max SM clock are read in the same run.
"""
from __future__ import annotations

import argparse
import json
import re
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "scripts"))
sys.dont_write_bytecode = True

from spec_pass_times import gpu_info, short_name  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--json", help="also write the result as JSON to this file")
    args = ap.parse_args()

    import torch
    from torch.profiler import ProfilerActivity, profile

    import bench
    from drmnet_b200 import _lib
    from drmnet_b200.renderer import render_batch
    from drmnet_b200.synth import sample_brdf, sample_view, synthetic_envmap
    assert torch.cuda.is_available(), "spec_eval_ab.py needs a CUDA device"
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    card = gpu_info()

    n = 64
    envs = torch.stack([synthetic_envmap(bench.HE, bench.WE, seed=1000 + b, device=dev, as_numpy=False) for b in range(n)])
    z = torch.stack([sample_brdf(1000 + b) for b in range(n)]).to(dev)
    view = torch.stack([sample_view(1000 + b) for b in range(n)]).to(dev)
    S = bench.footprints(z.cpu(), "auto")
    opts = {}
    for name, v in (("pinned", 1), ("new", 0)):
        o = _lib.default_render_options()
        o.spec_kernels = v
        opts[name] = o
    outs = {name: torch.empty((n, 3, bench.RES, bench.RES), dtype=torch.float32, device=dev) for name in opts}

    def step(name):
        return render_batch(envs, z, view, res=bench.RES, footprint_S=S, out=outs[name], options=opts[name])

    for name in opts:
        for _ in range(3):
            step(name)
    torch.cuda.synchronize()

    res = {name: {"step_ms": [], "pass_ms": []} for name in opts}
    for _ in range(args.rounds):
        for name in opts:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.steps):
                step(name)
            e1.record()
            torch.cuda.synchronize()
            res[name]["step_ms"].append(e0.elapsed_time(e1) / args.steps)
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                step(name)
                torch.cuda.synchronize()
            passes = {}
            for e in prof.events():
                if e.device_type != torch.autograd.DeviceType.CUDA or "drm::" not in e.name:
                    continue
                k = short_name(e.name)
                m = re.match(r"tree_spec_pass2?_kernel(?:_h)?<(\d)>", k)
                key = f"spec pass {m.group(1)}" if m else ("diffuse" if k.startswith("tree_diff_kernel") else None)
                if key:
                    passes[key] = passes.get(key, 0.0) + e.time_range.elapsed_us() / 1e3
            res[name]["pass_ms"].append(dict(sorted(passes.items())))

    new, old = outs["new"].flatten(1).double(), outs["pinned"].flatten(1).double()
    rel = ((new - old).norm(dim=1) / old.norm(dim=1)).cpu()
    worst = ((new - old).abs().amax(dim=1) / old.abs().amax(dim=1)).cpu()
    result = {"card": card, "inputs": f"bench render: {n} x {bench.HE}x{bench.WE} fp32 envmaps, 128^2 refmaps, "
                                      f"footprints {{S: count}} = { {s: S.count(s) for s in sorted(set(S))} }",
              "rounds": args.rounds, "steps": args.steps, **res,
              "new_vs_pinned": {"rel_l2_max": float(rel.max()), "rel_l2_median": float(rel.median()),
                                "worst_cell_over_peak_max": float(worst.max())}}
    print(f"# {card}")
    for r in range(args.rounds):
        for name in opts:
            p = res[name]["pass_ms"][r]
            print(f"round {r + 1} {name:6s} step {res[name]['step_ms'][r]:8.2f} ms  " +
                  "  ".join(f"{k.replace('spec pass ', 'p')} {v:6.2f}" for k, v in p.items()))
    print("new vs pinned: " + json.dumps(result["new_vs_pinned"]))
    if args.json:
        Path(args.json).write_text(json.dumps(result, indent=1) + "\n")


if __name__ == "__main__":
    main()
