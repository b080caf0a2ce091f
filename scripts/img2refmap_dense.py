"""What scattering dense images in place saves over compacting them first (GPU).

    python scripts/img2refmap_dense.py [--rounds R] [--steps K] [--batch B] [--json FILE]

Inputs: B sphere images of 512 x 512 (synth.sphere_normals(256), normals perturbed as normalise(n + N(0, 0.05)) inside
the sphere, SURVEY 8d (c)), shaded by refmap_lookup of a rendered 128^2 refmap and written as a dense colour image with
N(0, 0.01) relative noise (8d (b)); mask = ||n|| > 0.5 as ObsNet builds it.  Both layouts, [B,H,W,3] and [B,3,H,W],
each contiguous.  res 128, thr pi/256 (bench.py --workload img2refmap).

Each step goes from the dense tensors on the device to the four outputs:
  (a) today's route: boolean-mask compaction of colours and normals, offsets = running mask sums, img2refmap_batch;
  (b) img2refmap_images on the dense tensors.
Per step: device time between CUDA events around the step, and host wall time with a final synchronise.  (a) and (b)
alternate R times in one process, per layout, after a warm-up; the outputs of (a) and (b) are checked equal in the same
run (sel_index mapped through the compaction), and the card's name and power limit are read in the same run.
"""
from __future__ import annotations

import argparse
import json
import statistics
import subprocess
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.dont_write_bytecode = True


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm",
                            "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
        return q.splitlines()[0] if q else "unknown"
    except Exception as e:  # the numbers stand without it; say why it is missing
        return f"unknown ({e})"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--json", default=str(ROOT / "profiles" / "r7_img2refmap_dense.json"))
    args = ap.parse_args()
    if args.rounds < 3 or args.steps < 1 or args.batch < 1:
        ap.error("--rounds >= 3, --steps >= 1, --batch >= 1")

    import numpy as np
    import torch

    from drmnet_b200 import _lib
    from drmnet_b200.callers import refmap_lookup
    from drmnet_b200.img2refmap import img2refmap_batch, img2refmap_images
    from drmnet_b200.renderer import render_batch
    from drmnet_b200.synth import sphere_normals, synthetic_envmap
    assert torch.cuda.is_available(), "img2refmap_dense.py needs a CUDA device"
    dev = torch.device("cuda", 0)
    info = gpu_info()
    B, res, thr = args.batch, 128, float(np.pi / 128 / 2)

    # inputs
    env = torch.from_numpy(synthetic_envmap(250, 500, seed=9)).to(dev)
    refmap = render_batch(env[None], torch.tensor([[0.3, 0.8, 0.6, 0.4, 0.5, 0.7]]), torch.tensor([[0.0, 0.0, 1.0]]),
                          res=res, footprint_S=1)
    n0, m0 = sphere_normals(256)
    g = torch.Generator(device=dev).manual_seed(7)
    n = torch.from_numpy(n0).to(dev)[None].repeat(B, 1, 1, 1)
    n = n + 0.05 * torch.randn(n.shape, generator=g, device=dev)
    inside = torch.from_numpy(m0).to(dev)[None, ..., None]
    nrm = torch.where(inside, n / n.norm(dim=-1, keepdim=True), torch.zeros((), device=dev)).contiguous()
    col = refmap_lookup(refmap, nrm.view(-1, 3)).view(B, 512, 512, 3)
    col = (col * (1 + 0.01 * torch.randn(col.shape, generator=g, device=dev))).contiguous()
    mask = nrm.norm(dim=-1) > 0.5
    layouts = {"hwc": (col, nrm, False), "chw": (col.permute(0, 3, 1, 2).contiguous(),
                                                 nrm.permute(0, 3, 1, 2).contiguous(), True)}
    masked = int(mask.sum())

    def compacted(c, nm, channel_first):
        if channel_first:
            c, nm = c.permute(0, 2, 3, 1), nm.permute(0, 2, 3, 1)
        offsets = torch.zeros(B + 1, dtype=torch.int64, device=dev)
        offsets[1:] = mask.sum((1, 2)).cumsum(0)
        return img2refmap_batch(c[mask], nm[mask], offsets, res, thr)

    def dense(c, nm, channel_first):
        return img2refmap_images(c, nm, mask, res, thr, channel_first=channel_first)

    # equal outputs, in this run
    for name, (c, nm, cf) in layouts.items():
        a, b = compacted(c, nm, cf), dense(c, nm, cf)
        sel = a[3].clone()
        for k in range(B):
            idx = mask[k].flatten().nonzero().squeeze(1).to(torch.int32)
            hit = a[3][k] >= 0
            sel[k][hit] = idx[a[3][k][hit].long()]
        for x, y in zip((*a[:3], sel), b):
            assert torch.equal(x, y), f"{name}: outputs of (a) and (b) differ"
    print(f"outputs of (a) and (b) equal for both layouts ({masked} masked px in {B} images)")

    def timed(fn, c, nm, cf):
        dev_ms, wall_ms = [], []
        for _ in range(args.steps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            e0.record()
            fn(c, nm, cf)
            e1.record()
            torch.cuda.synchronize()
            wall_ms.append((time.perf_counter() - t0) * 1e3)
            dev_ms.append(e0.elapsed_time(e1))
        return statistics.median(dev_ms), statistics.median(wall_ms)

    routes = {"a_compact_then_batch": compacted, "b_img2refmap_images": dense}
    for name, (c, nm, cf) in layouts.items():  # warm-up of every shape the timed window uses
        for fn in routes.values():
            for _ in range(2):
                fn(c, nm, cf)
    torch.cuda.synchronize()
    rounds = []
    for r in range(args.rounds):
        row = {}
        for name, (c, nm, cf) in layouts.items():
            for route, fn in routes.items():
                d, w = timed(fn, c, nm, cf)
                row[f"{name}/{route}"] = {"device_ms_per_step": round(d, 3), "wall_ms_per_step": round(w, 3)}
        rounds.append(row)
        print(f"round {r}: " + "; ".join(f"{k} {v['device_ms_per_step']:.3f} / {v['wall_ms_per_step']:.3f} ms"
                                          for k, v in row.items()))

    summary = {}
    for key in rounds[0]:
        d = [rw[key]["device_ms_per_step"] for rw in rounds]
        w = [rw[key]["wall_ms_per_step"] for rw in rounds]
        summary[key] = {"device_ms_per_step_min_max": [min(d), max(d)], "wall_ms_per_step_min_max": [min(w), max(w)]}
    result = {
        "what": "image -> refmap scatter of dense images under a mask: (a) boolean-mask compaction + offsets + "
                "img2refmap_batch vs (b) img2refmap_images, each step from dense device tensors to the four outputs",
        "gpu_name_power_limit_max_sm_clock": info, "torch": torch.__version__,
        "inputs": {"images": B, "H": 512, "W": 512, "masked_pixels": masked, "res": res, "thr": thr,
                   "layouts": {"hwc": "[B,512,512,3] contiguous", "chw": "[B,3,512,512] contiguous"},
                   "colours": "refmap_lookup of a rendered 128^2 refmap, N(0, 0.01) relative noise",
                   "normals": "sphere_normals(256), normalise(n + N(0, 0.05)) inside the sphere", "mask": "||n|| > 0.5"},
        "method": f"{args.rounds} rounds alternating (a) and (b) per layout in one process, {args.steps} steps each after "
                  "2 warm-up steps; per-step medians; device time = CUDA events around the step, wall = host clock "
                  "around the step and a final synchronise",
        "outputs_equal": True,
        "workspace_bytes": {"a": int(_lib.lib().drm_img2refmap_workspace_bytes(masked, B, res, thr)),
                            "b": int(_lib.lib().drm_img2refmap_dense_workspace_bytes(B, 512, 512, res, thr))},
        "rounds": rounds, "summary": summary,
    }
    print(f"GPU (name, power limit, max SM clock): {info}")
    for k, v in summary.items():
        print(f"{k}: device {v['device_ms_per_step_min_max']} ms, wall {v['wall_ms_per_step_min_max']} ms per step")
    Path(args.json).parent.mkdir(parents=True, exist_ok=True)
    Path(args.json).write_text(json.dumps(result, indent=1) + "\n")


if __name__ == "__main__":
    main()
